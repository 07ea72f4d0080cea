// Persistent, warp-specialised tcgen05 GEMM for sm_100a.
//
//   D[M,N] = alpha[n/64] * sum_s A_s[M,K_s] * B_s[K_s,N]  (+ bias[N])        s = 0 .. nseg-1 (<= 4 segments)
//
// One CTA per SM, 256 threads:
//   warp 0 / lane 0 : TMA producer  (global -> 128B-swizzled smem ring, mbarrier complete_tx)
//   warp 1 / lane 0 : MMA issuer    (tcgen05.mma, M=128 x N=BN x K=16, fp32 accumulators in TMEM, 2 stages)
//   warp 2          : TMEM allocator / deallocator
//   warps 4..7      : epilogue      (tcgen05.ld -> registers -> {bf16 / fp16 via swizzled smem + TMA store | fp32 split-K partial})
//
// F16 selects the 16-bit operand type: bf16 (false) or IEEE fp16 (true) -- the instruction-descriptor format, the TMA
// element type (host side) and the EPI_BF16_TMA conversion; everything else is shared.
//
// Operand "majorness" is a template parameter because the SoW hot path needs all four combinations without
// re-laying-out any user-visible tensor (reference layout of W is (in,out), tn_gradient/layer/sow.py:28,74-79):
//   forward   y  = x.W      : A K-major,  B MN-major  (W rows are K, N contiguous)
//   backward  dX = dY.W^T   : A K-major,  B K-major   (same W buffer, rows are N, K contiguous)
//   backward  dA = x^T.dt   : A MN-major, B MN-major  (split-K over tokens, fp32 partials summed in a fixed order)
// The contraction is a list of K-SEGMENTS, each with its own pair of tensor maps, accumulated into the same TMEM tile:
//   * the rank-r "tail" (t.B in the forward, dt.A^T in dX) is one more segment, which is how the low-rank term is fused
//     into the base GEMM (no second pass over y / dX);
//   * projections that share their input (q/k/v, gate/up) share ONE dX launch: dX = sum_p dY_p.W_p^T + dt_cat.A_cat^T is
//     a 4-segment contraction, so dX is written once instead of n times plus n-1 elementwise adds;
//   * fp32 modules run as bf16x3: [x_hi | x_hi | x_lo].[W_hi ; W_lo ; W_hi] is a 3-segment contraction.
// alpha is looked up per 64-wide column block so that one skinny launch t_cat = x.[A_q|A_k|A_v] can apply each
// projection's own scale.
#pragma once
#include "ptx.cuh"

namespace sowb {

constexpr int kBM = 128;      // UMMA M (cta_group::1)
constexpr int kBK = 64;       // k-block depth in elements (= one 128B swizzle span of bf16)
constexpr int kUmmaK = 16;    // bf16 UMMA K
constexpr int kGemmThreads = 256;
constexpr int kEpiThreads = 128;
constexpr int kStoreBoxCols = 64;                                  // bf16 columns per TMA store box (128 B)
constexpr int kStageCBytes = kBM * kStoreBoxCols * 2;              // 16 KB per staging buffer

enum EpiMode : int {
  EPI_BF16_TMA = 0,    // D -> 16-bit (bf16, or fp16 with F16), via smem staging + TMA store (clips M/N tails)
  EPI_F32_PARTIAL = 1,  // D -> fp32 PARTIAL of split s stored at out_f32[s*split_stride + row*ldc + col]; the caller sums the
                       // splits in a fixed order (bit-reproducible, unlike red.global.add; no zero-fill needed)
  EPI_F32_TMA = 2,     // D -> fp32 (+ fp32 bias), via smem staging + TMA store: the output of the bf16x3 path of fp32 modules
};

constexpr int kMaxSeg = 10;   // 3 members x 3 bf16x3 pieces + the rank-r tail
constexpr int kMaxAlphaBlocks = 16;   // per-64-column alpha table covers N <= 1024 (wider outputs use alpha[0])

struct GemmMaps {
  CUtensorMap a[kMaxSeg];
  CUtensorMap b[kMaxSeg];
  CUtensorMap c;
};

struct GemmParams {
  int M, N;
  int nseg;
  int kb_end[kMaxSeg];  // cumulative count of kBK-deep k-blocks after segment s
  int m_tiles, n_tiles, splits;
  int kb_per_split;
  int alpha_blocks;     // 0: alpha[0] for every column; else alpha[(col / 64)]
  float alpha[kMaxAlphaBlocks];
  const uint16_t* bias;       // nullable, length N, the operands' 16-bit type (EPI_BF16_TMA only)
  const float* bias_f32;      // nullable, length N (EPI_F32_TMA only)
  float* out_f32;             // EPI_F32_PARTIAL only
  int64_t split_stride;       // EPI_F32_PARTIAL only: elements between the partial outputs of consecutive splits
  int ldc;
};

// MT = M tiles (of 128 rows) per CTA.  MT = 2 makes the CTA tile 256 x BN: both M tiles are multiplied by the SAME B tile,
// so a k-block moves 32 KB (A) + 32 KB (B) from L2 for twice the MACs of the 128 x 256 tile (16 + 32 KB) -- 62 instead of 94
// B/clk/SM at full tensor rate, which is what holds the 17-k-block forward tiles at ~65 % tensor-pipe activity.  The two
// accumulators take the place of the two TMEM stages, so the epilogue of a work item is not overlapped with the next one's
// MMAs; the launcher picks MT = 2 only where the wave quantisation of the larger tiles does not eat the gain.
template <int BN, int MT = 1>
struct GemmSmem {
  static constexpr int kABytes = MT * kBM * kBK * 2;
  static constexpr int kBBytes = BN * kBK * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  // leave room for 2 staging buffers (32 KB) + barriers inside the 227 KB opt-in limit
  static constexpr int kFit = (232448 - 1024 - 2 * kStageCBytes - 256) / kStageBytes;
  static constexpr int kStages = kFit > 8 ? 8 : kFit;
  static constexpr int kRingBytes = kStages * kStageBytes;
  static constexpr int kStagingBytes = 2 * kStageCBytes;
  static constexpr int kBarBytes = 256;
  static constexpr int kTotal = 1024 /*align slack*/ + kRingBytes + kStagingBytes + kBarBytes;
  static constexpr uint32_t kTmemCols = (2 * BN <= 32) ? 32 : (2 * BN <= 64 ? 64 : (2 * BN <= 128 ? 128 : (2 * BN <= 256 ? 256 : 512)));
};

// EPI_BF16_TMA epilogue of one 128-row accumulator, run by the 128 epilogue threads: TMEM (this warp's lane quarter, columns
// taddr ..) -> alpha, bias, round to 16 bits -> 128B-swizzled staging -> TMA store of 64-column boxes, clipped at M / N.
// The two staging buffers alternate; boxes_issued counts this CTA's stores across calls.  The same code as the EPI_BF16_TMA
// branch of sow_gemm_kernel, which keeps its inline copy: calling this from there renames registers in every instantiation.
template <int BN, bool F16>
__device__ __forceinline__ void epilogue_store16(const GemmParams& p, const CUtensorMap* map_c, uint8_t* staging, uint32_t taddr,
                                                 int m0, int n0, int row_in_tile, int et, uint32_t& boxes_issued) {
#pragma unroll 1
  for (int b = 0; b < BN / kStoreBoxCols; ++b) {
    if (n0 + b * kStoreBoxCols >= p.N) break;  // uniform across the CTA
    uint8_t* stg = staging + (boxes_issued & 1) * kStageCBytes;
    const float alpha = p.alpha[p.alpha_blocks ? min(p.alpha_blocks - 1, (n0 >> 6) + b) : 0];
    if (boxes_issued >= 2) {
      if (et == 0) tma_store_wait_read<1>();  // the store that last used this buffer has read it
      named_barrier_sync(1, kEpiThreads);
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      uint32_t v[32];
      tmem_ld32(taddr + b * kStoreBoxCols + h * 32, v);
      tmem_ld_wait();
      const int colbase = n0 + b * kStoreBoxCols + h * 32;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        float f[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          f[j] = alpha * __uint_as_float(v[c * 8 + j]);
          if (p.bias != nullptr) {
            const int col = colbase + c * 8 + j;
            if (col < p.N) f[j] += lo16_to_f32<F16>(p.bias[col]);
          }
        }
        uint4 pk;
        pk.x = pack16x2<F16>(f[0], f[1]);
        pk.y = pack16x2<F16>(f[2], f[3]);
        pk.z = pack16x2<F16>(f[4], f[5]);
        pk.w = pack16x2<F16>(f[6], f[7]);
        const int chunk = h * 4 + c;  // 16-byte chunk index inside the 128-byte row
        *reinterpret_cast<uint4*>(stg + row_in_tile * 128 + ((chunk ^ (row_in_tile & 7)) << 4)) = pk;
      }
    }
    fence_proxy_async_smem();
    named_barrier_sync(1, kEpiThreads);
    if (et == 0) {
      tma_store_2d(map_c, stg, n0 + b * kStoreBoxCols, m0);
      tma_store_commit();
    }
    ++boxes_issued;
  }
}

template <int BN, bool A_MN, bool B_MN, int EPI, int MT = 1, bool F16 = false>
__global__ void __launch_bounds__(kGemmThreads, 1)
sow_gemm_kernel(const __grid_constant__ GemmMaps maps, const GemmParams p) {
  using S = GemmSmem<BN, MT>;
  static_assert(MT == 1 || MT == 2, "one or two M tiles per CTA");
  extern __shared__ uint8_t smem_raw[];
  // SWIZZLE_128B atoms need 1024-byte alignment
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* ring = smem;
  uint8_t* staging = smem + S::kRingBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(staging + S::kStagingBytes);
  uint64_t* full_bar = bars;                       // [kStages]
  uint64_t* empty_bar = bars + S::kStages;         // [kStages]
  uint64_t* tfull_bar = bars + 2 * S::kStages;     // [2]
  uint64_t* tempty_bar = bars + 2 * S::kStages + 2;  // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * S::kStages + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    for (int sg = 0; sg < p.nseg; ++sg) {
      tma_prefetch_desc(&maps.a[sg]);
      tma_prefetch_desc(&maps.b[sg]);
    }
    if (EPI != EPI_F32_PARTIAL) tma_prefetch_desc(&maps.c);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < S::kStages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], kEpiThreads);
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, S::kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int total_work = p.m_tiles * p.n_tiles * p.splits;
  const int kb_total = p.kb_end[p.nseg - 1];

  if (warp == 0 && lane == 0) {
    // ===================== TMA producer =====================
    int stage = 0;
    uint32_t phase = 0;
    for (int w = blockIdx.x; w < total_work; w += gridDim.x) {
      const int split = w % p.splits;
      const int tile = w / p.splits;
      const int m0 = (tile / p.n_tiles) * kBM * MT;
      const int n0 = (tile % p.n_tiles) * BN;
      const int kb_begin = split * p.kb_per_split;
      const int kb_end = min(kb_total, kb_begin + p.kb_per_split);
      int seg = 0;
      while (kb_begin >= p.kb_end[seg]) ++seg;
      for (int kb = kb_begin; kb < kb_end; ++kb) {
        mbar_wait(&empty_bar[stage], phase ^ 1);
        uint8_t* sa = ring + stage * S::kStageBytes;
        uint8_t* sb = sa + S::kABytes;
        mbar_expect_tx(&full_bar[stage], S::kStageBytes);
        while (kb >= p.kb_end[seg]) ++seg;
        const CUtensorMap* ma = &maps.a[seg];
        const CUtensorMap* mb = &maps.b[seg];
        const int k0 = (kb - (seg ? p.kb_end[seg - 1] : 0)) * kBK;
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) {
          if (A_MN) {
            // global [K rows, M contiguous]: two boxes of (64 M) x (64 K) per M tile
#pragma unroll
            for (int j = 0; j < kBM / 64; ++j)
              tma_load_2d(sa + mt * 16384 + j * 8192, ma, &full_bar[stage], m0 + mt * kBM + 64 * j, k0);
          } else {
            // global [M rows, K contiguous]: one box of (64 K) x (128 M) per M tile (rows beyond M are zero-filled)
            tma_load_2d(sa + mt * 16384, ma, &full_bar[stage], k0, m0 + mt * kBM);
          }
        }
        if (B_MN) {
          // global [K rows, N contiguous]: BN/64 boxes of (64 N) x (64 K)
#pragma unroll
          for (int j = 0; j < BN / 64; ++j) tma_load_2d(sb + j * 8192, mb, &full_bar[stage], n0 + 64 * j, k0);
        } else {
          // global [N rows, K contiguous]: one box of (64 K) x (BN N)
          tma_load_2d(sb, mb, &full_bar[stage], k0, n0);
        }
        if (++stage == S::kStages) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 1 && lane == 0) {
    // ===================== MMA issuer =====================
    constexpr uint32_t idesc = make_idesc(ab_format16<F16>(), kBM, BN, A_MN ? 1 : 0, B_MN ? 1 : 0);
    // K-major:  SBO = 1024 B between 8-row atoms; advance 32 B per UMMA_K inside the 128 B swizzle span.
    // MN-major: LBO = 8192 B between 64-wide MN blocks (one TMA box each), SBO = 1024 B between 8-deep K groups;
    //           advance 2 K-groups = 2048 B per UMMA_K.
    constexpr uint32_t a_lbo = A_MN ? 8192 : 16, a_sbo = 1024, a_kstep = A_MN ? 2048 : 32;
    constexpr uint32_t b_lbo = B_MN ? 8192 : 16, b_sbo = 1024, b_kstep = B_MN ? 2048 : 32;
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int w = blockIdx.x; w < total_work; w += gridDim.x) {
      const int split = w % p.splits;
      const int kb_begin = split * p.kb_per_split;
      const int kb_end = min(kb_total, kb_begin + p.kb_per_split);
      mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + (MT == 2 ? 0 : acc * BN);
      for (int kb = kb_begin; kb < kb_end; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        const uint32_t sa = smem_u32(ring + stage * S::kStageBytes);
        const uint32_t sb = sa + S::kABytes;
#pragma unroll
        for (int k = 0; k < kBK / kUmmaK; ++k) {
          const uint64_t ad = make_smem_desc(sa + k * a_kstep, a_lbo, a_sbo);
          const uint64_t bd = make_smem_desc(sb + k * b_kstep, b_lbo, b_sbo);
          umma_bf16(tmem_d, ad, bd, idesc, (kb > kb_begin || k > 0) ? 1u : 0u);
          if (MT == 2) {
            const uint64_t ad1 = make_smem_desc(sa + 16384 + k * a_kstep, a_lbo, a_sbo);
            umma_bf16(tmem_d + BN, ad1, bd, idesc, (kb > kb_begin || k > 0) ? 1u : 0u);
          }
        }
        umma_commit(&empty_bar[stage]);  // frees the smem slot once these MMAs have read it
        if (++stage == S::kStages) {
          stage = 0;
          phase ^= 1;
        }
      }
      umma_commit(&tfull_bar[acc]);  // accumulator complete -> epilogue
      if (++acc == (MT == 2 ? 1 : 2)) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue =====================
    const int q = warp - 4;                  // TMEM lane quarter owned by this warp (warp % 4)
    const int row_in_tile = q * 32 + lane;   // accumulator row == TMEM lane
    const int et = threadIdx.x - 128;        // 0..127
    int acc = 0;
    uint32_t acc_phase = 0;
    uint32_t boxes_issued = 0;  // TMA-store boxes issued so far by this CTA (for staging double-buffer)
    for (int w = blockIdx.x; w < total_work; w += gridDim.x) {
      const int tile = w / p.splits;
      const int m0_first = (tile / p.n_tiles) * kBM * MT;
      const int n0 = (tile % p.n_tiles) * BN;
      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after();
#pragma unroll 1
      for (int mt = 0; mt < MT; ++mt) {
      const int m0 = m0_first + mt * kBM;
      if (m0 >= p.M) break;  // uniform across the CTA
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + (MT == 2 ? mt * BN : acc * BN);
      if (EPI == EPI_BF16_TMA) {
#pragma unroll 1
        for (int b = 0; b < BN / kStoreBoxCols; ++b) {
          if (n0 + b * kStoreBoxCols >= p.N) break;  // uniform across the CTA
          uint8_t* stg = staging + (boxes_issued & 1) * kStageCBytes;
          const float alpha = p.alpha[p.alpha_blocks ? min(p.alpha_blocks - 1, (n0 >> 6) + b) : 0];
          if (boxes_issued >= 2) {
            if (et == 0) tma_store_wait_read<1>();  // the store that last used this buffer has read it
            named_barrier_sync(1, kEpiThreads);
          }
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            uint32_t v[32];
            tmem_ld32(taddr + b * kStoreBoxCols + h * 32, v);
            tmem_ld_wait();
            const int colbase = n0 + b * kStoreBoxCols + h * 32;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              float f[8];
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                f[j] = alpha * __uint_as_float(v[c * 8 + j]);
                if (p.bias != nullptr) {
                  const int col = colbase + c * 8 + j;
                  if (col < p.N) f[j] += lo16_to_f32<F16>(p.bias[col]);
                }
              }
              uint4 pk;
              pk.x = pack16x2<F16>(f[0], f[1]);
              pk.y = pack16x2<F16>(f[2], f[3]);
              pk.z = pack16x2<F16>(f[4], f[5]);
              pk.w = pack16x2<F16>(f[6], f[7]);
              const int chunk = h * 4 + c;  // 16-byte chunk index inside the 128-byte row
              *reinterpret_cast<uint4*>(stg + row_in_tile * 128 + ((chunk ^ (row_in_tile & 7)) << 4)) = pk;
            }
          }
          fence_proxy_async_smem();
          named_barrier_sync(1, kEpiThreads);
          if (et == 0) {
            tma_store_2d(&maps.c, stg, n0 + b * kStoreBoxCols, m0);
            tma_store_commit();
          }
          ++boxes_issued;
        }
      } else if (EPI == EPI_F32_TMA) {
        // one 32-column fp32 box (128 B per row) per TMEM load; same double-buffered staging as the bf16 path
#pragma unroll 1
        for (int b = 0; b < BN / 32; ++b) {
          if (n0 + b * 32 >= p.N) break;  // uniform across the CTA
          uint8_t* stg = staging + (boxes_issued & 1) * kStageCBytes;
          if (boxes_issued >= 2) {
            if (et == 0) tma_store_wait_read<1>();
            named_barrier_sync(1, kEpiThreads);
          }
          const float alpha = p.alpha[p.alpha_blocks ? min(p.alpha_blocks - 1, (n0 + b * 32) >> 6) : 0];
          uint32_t v[32];
          tmem_ld32(taddr + b * 32, v);
          tmem_ld_wait();
          const int colbase = n0 + b * 32;
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            float f[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              f[j] = alpha * __uint_as_float(v[c * 4 + j]);
              if (p.bias_f32 != nullptr) {
                const int col = colbase + c * 4 + j;
                if (col < p.N) f[j] += p.bias_f32[col];
              }
            }
            *reinterpret_cast<float4*>(stg + row_in_tile * 128 + ((c ^ (row_in_tile & 7)) << 4)) = make_float4(f[0], f[1], f[2], f[3]);
          }
          fence_proxy_async_smem();
          named_barrier_sync(1, kEpiThreads);
          if (et == 0) {
            tma_store_2d(&maps.c, stg, n0 + b * 32, m0);
            tma_store_commit();
          }
          ++boxes_issued;
        }
      } else {
        const int row = m0 + row_in_tile;
        const int split = w % p.splits;
        float* part = p.out_f32 + static_cast<int64_t>(split) * p.split_stride;
        const float alpha = p.alpha[0];
#pragma unroll 1
        for (int c32 = 0; c32 < BN / 32; ++c32) {
          if (n0 + c32 * 32 >= p.N) break;
          uint32_t v[32];
          tmem_ld32(taddr + c32 * 32, v);
          tmem_ld_wait();
          if (row < p.M) {
            float* dst = part + static_cast<int64_t>(row) * p.ldc + n0 + c32 * 32;
            if (n0 + c32 * 32 + 32 <= p.N && (p.ldc & 3) == 0) {
#pragma unroll
              for (int j = 0; j < 8; ++j)
                *reinterpret_cast<float4*>(dst + 4 * j) =
                    make_float4(alpha * __uint_as_float(v[4 * j]), alpha * __uint_as_float(v[4 * j + 1]),
                                alpha * __uint_as_float(v[4 * j + 2]), alpha * __uint_as_float(v[4 * j + 3]));
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (n0 + c32 * 32 + j < p.N) dst[j] = alpha * __uint_as_float(v[j]);
            }
          }
        }
      }
      }  // mt
      // all TMEM reads of this accumulator stage are done -> hand it back to the MMA warp
      tc_fence_before();
      mbar_arrive(&tempty_bar[acc]);
      if (++acc == (MT == 2 ? 1 : 2)) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
    if (EPI != EPI_F32_PARTIAL && et == 0) tma_store_wait_all<0>();  // smem must outlive the bulk stores
  }

  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 2) tmem_dealloc(tmem_base, S::kTmemCols);
}

// CTA-pair tile: a cluster of two CTAs computes 256 x 256 of D with tcgen05.mma.cta_group::2 (M = 256).  Each CTA loads its
// own 128 rows of A and one 128-column half of the B tile, so a k-block moves 16 + 16 KB per SM instead of 16 + 32 KB of the
// 128 x 256 tile (62.5 instead of 94 B/clk/SM at full tensor rate), while each CTA still holds only its own 128 x 256 fp32
// accumulator: both TMEM stages stay, and the epilogue of one tile overlaps the MMAs of the next.  The 32 KB stage gives a
// 6-deep ring.
struct GemmPairSmem {
  static constexpr int kABytes = kBM * kBK * 2;           // this CTA's 128 rows of A
  static constexpr int kBBytes = 128 * kBK * 2;           // this CTA's 128 of the tile's 256 B columns
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kStages = (232448 - 1024 - 2 * kStageCBytes - 256) / kStageBytes;
  static constexpr int kRingBytes = kStages * kStageBytes;
  static constexpr int kStagingBytes = 2 * kStageCBytes;
  static constexpr int kBarBytes = 256;
  static constexpr int kTotal = 1024 /*align slack*/ + kRingBytes + kStagingBytes + kBarBytes;
  static constexpr uint32_t kTmemCols = 512;              // two 256-column accumulator stages
};

// EPI_BF16_TMA, BN = 256, A K-major, B MN-major (forward) or K-major (dX); launched in clusters of 2 CTAs along x.
//   even CTA ("leader"): its full barriers count both CTAs' TMA bytes; warp 1 issues every MMA of the pair and commits to
//                        both CTAs' empty / accumulator-full barriers; its accumulator-empty barriers count both epilogues.
//   odd CTA            : producer and epilogue only.
// Per output element the MMAs, their operands, their k-block order and the epilogue are those of sow_gemm_kernel<256, ..>.
template <bool B_MN, bool F16>
__global__ void __launch_bounds__(kGemmThreads, 1)
sow_gemm_pair_kernel(const __grid_constant__ GemmMaps maps, const GemmParams p) {
  using S = GemmPairSmem;
  constexpr int BN = 256;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* ring = smem;
  uint8_t* staging = smem + S::kRingBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(staging + S::kStagingBytes);
  uint64_t* full_bar = bars;                       // [kStages]  (used in the leader only)
  uint64_t* empty_bar = bars + S::kStages;         // [kStages]
  uint64_t* tfull_bar = bars + 2 * S::kStages;     // [2]
  uint64_t* tempty_bar = bars + 2 * S::kStages + 2;  // [2]     (used in the leader only)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * S::kStages + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int cluster = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;

  if (warp == 0 && lane == 0) {
    for (int sg = 0; sg < p.nseg; ++sg) {
      tma_prefetch_desc(&maps.a[sg]);
      tma_prefetch_desc(&maps.b[sg]);
    }
    tma_prefetch_desc(&maps.c);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < S::kStages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], 2 * kEpiThreads);
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc_pair(tmem_slot, S::kTmemCols);
    tmem_relinquish_pair();
  }
  tc_fence_before();
  cluster_sync_all();   // both CTAs' barriers are initialised before the peer's TMA or the leader's commits reach them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int total_work = p.m_tiles * p.n_tiles;
  const int kb_total = p.kb_end[p.nseg - 1];

  if (warp == 0 && lane == 0) {
    // ===================== TMA producer (both CTAs) =====================
    const uint32_t full_leader = map_to_cta(smem_u32(full_bar), 0);
    int stage = 0;
    uint32_t phase = 0;
    for (int w = cluster; w < total_work; w += n_clusters) {
      const int m0 = (w / p.n_tiles) * 2 * kBM + static_cast<int>(rank) * kBM;
      const int n0 = (w % p.n_tiles) * BN + static_cast<int>(rank) * (BN / 2);
      int seg = 0;
      for (int kb = 0; kb < kb_total; ++kb) {
        mbar_wait(&empty_bar[stage], phase ^ 1);
        uint8_t* sa = ring + stage * S::kStageBytes;
        uint8_t* sb = sa + S::kABytes;
        if (rank == 0) mbar_expect_tx(&full_bar[stage], 2 * S::kStageBytes);
        while (kb >= p.kb_end[seg]) ++seg;
        const CUtensorMap* ma = &maps.a[seg];
        const CUtensorMap* mb = &maps.b[seg];
        const int k0 = (kb - (seg ? p.kb_end[seg - 1] : 0)) * kBK;
        const uint32_t fb = full_leader + stage * 8;
        tma_load_2d_pair(sa, ma, fb, k0, m0);   // (64 K) x (128 M); rows beyond M are zero-filled
        if (B_MN) {
          // global [K rows, N contiguous]: two boxes of (64 N) x (64 K)
#pragma unroll
          for (int j = 0; j < 2; ++j) tma_load_2d_pair(sb + j * 8192, mb, fb, n0 + 64 * j, k0);
        } else {
          // global [N rows, K contiguous]: one box of (64 K) x (128 N)
          tma_load_2d_pair(sb, mb, fb, k0, n0);
        }
        if (++stage == S::kStages) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
    // every slot's last release (a commit of the leader's MMA warp) has landed before this CTA may exit
    for (int i = 0; i < S::kStages; ++i) {
      mbar_wait(&empty_bar[stage], phase ^ 1);
      if (++stage == S::kStages) {
        stage = 0;
        phase ^= 1;
      }
    }
  } else if (warp == 1 && lane == 0 && rank == 0) {
    // ===================== MMA issuer (leader only) =====================
    constexpr uint32_t idesc = make_idesc(ab_format16<F16>(), 2 * kBM, BN, 0, B_MN ? 1 : 0);
    constexpr uint32_t a_lbo = 16, a_sbo = 1024, a_kstep = 32;
    constexpr uint32_t b_lbo = B_MN ? 8192 : 16, b_sbo = 1024, b_kstep = B_MN ? 2048 : 32;
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int w = cluster; w < total_work; w += n_clusters) {
      mbar_wait_cluster(&tempty_bar[acc], acc_phase ^ 1);
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + acc * BN;
      for (int kb = 0; kb < kb_total; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        const uint32_t sa = smem_u32(ring + stage * S::kStageBytes);
        const uint32_t sb = sa + S::kABytes;
#pragma unroll
        for (int k = 0; k < kBK / kUmmaK; ++k) {
          const uint64_t ad = make_smem_desc(sa + k * a_kstep, a_lbo, a_sbo);
          const uint64_t bd = make_smem_desc(sb + k * b_kstep, b_lbo, b_sbo);
          umma_bf16_pair(tmem_d, ad, bd, idesc, (kb > 0 || k > 0) ? 1u : 0u);
        }
        umma_commit_pair(&empty_bar[stage], 0x3);  // frees the slot in both CTAs once these MMAs have read it
        if (++stage == S::kStages) {
          stage = 0;
          phase ^= 1;
        }
      }
      umma_commit_pair(&tfull_bar[acc], 0x3);  // both halves of the accumulator complete -> both epilogues
      if (++acc == 2) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue (both CTAs, each over its own 128 TMEM lanes) =====================
    const int q = warp - 4;
    const int row_in_tile = q * 32 + lane;
    const int et = threadIdx.x - 128;
    const uint32_t tempty_leader = map_to_cta(smem_u32(tempty_bar), 0);
    int acc = 0;
    uint32_t acc_phase = 0;
    uint32_t boxes_issued = 0;
    for (int w = cluster; w < total_work; w += n_clusters) {
      const int m0 = (w / p.n_tiles) * 2 * kBM + static_cast<int>(rank) * kBM;
      const int n0 = (w % p.n_tiles) * BN;
      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after();
      if (m0 < p.M)   // uniform across the CTA; the odd CTA of a tile with <= 128 valid rows has nothing to store
        epilogue_store16<BN, F16>(p, &maps.c, staging, tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * BN, m0, n0,
                                  row_in_tile, et, boxes_issued);
      // this CTA's TMEM reads of the stage are done -> hand it back to the leader's MMA warp
      tc_fence_before();
      mbar_arrive_remote(tempty_leader + acc * 8);
      if (++acc == 2) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
    if (et == 0) tma_store_wait_all<0>();  // smem must outlive the bulk stores
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // neither CTA frees TMEM or exits while the pair's MMAs, commits or remote arrives may touch it
  tc_fence_after();
  if (warp == 2) tmem_dealloc_pair(tmem_base, S::kTmemCols);
}

}  // namespace sowb
