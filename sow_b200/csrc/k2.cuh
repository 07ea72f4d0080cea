// K2: ONE pass over dY that produces both rank-r backward products of a SoW linear
//
//     dt   [T, 64]   = scale * dY [T, out] . B^T [out, 64]          (contraction over out)
//     dB^T [out, 64] = dY^T [out, T] . t [T, 64]                    (contraction over T)
//
// (autograd of tn_gradient/layer/sow.py:117-121; the reference issues two cuBLAS GEMMs that each stream dY from HBM).
// Both products consume the SAME shared-memory tile of dY: a [128 T-rows x 128 out-cols] tile lands once by TMA
// (two 64-column boxes, 128B swizzle) and is read by the tensor core
//   * as a K-major  A operand (M = T rows,   K = out cols)  for dt  (+= against the B tile, N = r),
//   * as an MN-major A operand (M = out cols, K = T rows)   for dB^T (+= against the t tile, N = r).
// HBM-bound: 16 UMMAs (M128 x N64 x K16) per 32 KB of dY, about a third of the tensor pipe at full bandwidth.
//
// Decomposition.  TMEM holds 512 fp32 columns: 2 x 64 for a double-buffered dt accumulator plus 64 per 128-wide
// block of dB^T, i.e. at most 6 blocks = 768 out-columns per CTA.  The out range is therefore cut into G column
// groups of `bpg` blocks, and the G CTAs of one thread-block CLUSTER (G = 1, 2, 4, 8, 16) take one group each while
// walking the same T-chunks (128 rows; cluster k handles chunks k, k + n_clusters, ...):
//   * dB^T of a CTA accumulates in TMEM across all of its chunks and leaves the SM once, as the fp32 partial of split
//     k (summed over the splits in a fixed order by the finalize kernel: bit-reproducible, no atomics); the write is
//     staged through the idle shared-memory ring (128B-swizzled, conflict-free) and written by TMA tensor stores;
//   * dt of a chunk needs all G groups: a reduce-scatter over DISTRIBUTED SHARED MEMORY.  Row i of the chunk is
//     finalised by CTA i % G: every other CTA stores its fp32 partial of that row into the owner's receive buffer
//     (st.shared::cluster) and arrives on the owner's mbarrier; the owner adds the G partials in the fixed order
//     0..G-1, scales, converts and writes the 16-bit row.  No global partials, fences or atomics (the first version
//     exchanged the partials through L2 with a last-arriver counter: 16 k cycles per chunk against a 6 k-cycle main
//     loop, profiles/r02_k2_timeline.txt).
//
// Roles (256 threads): warp 0 lane 0 TMA producer, warp 1 lane 0 UMMA issuer, warp 2 TMEM allocator, warps 4-7 epilogue.
// F16: dY, B, t and dt are IEEE fp16 instead of bf16 (instruction-descriptor format and the dt conversion; TMA maps on
// the host side).  The dB^T partials are fp32 either way.
#pragma once
#include "ptx.cuh"

namespace sowb {

constexpr int kK2Threads = 256;
constexpr int kK2EpiThreads = 128;
constexpr int kK2Stages = 3;
constexpr int kK2DyBytes = 128 * 128 * 2;          // dY tile: 2 boxes of [128 rows x 64 cols]
constexpr int kK2BBytes = 64 * 128 * 2;            // B tile : 2 boxes of [64 r-rows x 64 cols]
constexpr int kK2StageBytes = kK2DyBytes + kK2BBytes;
constexpr int kK2TBytes = 128 * 64 * 2;            // t tile : [128 rows x 64 r-cols]
constexpr int kK2RxBufBytes = 24576;               // one receive buffer for G <= 4: [G-1 sources][128 / G row slots][64] fp32
constexpr int kK2RxBytes = 2 * kK2RxBufBytes;      // double-buffered for G <= 4; one 30 KB buffer for G = 8, 16
constexpr int kK2MaxBpg = 6;
constexpr int kK2MaxG = 16;
constexpr int kK2BarBytes = 256;
constexpr int kK2SmemTotal = 1024 + kK2Stages * kK2StageBytes + 2 * kK2TBytes + kK2RxBytes + kK2BarBytes;
static_assert(kK2SmemTotal <= 232448, "K2 exceeds the 227 KB shared-memory opt-in limit");
static_assert(kK2Stages * kK2StageBytes >= 4 * 8192, "the ring doubles as the dB^T staging area (8 KB per epilogue warp)");

constexpr int kK2MaxMembers = 4;

struct K2MemberMaps {
  CUtensorMap dy;   // dY [T, out]        box 64 cols x 128 rows
  CUtensorMap b;    // B  [r, out]        box 64 cols x 64 rows  (rows >= r read as zero)
  CUtensorMap t;    // t  [T, >= 64]      box 64 cols x 128 rows
  CUtensorMap dbp;  // dB^T partials [n_clusters * out_pad, 64] fp32, box 32 cols x 32 rows (stores)
};
struct K2Maps {
  K2MemberMaps m[kK2MaxMembers];
};

// One launch serves every member of a projection group that shares the cluster size G (q/k/v; gate/up): the clusters
// are PARTITIONED among the members (member i owns clusters [cl_begin[i], cl_begin[i+1])), so a cluster walks ~n times
// more T-chunks of one dY than it would in a per-member launch -- pipeline fill / drain and the dB^T flush are
// amortised over them and every dB^T has n times fewer split partials.
struct K2Member {
  int out, out_pad;         // out_pad: rows per split in the dB^T partial buffer (out rounded up to 128)
  int bpg;                  // 128-col blocks per column group
  int blk_first, blk_end;   // 128-col blocks [blk_first, blk_end) of dY covered by this launch
  int dt_accumulate;        // add onto the dt already in memory (second launch over a very wide `out`)
  float scale;
  void* dt;                 // [T, ldt] 16-bit (this member's / rank chunk's 64 columns)
};
struct K2Params {
  int T, G, n_members;
  int n_chunks;             // ceil(T / 128)
  int ldt;
  int cl_begin[kK2MaxMembers + 1];
  K2Member m[kK2MaxMembers];
  long long* dbg;           // debug timeline (tools/k2_timeline.py): CTA 0 records clock64 stamps [chunk][16], or NULL
};

template <bool F16>
__global__ void __launch_bounds__(kK2Threads, 1)
sow_k2_kernel(const __grid_constant__ K2Maps allmaps, const __grid_constant__ K2Params p) {
  extern __shared__ uint8_t smem_raw[];
  // identical offsets in every CTA of the cluster (mapa translates by offset): align relative to the window base
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* ring = smem;
  uint8_t* tbuf = smem + kK2Stages * kK2StageBytes;
  float* rx = reinterpret_cast<float*>(tbuf + 2 * kK2TBytes);
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(rx) + kK2RxBytes);
  uint64_t* full_bar = bars;                       // [stages]
  uint64_t* empty_bar = bars + kK2Stages;          // [stages]
  uint64_t* t_full = bars + 2 * kK2Stages;         // [2]
  uint64_t* t_empty = t_full + 2;                  // [2]
  uint64_t* dt_full = t_empty + 2;                 // [2]
  uint64_t* dt_empty = dt_full + 2;                // [2]
  uint64_t* db_full = dt_empty + 2;                // [1]
  uint64_t* rx_full = db_full + 1;                 // [2] (G-1) * 128/G remote arrivals per use of the buffer
  uint64_t* rx_credit = rx_full + 2;               // [2] G-1 remote arrivals per use: every peer has consumed its buffer
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(rx_credit + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  auto stamp = [&](int chunk_local, int k) {
    if (p.dbg != nullptr && blockIdx.x == 0 && chunk_local < 64) p.dbg[chunk_local * 16 + k] = clock64();
  };
  if (p.dbg != nullptr && threadIdx.x == 0 && blockIdx.x < 512) {   // per-CTA start time + SM id (debug)
    unsigned long long t;
    unsigned int smid;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    p.dbg[1024 + blockIdx.x * 3] = static_cast<long long>(t);
    p.dbg[1024 + blockIdx.x * 3 + 2] = smid;
  }
  const int G = p.G;
  const int g = (G > 1) ? static_cast<int>(cluster_ctarank()) : 0;
  const int cluster = (G > 1) ? static_cast<int>(cluster_id_x()) : static_cast<int>(blockIdx.x);
  int mi = 0;
  while (mi + 1 < p.n_members && cluster >= p.cl_begin[mi + 1]) ++mi;
  const K2Member& M = p.m[mi];
  const K2MemberMaps& maps = allmaps.m[mi];
  const int split = cluster - p.cl_begin[mi];                  // this cluster's index among the member's clusters
  const int n_clusters = p.cl_begin[mi + 1] - p.cl_begin[mi];
  const int blk0 = M.blk_first + g * M.bpg;                     // first 128-col block of this group
  const int nblk = max(0, min(M.bpg, M.blk_end - blk0));       // blocks this CTA owns (0: only helps with nothing)
  const int rows_per = 128 / G;                                // rows of a chunk finalised by each CTA

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&maps.dy);
    tma_prefetch_desc(&maps.b);
    tma_prefetch_desc(&maps.t);
    tma_prefetch_desc(&maps.dbp);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < kK2Stages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&t_full[i], 1);
      mbar_init(&t_empty[i], 1);
      mbar_init(&dt_full[i], 1);
      mbar_init(&dt_empty[i], kK2EpiThreads);
    }
    mbar_init(db_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&rx_full[i], G > 1 ? (G - 1) * rows_per : 1);
      mbar_init(&rx_credit[i], G > 1 ? (G - 1) : 1);
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  if (G > 1) cluster_sync_all();     // peers' barriers are initialised before anyone arrives on them remotely
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // TMEM columns: [0,128) two dt accumulators, [128 + 64 j, +64) dB^T block j

  if (warp == 0 && lane == 0) {
    // ===================== TMA producer =====================
    int stage = 0, tb = 0;
    uint32_t phase = 0, tphase = 0;
    int cl = 0;
    for (int c = split; c < p.n_chunks; c += n_clusters, ++cl) {
      const int row0 = c * 128;
      stamp(cl, 0);
      if (nblk > 0) {
        mbar_wait(&t_empty[tb], tphase ^ 1);
        mbar_expect_tx(&t_full[tb], kK2TBytes);
        tma_load_2d(tbuf + tb * kK2TBytes, &maps.t, &t_full[tb], 0, row0);
      }
      for (int j = 0; j < nblk; ++j) {
        const int n0 = (blk0 + j) * 128;
        mbar_wait(&empty_bar[stage], phase ^ 1);
        uint8_t* sdy = ring + stage * kK2StageBytes;
        uint8_t* sb = sdy + kK2DyBytes;
        mbar_expect_tx(&full_bar[stage], kK2StageBytes);
        tma_load_2d(sdy, &maps.dy, &full_bar[stage], n0, row0);
        tma_load_2d(sdy + 16384, &maps.dy, &full_bar[stage], n0 + 64, row0);
        tma_load_2d(sb, &maps.b, &full_bar[stage], n0, 0);
        tma_load_2d(sb + 8192, &maps.b, &full_bar[stage], n0 + 64, 0);
        if (++stage == kK2Stages) {
          stage = 0;
          phase ^= 1;
        }
      }
      stamp(cl, 2);
      if (++tb == 2) {
        tb = 0;
        tphase ^= 1;
      }
    }
  } else if (warp == 1 && lane == 0) {
    // ===================== UMMA issuer =====================
    constexpr uint32_t idesc_dt = make_idesc(ab_format16<F16>(), 128, 64, 0, 0);   // A K-major (dY), B K-major (B rows = r)
    constexpr uint32_t idesc_db = make_idesc(ab_format16<F16>(), 128, 64, 1, 1);   // A MN-major (dY^T), B MN-major (t)
    int stage = 0, tb = 0, acc = 0;
    uint32_t phase = 0, tphase = 0, aphase = 0;
    bool first_chunk = true;
    int cl = 0;
    if (nblk > 0) {
      for (int c = split; c < p.n_chunks; c += n_clusters, ++cl) {
        stamp(cl, 3);
        mbar_wait(&t_full[tb], tphase);
        mbar_wait(&dt_empty[acc], aphase ^ 1);
        stamp(cl, 5);
        tc_fence_after();
        const uint32_t st = smem_u32(tbuf + tb * kK2TBytes);
        const uint32_t d_dt = tmem_base + acc * 64;
        for (int j = 0; j < nblk; ++j) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sdy = smem_u32(ring + stage * kK2StageBytes);
          const uint32_t sb = sdy + kK2DyBytes;
          // dt += dY_tile . B_tile^T : per 64-col box, 4 UMMAs of K = 16 (32 B inside the 128 B swizzle span)
#pragma unroll
          for (int box = 0; box < 2; ++box) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const uint64_t ad = make_smem_desc(sdy + box * 16384 + k * 32, 16, 1024);
              const uint64_t bd = make_smem_desc(sb + box * 8192 + k * 32, 16, 1024);
              umma_bf16(d_dt, ad, bd, idesc_dt, (j > 0 || box > 0 || k > 0) ? 1u : 0u);
            }
          }
          // dB^T block j += dY_tile^T . t_tile : K = 128 T-rows = 8 UMMAs; 16 rows of 128 B = 2048 B per K step;
          // the two 64-wide M blocks (boxes) are LBO = 16384 B apart
          const uint32_t d_db = tmem_base + 128 + j * 64;
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            const uint64_t ad = make_smem_desc(sdy + k * 2048, 16384, 1024);
            const uint64_t bd = make_smem_desc(st + k * 2048, 16384, 1024);
            umma_bf16(d_db, ad, bd, idesc_db, (!first_chunk || k > 0) ? 1u : 0u);
          }
          umma_commit(&empty_bar[stage]);
          if (++stage == kK2Stages) {
            stage = 0;
            phase ^= 1;
          }
        }
        umma_commit(&dt_full[acc]);
        umma_commit(&t_empty[tb]);
        stamp(cl, 6);
        first_chunk = false;
        if (++tb == 2) {
          tb = 0;
          tphase ^= 1;
        }
        if (++acc == 2) {
          acc = 0;
          aphase ^= 1;
        }
      }
      umma_commit(db_full);
    }
  } else if (warp >= 4) {
    // ===================== epilogue =====================
    const int q = warp - 4;
    const int rit = q * 32 + lane;              // row inside the 128-row tile == TMEM lane
    const int et = threadIdx.x - 128;
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const int owner = rit % G;                  // CTA of the cluster that finalises this row
    const int slot = rit / G;
    // receive buffers: [source CTA, own rank skipped][16-byte chunk of the row (16)][row slot] float4 -- the lanes of one
    // st.shared::cluster instruction write CONSECUTIVE 16-byte chunks (DSMEM wants coalesced traffic like global
    // memory; a row-major layout, 256 B between lanes, measured 3x slower); two buffers when they fit (G <= 4), so
    // that a CTA can send chunk c+1 while the owner is still summing chunk c
    const int nbuf = (G <= 4) ? 2 : 1;
    const uint32_t rx_local = smem_u32(rx);
    const int src_idx = g < owner ? g : g - 1;     // my index among the owner's sources
    const uint32_t rx_dst = (G > 1) ? map_to_cta(rx_local + static_cast<uint32_t>((src_idx * 16 * rows_per + slot) * 16), owner) : 0u;
    const uint32_t chunk_pitch = static_cast<uint32_t>(rows_per) * 16u;
    const uint32_t full_dst = (G > 1) ? map_to_cta(smem_u32(rx_full), owner) : 0u;
    int acc = 0;
    uint32_t aphase = 0, rphase = 0, cphase = 0;   // rphase / cphase: one parity bit per receive buffer
    int cl = 0;
    for (int c = split; c < p.n_chunks; c += n_clusters, ++cl) {
      if (et == 0) stamp(cl, 7);
      float v[64];
      if (nblk > 0) {
        mbar_wait(&dt_full[acc], aphase);
        tc_fence_after();
        uint32_t v0[32], v1[32];
        tmem_ld32(lane_addr + acc * 64, v0);
        tmem_ld32(lane_addr + acc * 64 + 32, v1);
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive(&dt_empty[acc]);
        if (++acc == 2) {
          acc = 0;
          aphase ^= 1;
        }
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          v[i] = __uint_as_float(v0[i]);
          v[32 + i] = __uint_as_float(v1[i]);
        }
      } else {
#pragma unroll
        for (int i = 0; i < 64; ++i) v[i] = 0.f;
      }
      if (et == 0) stamp(cl, 8);
      const int row = c * 128 + rit;
      if (G > 1) {
        const int buf = (nbuf == 2) ? (cl & 1) : 0;
        // every peer has summed the chunk that used this buffer last out of it
        if (cl >= nbuf) {
          mbar_wait_cluster(&rx_credit[buf], (cphase >> buf) & 1u);
          cphase ^= 1u << buf;
        }
        if (owner != g) {
          const uint32_t dst = rx_dst + buf * kK2RxBufBytes;
#pragma unroll
          for (int i = 0; i < 16; ++i) st_cluster_f32x4(dst + i * chunk_pitch, v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
          mbar_arrive_remote(full_dst + buf * 8);
        }
        if (et == 0) stamp(cl, 9);
        if (owner == g) {
          mbar_wait_cluster(&rx_full[buf], (rphase >> buf) & 1u);
          // fixed summation order 0..G-1 whatever the arrival order: bit-reproducible
          float s[64];
#pragma unroll
          for (int i = 0; i < 64; ++i) s[i] = 0.f;
          for (int gg = 0; gg < G; ++gg) {
            if (gg == g) {
#pragma unroll
              for (int i = 0; i < 64; ++i) s[i] += v[i];
            } else {
              const float4* src = reinterpret_cast<const float4*>(
                  reinterpret_cast<const uint8_t*>(rx) + buf * kK2RxBufBytes + ((gg < g ? gg : gg - 1) * 16 * rows_per + slot) * 16);
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                const float4 x = src[i * rows_per];
                s[4 * i] += x.x;
                s[4 * i + 1] += x.y;
                s[4 * i + 2] += x.z;
                s[4 * i + 3] += x.w;
              }
            }
          }
#pragma unroll
          for (int i = 0; i < 64; ++i) v[i] = s[i];
        }
        rphase ^= 1u << buf;
        if (et == 0) stamp(cl, 10);
      }
      if (owner == g && row < p.T) {
        uint4* dst = reinterpret_cast<uint4*>(static_cast<uint16_t*>(M.dt) + static_cast<int64_t>(row) * p.ldt);
#pragma unroll
        for (int ch = 0; ch < 8; ++ch) {
          float f[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) f[i] = M.scale * v[8 * ch + i];
          if (M.dt_accumulate) {
            const uint4 old = dst[ch];
            const uint32_t ow[4] = {old.x, old.y, old.z, old.w};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              f[2 * i] += lo16_to_f32<F16>(ow[i]);
              f[2 * i + 1] += hi16_to_f32<F16>(ow[i]);
            }
          }
          uint4 pk;
          pk.x = pack16x2<F16>(f[0], f[1]);
          pk.y = pack16x2<F16>(f[2], f[3]);
          pk.z = pack16x2<F16>(f[4], f[5]);
          pk.w = pack16x2<F16>(f[6], f[7]);
          dst[ch] = pk;
        }
      }
      if (G > 1) {
        // this CTA's receive buffer is free again: tell every peer (one arrival per peer CTA)
        named_barrier_sync(1, kK2EpiThreads);
        if (et < G && et != g) mbar_arrive_remote(map_to_cta(smem_u32(&rx_credit[(nbuf == 2) ? (cl & 1) : 0]), et));
      }
      if (et == 0) stamp(cl, 11);
    }
    // dB^T partial of this split: rows = out columns of the group's blocks; staged through the (now idle) ring as
    // one contiguous 8 KB block per warp and written with a bulk copy
    if (nblk > 0) {
      if (et == 0) stamp(63, 0);
      mbar_wait(db_full, 0);
      tc_fence_after();
      if (et == 0) stamp(63, 1);
      uint8_t* stg = ring + q * 8192;       // two [32 rows x 128 B] boxes, 128B-swizzled like the tensor map expects
      for (int j = 0; j < nblk; ++j) {
        uint32_t v0[32], v1[32];
        tmem_ld32(lane_addr + 128 + j * 64, v0);
        tmem_ld32(lane_addr + 128 + j * 64 + 32, v1);
        tmem_ld_wait();
        if (j > 0) {
          if (lane == 0) tma_store_wait_read<0>();     // the previous block's stores have read the staging area
          __syncwarp();
        }
#pragma unroll
        for (int ch = 0; ch < 8; ++ch) {
          const int sw = (ch ^ (lane & 7)) << 4;       // conflict-free: 8 lanes cover the 32 banks
          *reinterpret_cast<uint4*>(stg + lane * 128 + sw) = make_uint4(v0[4 * ch], v0[4 * ch + 1], v0[4 * ch + 2], v0[4 * ch + 3]);
          *reinterpret_cast<uint4*>(stg + 4096 + lane * 128 + sw) = make_uint4(v1[4 * ch], v1[4 * ch + 1], v1[4 * ch + 2], v1[4 * ch + 3]);
        }
        fence_proxy_async_smem();
        __syncwarp();
        const int o0 = (blk0 + j) * 128 + q * 32;
        if (lane == 0 && o0 < M.out) {
          const int row = split * M.out_pad + o0;
          tma_store_2d(&maps.dbp, stg, 0, row);
          tma_store_2d(&maps.dbp, stg + 4096, 32, row);
          tma_store_commit();
        }
      }
      if (lane == 0) tma_store_wait_all<0>();
      if (et == 0) stamp(63, 2);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (G > 1) cluster_sync_all();     // no CTA exits while a peer may still write into its shared memory
  tc_fence_after();
  if (warp == 2) tmem_dealloc(tmem_base, 512);
  if (p.dbg != nullptr && threadIdx.x == 0 && blockIdx.x < 512) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    p.dbg[1024 + blockIdx.x * 3 + 1] = static_cast<long long>(t);
  }
}

}  // namespace sowb
