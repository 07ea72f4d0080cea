// Order-2 TT-Adam on the tensor cores (tcgen05 / TMEM / TMA): Adam update + re-compression in one pass over p and g.
//
// Per element the step needs two rank-r products -- the reconstruction of the old moments from the cores,
// m = G1m.G2m and v = G1v.G2v, and the projection of the new moments onto the new bases, R' = Q'^T m' -- 8.r flop per
// element, which at r = 64 is 8x more fp32 FMA time than HBM time.  Both products therefore run as bf16 UMMAs on
// operands split into three bf16 pieces (x = x0 + x1 + x2, 24 mantissa bits; products x_i.y_j with i + j <= 2, fp32
// accumulation in TMEM), which is fp32-accurate -- plain bf16 or TF32 would break the 1e-5 reconstruction criterion.
//
// CTA = (strip of 128 columns of the P x P interleaved moment matrix, range of 128-row tiles).  Per tile:
//   1. TMA: pieces of G1{m,v}[tile rows] and G2{m,v}[:, strip]; 6 x ksteps UMMAs each -> S_m, S_v (128x128 fp32, TMEM)
//   2. epilogue A (thread per row, 64 columns per thread): S_m, S_v from TMEM, g and p from HBM (16-byte vectors),
//      Adam (ttadam.py:84-111), p written back, m' split into bf16 pieces -> shared memory as the MN-major A operand
//   3. UMMA: D_m[128 cols x 64] += m'^T . Q'm[tile rows]   (pieces of Q' loaded by TMA, accumulated over the tiles)
//   4. epilogue B: v' recomputed from S_v and g (keeping both moments' operand tiles would not fit 227 KB), pieces,
//      UMMA: D_v += v'^T . Q'v
// At the end of the range D_m, D_v are stored as that range's partial of R'{m,v}[r, P] (summed in range order by
// sum_splits_kernel: bit-reproducible).  The dense moments never exist in HBM.
// This first version is phase-serial inside a CTA (one thread issues TMA and UMMAs, everybody waits on the mbarriers);
// the next step is to overlap the phases of consecutive tiles.
#include "common.cuh"
#include "ptx.cuh"

#include <algorithm>
#include <stdlib.h>

namespace sowb {

constexpr int kTcTile = 128;
constexpr int kTcThreads = 256;
constexpr int kTcOpBytes = 96 * 1024;    // phase 1: G1 pieces 48 KB + G2 pieces 48 KB; phase 2: 3 pieces of m'/v' (32 KB each)
constexpr int kTcQBytes = 96 * 1024;     // Q'm pieces 48 KB + Q'v pieces 48 KB
constexpr int kTcSmem = 1024 + kTcOpBytes + kTcQBytes + 128;
constexpr uint32_t kTcTmemCols = 512;

// x -> three bf16 pieces, written to dst[piece][rows_pad][cols_pad] (zero outside the source extent).  Up to six
// operand arrays (old cores and new bases of both moments) in ONE launch: blockIdx.y selects the job.
struct SplitJobs {
  const float* src[6];
  __nv_bfloat16* dst[6];
  int rows[6], cols[6], ld[6], rows_pad[6], cols_pad[6];
};

__global__ void tt_split3_kernel(const __grid_constant__ SplitJobs jobs) {
  pdl_trigger();
  pdl_wait();
  const int jb = blockIdx.y;
  const float* __restrict__ src = jobs.src[jb];
  __nv_bfloat16* __restrict__ dst = jobs.dst[jb];
  const int rows = jobs.rows[jb], cols = jobs.cols[jb], ld = jobs.ld[jb], cols_pad = jobs.cols_pad[jb];
  const int64_t n = static_cast<int64_t>(jobs.rows_pad[jb]) * cols_pad;
  for (int64_t idx = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; idx < n;
       idx += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int i = static_cast<int>(idx / cols_pad), j = static_cast<int>(idx - static_cast<int64_t>(i) * cols_pad);
    float x = (i < rows && j < cols) ? src[static_cast<int64_t>(i) * ld + j] : 0.f;
    const __nv_bfloat16 b0 = __float2bfloat16(x);
    x -= __bfloat162float(b0);
    const __nv_bfloat16 b1 = __float2bfloat16(x);
    x -= __bfloat162float(b1);
    const __nv_bfloat16 b2 = __float2bfloat16(x);
    dst[idx] = b0;
    dst[n + idx] = b1;
    dst[2 * n + idx] = b2;
  }
}

// MUFU square root / reciprocal (<= 2 ulp each): the update term is scaled by the step size before it meets p (same choice
// and same trajectory bound as tt_adam2_reg_kernel)
__device__ __forceinline__ float sqrt_approx(float x) {
  float y;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ void split3(float x, uint16_t& b0, uint16_t& b1, uint16_t& b2) {
  const __nv_bfloat16 h0 = __float2bfloat16(x);
  x -= __bfloat162float(h0);
  const __nv_bfloat16 h1 = __float2bfloat16(x);
  x -= __bfloat162float(h1);
  const __nv_bfloat16 h2 = __float2bfloat16(x);
  b0 = __bfloat16_as_ushort(h0);
  b1 = __bfloat16_as_ushort(h1);
  b2 = __bfloat16_as_ushort(h2);
}

template <typename T>
__device__ __forceinline__ void load8(const T* p, int64_t i, float (&v)[8]);
template <>
__device__ __forceinline__ void load8<float>(const float* p, int64_t i, float (&v)[8]) {
  const float4 a = *reinterpret_cast<const float4*>(p + i), b = *reinterpret_cast<const float4*>(p + i + 4);
  v[0] = a.x, v[1] = a.y, v[2] = a.z, v[3] = a.w, v[4] = b.x, v[5] = b.y, v[6] = b.z, v[7] = b.w;
}
template <>
__device__ __forceinline__ void load8<__nv_bfloat16>(const __nv_bfloat16* p, int64_t i, float (&v)[8]) {
  const uint4 t = *reinterpret_cast<const uint4*>(p + i);
  const uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    v[2 * j] = __uint_as_float(w[j] << 16);
    v[2 * j + 1] = __uint_as_float(w[j] & 0xffff0000u);
  }
}
template <typename T>
__device__ __forceinline__ void store8(T* p, int64_t i, const float (&v)[8]);
template <>
__device__ __forceinline__ void store8<float>(float* p, int64_t i, const float (&v)[8]) {
  *reinterpret_cast<float4*>(p + i) = make_float4(v[0], v[1], v[2], v[3]);
  *reinterpret_cast<float4*>(p + i + 4) = make_float4(v[4], v[5], v[6], v[7]);
}
template <>
__device__ __forceinline__ void store8<__nv_bfloat16>(__nv_bfloat16* p, int64_t i, const float (&v)[8]) {
  uint4 t;
  t.x = pack_bf16x2(v[0], v[1]);
  t.y = pack_bf16x2(v[2], v[3]);
  t.z = pack_bf16x2(v[4], v[5]);
  t.w = pack_bf16x2(v[6], v[7]);
  *reinterpret_cast<uint4*>(p + i) = t;
}
template <typename T>
__device__ __forceinline__ float load1(const T* p, int64_t i);
template <>
__device__ __forceinline__ float load1<float>(const float* p, int64_t i) { return p[i]; }
template <>
__device__ __forceinline__ float load1<__nv_bfloat16>(const __nv_bfloat16* p, int64_t i) { return __bfloat162float(p[i]); }
template <typename T>
__device__ __forceinline__ void store1(T* p, int64_t i, float v);
template <>
__device__ __forceinline__ void store1<float>(float* p, int64_t i, float v) { p[i] = v; }
template <>
__device__ __forceinline__ void store1<__nv_bfloat16>(__nv_bfloat16* p, int64_t i, float v) { p[i] = __float2bfloat16(v); }

// 8 consecutive elements as raw 16-byte loads (issued early, unpacked late)
template <typename T>
struct Raw8;
template <>
struct Raw8<__nv_bfloat16> {
  uint4 a;
  __device__ __forceinline__ void load(const __nv_bfloat16* p, int64_t i) { a = *reinterpret_cast<const uint4*>(p + i); }
  __device__ __forceinline__ void unpack(float (&v)[8]) const {
    const uint32_t w[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      v[2 * j] = __uint_as_float(w[j] << 16);
      v[2 * j + 1] = __uint_as_float(w[j] & 0xffff0000u);
    }
  }
};
template <>
struct Raw8<float> {
  float4 a, b;
  __device__ __forceinline__ void load(const float* p, int64_t i) {
    a = *reinterpret_cast<const float4*>(p + i);
    b = *reinterpret_cast<const float4*>(p + i + 4);
  }
  __device__ __forceinline__ void unpack(float (&v)[8]) const {
    v[0] = a.x, v[1] = a.y, v[2] = a.z, v[3] = a.w, v[4] = b.x, v[5] = b.y, v[6] = b.z, v[7] = b.w;
  }
};
// register-resident 8-entry tables indexed by a run-time chunk number (a select chain instead of local memory)
__device__ __forceinline__ int col_i2(const int (&t)[8], int c) {
  int v = t[0];
#pragma unroll
  for (int k = 1; k < 8; ++k) v = (c == k) ? t[k] : v;
  return v;
}
__device__ __forceinline__ int col_o2(const int (&t)[8], int c) { return col_i2(t, c); }

struct TcParams {
  int M, N, mm, nn, P, P_pad, r;
  float beta1, omb1, beta2, omb2, eps, step_size, lr_wd;
  int first_step, tiles_per_cta;
  float* Rm;             // results (one split) or the split partials [split][r][P] of each moment
  float* Rv;
  int64_t split_stride;  // r * P when the row-range splits store partials, else 0
  long long* dbg;   // debug timeline (clock64 stamps of CTA (0,0), 8 per tile) or nullptr
};

template <typename T>
__global__ void __launch_bounds__(kTcThreads, 1)
tt_adam2_tc_kernel(const __grid_constant__ CUtensorMap tmG1m, const __grid_constant__ CUtensorMap tmG1v,
                   const __grid_constant__ CUtensorMap tmG2m, const __grid_constant__ CUtensorMap tmG2v,
                   const __grid_constant__ CUtensorMap tmQm, const __grid_constant__ CUtensorMap tmQv,
                   T* __restrict__ p, const T* __restrict__ g, const TcParams prm) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sOp = smem;
  uint8_t* sQ = smem + kTcOpBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sQ + kTcQBytes);
  uint64_t* bar_ld = bars;        // TMA: core pieces landed
  uint64_t* bar_q = bars + 1;     // TMA: Q' pieces landed
  uint64_t* bar_mma = bars + 2;   // UMMA batch complete
  uint64_t* bar_ld2 = bars + 3;   // TMA: second moment's core pieces landed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int P = prm.P, nn = prm.nn, mm = prm.mm, M = prm.M, N = prm.N;
  if (tid == 0) {
    tma_prefetch_desc(&tmG1m);
    tma_prefetch_desc(&tmG1v);
    tma_prefetch_desc(&tmG2m);
    tma_prefetch_desc(&tmG2v);
    tma_prefetch_desc(&tmQm);
    tma_prefetch_desc(&tmQv);
    mbar_init(bar_ld, 1);
    mbar_init(bar_ld2, 1);
    mbar_init(bar_q, 1);
    mbar_init(bar_mma, 1);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, kTcTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_trigger();
  pdl_wait();       // barriers, tensor-map prefetch and the TMEM allocation overlap the predecessor's tail
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tS_m = tmem_base, tS_v = tmem_base + 128, tD_m = tmem_base + 256, tD_v = tmem_base + 320;

  const int b0 = blockIdx.x * kTcTile;
  const int n_tiles = (P + kTcTile - 1) / kTcTile;
  const int t_begin = blockIdx.y * prm.tiles_per_cta;
  const int t_end = min(n_tiles, t_begin + prm.tiles_per_cta);
  const int ksteps1 = (prm.r + 15) >> 4;                       // UMMA K = 16 steps covering the rank

  // epilogue mapping: row of the tile = TMEM lane, 64-column half per warp group
  const int q = warp & 3, half = warp >> 2;
  const int rloc = q * 32 + lane;                              // 0..127
  const uint32_t lane_off = static_cast<uint32_t>(q * 32) << 16;
  // column decode (strip-constant): 8 chunks of 8 consecutive columns
  int ci2[8], co2[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    const int gb = b0 + half * 64 + c * 8;
    ci2[c] = gb / nn;
    co2[c] = gb - ci2[c] * nn;
  }
  const bool vec_ok = (nn % 8 == 0) && (N % 8 == 0);

  uint32_t ph_ld = 0, ph_q = 0, ph_mma = 0;
  constexpr uint32_t idesc1 = make_idesc(1, 128, 128, 0, 1);   // S = G1 (K-major) . G2 (MN-major)
  constexpr uint32_t idesc2 = make_idesc(1, 128, 64, 1, 1);    // D = M'^T (MN-major A) . Q' (MN-major B)
  const uint32_t sOp_u = smem_u32(sOp), sQ_u = smem_u32(sQ);

  auto stamp = [&](int t, int k) {
    if (prm.dbg != nullptr && blockIdx.x == 0 && blockIdx.y == 0 && tid == 0 && t - t_begin < 64) prm.dbg[(t - t_begin) * 8 + k] = clock64();
  };
  // CTAs of different strips read the same core / Q' rows: start each strip at a different row tile so that they do not
  // hit the same L2 lines at the same time (the projection sum is order-independent)
  const int n_local = t_end - t_begin;
  for (int it = 0; it < n_local; ++it) {
    const int t = t_begin + (it + static_cast<int>(blockIdx.x)) % n_local;
    const int a0 = t * kTcTile;
    stamp(t_begin + it, 0);
    const int ga = a0 + rloc;
    const int i1 = ga / nn, o1 = ga - i1 * nn;
    const int64_t rowbase = static_cast<int64_t>(i1) * mm * N + static_cast<int64_t>(o1) * nn;
    const int rlim = (ga < P) ? M - i1 * mm : 0;       // element valid iff i2 < rlim && o2 < clim
    const int clim = N - o1 * nn;
    // validity mask / vector flag of one 8-column chunk of this thread's row, and its (early) 16-byte loads
    auto chunk_mask = [&](int c, int bi2, int bo2, bool& vec) -> uint32_t {
      const int gb = b0 + half * 64 + c * 8;
      uint32_t m = 0;
      if (bo2 + 7 < nn) {
        // the chunk lies inside one nn-block (always, when nn % 8 == 0): one row test, a prefix of valid columns
        const int cnt = min(min(clim - bo2, P - gb), 8);
        m = (bi2 < rlim && cnt > 0) ? ((1u << cnt) - 1u) : 0u;
      } else {
#pragma unroll 1
        for (int e = 0; e < 8; ++e) {                  // chunk straddles an nn-block (only when nn % 8 != 0)
          int i2 = bi2, o2 = bo2 + e;
          const int carry = o2 / nn;
          i2 += carry;
          o2 -= carry * nn;
          if ((gb + e < P) && i2 < rlim && o2 < clim) m |= 1u << e;
        }
      }
      const int64_t e0 = rowbase + static_cast<int64_t>(bi2) * N + bo2;
      vec = vec_ok && m == 0xffu && (bo2 + 7 < nn) && ((e0 & 7) == 0);
      return m;
    };
    // 16-bit parameters: the whole row (8 chunks of g and p = 64 registers) is requested BEFORE the reconstruction
    // phase, so the HBM round trip hides behind the TMA loads and UMMAs; pass 1 reuses the g registers
    constexpr bool kPrefetchRow = sizeof(T) == 2;
    Raw8<T> grow[kPrefetchRow ? 8 : 1], prow[kPrefetchRow ? 8 : 1];
    uint32_t mrow[kPrefetchRow ? 8 : 1];
    uint32_t vrow = 0;                                  // bit c: chunk c takes the vector path
    if constexpr (kPrefetchRow) {
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        bool vec;
        mrow[c] = chunk_mask(c, ci2[c], co2[c], vec);
        if (vec) {
          const int64_t e0 = rowbase + static_cast<int64_t>(ci2[c]) * N + co2[c];
          grow[c].load(g, e0);
          prow[c].load(p, e0);
          vrow |= 1u << c;
        }
      }
    }
    // ---------------- 1. loads + reconstruction UMMAs (one thread) ----------------
    if (tid == 0) {
      if (!prm.first_step) {
        // both moments' core pieces at once: m into the operand region, v into the (still idle) Q' region -- one barrier per
        // moment, so that the reconstruction MMAs of m run while the pieces of v are still landing
        mbar_expect_tx(bar_ld, kTcOpBytes);
        mbar_expect_tx(bar_ld2, kTcOpBytes);
#pragma unroll
        for (int mom = 0; mom < 2; ++mom) {
          const CUtensorMap* m1 = mom ? &tmG1v : &tmG1m;
          const CUtensorMap* m2 = mom ? &tmG2v : &tmG2m;
          uint8_t* base = mom ? sQ : sOp;
          uint64_t* bar = mom ? bar_ld2 : bar_ld;
#pragma unroll
          for (int pc = 0; pc < 3; ++pc) {
            tma_load_2d(base + pc * 16384, m1, bar, 0, pc * prm.P_pad + a0);
            tma_load_2d(base + 49152 + pc * 16384, m2, bar, b0, pc * 64);
            tma_load_2d(base + 49152 + pc * 16384 + 8192, m2, bar, b0 + 64, pc * 64);
          }
        }
#pragma unroll
        for (int mom = 0; mom < 2; ++mom) {
          mbar_wait(mom ? bar_ld2 : bar_ld, ph_ld);
          tc_fence_after();
          const uint32_t tS = mom ? tS_v : tS_m;
          const uint32_t ob = mom ? sQ_u : sOp_u;
          bool first = true;
#pragma unroll
          for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j) {
              if (i + j > 2) continue;
              for (int k = 0; k < ksteps1; ++k) {
                const uint64_t ad = make_smem_desc(ob + i * 16384 + k * 32, 16, 1024);
                const uint64_t bd = make_smem_desc(ob + 49152 + j * 16384 + k * 2048, 8192, 1024);
                umma_bf16(tS, ad, bd, idesc1, first ? 0u : 1u);
                first = false;
              }
            }
        }
        ph_ld ^= 1;
        umma_commit(bar_mma);
        mbar_wait(bar_mma, ph_mma);     // both operand regions are overwritten next (m' pieces / Q' pieces)
        ph_mma ^= 1;
      }
      // the Q' pieces of this row tile land while the Adam epilogue runs
      mbar_expect_tx(bar_q, kTcQBytes);
#pragma unroll
      for (int pc = 0; pc < 3; ++pc) {
        tma_load_2d(sQ + pc * 16384, &tmQm, bar_q, 0, pc * prm.P_pad + a0);
        tma_load_2d(sQ + 49152 + pc * 16384, &tmQv, bar_q, 0, pc * prm.P_pad + a0);
      }
    }
    __syncthreads();
    __syncwarp();                 // lane 0 of warp 0 diverged above; tcgen05.ld is .sync.aligned
    tc_fence_after();
    stamp(t_begin + it, 1);

    // ---------------- 2./4. epilogues: pass 0 = Adam + m' pieces, pass 1 = v' pieces ----------------
#pragma unroll 1
    for (int pass = 0; pass < 2; ++pass) {
#pragma unroll 1
      for (int h32 = 0; h32 < 2; ++h32) {              // 32 columns at a time (register budget)
        // ---- A. issue every global load of this half row first: the HBM round trip is paid once, not per chunk ----
        Raw8<T> graw[4], praw[4];
        uint32_t okmask[4];
        bool vecf[4];
#pragma unroll
        for (int c4 = 0; c4 < 4; ++c4) {
          if constexpr (kPrefetchRow) {
            graw[c4] = h32 ? grow[c4 + 4] : grow[c4];
            praw[c4] = h32 ? prow[c4 + 4] : prow[c4];
            okmask[c4] = h32 ? mrow[c4 + 4] : mrow[c4];
            vecf[c4] = (vrow >> (h32 * 4 + c4)) & 1u;
          } else {
            const int bi2 = h32 ? ci2[c4 + 4] : ci2[c4], bo2 = h32 ? co2[c4 + 4] : co2[c4];
            okmask[c4] = chunk_mask(h32 * 4 + c4, bi2, bo2, vecf[c4]);
            if (vecf[c4]) {
              const int64_t e0 = rowbase + static_cast<int64_t>(bi2) * N + bo2;
              graw[c4].load(g, e0);
              if (pass == 0) praw[c4].load(p, e0);
            }
          }
        }
        uint32_t sm[32], sv[32];
#pragma unroll
        for (int k = 0; k < 32; ++k) sm[k] = sv[k] = 0u;
        if (!prm.first_step) {
          if (pass == 0) tmem_ld32(tS_m + lane_off + half * 64 + h32 * 32, sm);
          tmem_ld32(tS_v + lane_off + half * 64 + h32 * 32, sv);
          tmem_ld_wait();
        }
        // ---- B. per chunk: Adam, write-back, operand pieces ----
#pragma unroll
        for (int c4 = 0; c4 < 4; ++c4) {
          const int c = h32 * 4 + c4;
          const int bi2 = h32 ? ci2[c4 + 4] : ci2[c4], bo2 = h32 ? co2[c4 + 4] : co2[c4];
          const uint32_t okm = okmask[c4];
          // MN-major A operand tiles [piece][k-block][M-block][64 rows][128 B]: this thread's 16-byte chunk of its row
          uint8_t* dst = sOp + (rloc >> 6) * 16384 + half * 8192 + (rloc & 63) * 128 + ((c ^ (rloc & 7)) << 4);
          if (vecf[c4]) {
            const int64_t e0 = rowbase + static_cast<int64_t>(bi2) * N + bo2;
            float gv[8], pv[8];
            graw[c4].unpack(gv);
            if (pass == 0) praw[c4].unpack(pv);
            uint16_t b[3][8];
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              const float mp = __uint_as_float(sm[c4 * 8 + e]);
              const float vp = fmaxf(__uint_as_float(sv[c4 * 8 + e]), 0.f);                          // ttadam.py:84
              const float vo = prm.beta2 * vp + prm.omb2 * gv[e] * gv[e];                            // ttadam.py:93
              if (pass == 0) {
                const float mo = prm.beta1 * mp + prm.omb1 * gv[e];                                  // ttadam.py:92
                pv[e] -= prm.step_size * mo * rcp_approx(sqrt_approx(vo) + prm.eps);                        // ttadam.py:94,103,108
                if (prm.lr_wd > 0.f) pv[e] -= prm.lr_wd * pv[e];                                     // ttadam.py:110-111
                split3(mo, b[0][e], b[1][e], b[2][e]);
              } else {
                split3(vo, b[0][e], b[1][e], b[2][e]);
              }
            }
            if (pass == 0) store8<T>(p, e0, pv);
#pragma unroll
            for (int pc = 0; pc < 3; ++pc) {
              uint4 w;
              w.x = b[pc][0] | (static_cast<uint32_t>(b[pc][1]) << 16);
              w.y = b[pc][2] | (static_cast<uint32_t>(b[pc][3]) << 16);
              w.z = b[pc][4] | (static_cast<uint32_t>(b[pc][5]) << 16);
              w.w = b[pc][6] | (static_cast<uint32_t>(b[pc][7]) << 16);
              *reinterpret_cast<uint4*>(dst + pc * 32768) = w;
            }
          } else {
            // ragged chunk (matrix edge, or nn % 8 != 0): element by element, compact code
#pragma unroll 1
            for (int e = 0; e < 8; ++e) {
              float mp = 0.f, vp = 0.f;
#pragma unroll
              for (int k = 0; k < 8; ++k) {           // register-file select instead of a dynamically indexed array
                mp = (k == e) ? __uint_as_float(sm[c4 * 8 + k]) : mp;
                vp = (k == e) ? __uint_as_float(sv[c4 * 8 + k]) : vp;
              }
              float mo = 0.f, vo = 0.f;
              if ((okm >> e) & 1u) {
                int i2 = bi2, o2 = bo2 + e;
                const int carry = o2 / nn;
                i2 += carry;
                o2 -= carry * nn;
                const int64_t ee = rowbase + static_cast<int64_t>(i2) * N + o2;
                const float gv = load1<T>(g, ee);
                mo = prm.beta1 * mp + prm.omb1 * gv;
                vo = prm.beta2 * fmaxf(vp, 0.f) + prm.omb2 * gv * gv;
                if (pass == 0) {
                  float pv = load1<T>(p, ee);
                  pv -= prm.step_size * mo * rcp_approx(sqrt_approx(vo) + prm.eps);
                  if (prm.lr_wd > 0.f) pv -= prm.lr_wd * pv;
                  store1<T>(p, ee, pv);
                }
              }
              uint16_t q0, q1, q2;
              split3(pass == 0 ? mo : vo, q0, q1, q2);
              uint16_t* d16 = reinterpret_cast<uint16_t*>(dst) + e;
              d16[0] = q0;
              d16[16384] = q1;       // + 32768 bytes: next piece
              d16[32768] = q2;
            }
          }
        }
      }
      fence_proxy_async_smem();     // generic-proxy writes of the operand tiles -> visible to the tensor core
      tc_fence_before();
      __syncthreads();
      stamp(t_begin + it, 2 + 2 * pass);
      // ---------------- 3./5. projection UMMAs ----------------
      if (tid == 0) {
        if (pass == 0) {
          mbar_wait(bar_q, ph_q);
          ph_q ^= 1;
        }
        tc_fence_after();
        const uint32_t tD = pass ? tD_v : tD_m;
        const uint32_t qb = sQ_u + (pass ? 49152 : 0);
        bool first = (it == 0);
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
          for (int j = 0; j < 3; ++j) {
            if (i + j > 2) continue;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
              const uint64_t ad = make_smem_desc(sOp_u + i * 32768 + (k >> 2) * 16384 + (k & 3) * 2048, 8192, 1024);
              const uint64_t bd = make_smem_desc(qb + j * 16384 + (k >> 2) * 8192 + (k & 3) * 2048, 8192, 1024);
              umma_bf16(tD, ad, bd, idesc2, first ? 0u : 1u);
              first = false;
            }
          }
        umma_commit(bar_mma);
        mbar_wait(bar_mma, ph_mma);   // operand tiles are rewritten by the next pass / tile
        ph_mma ^= 1;
      }
      __syncthreads();
      __syncwarp();
      tc_fence_after();
      stamp(t_begin + it, 3 + 2 * pass);
    }
  }

  // ---------------- R'[k, b0 + row] (this row-range's partial) = D[row, k]: warps 0-3 -> moment m, warps 4-7 -> v ----
  if (t_begin < t_end) {
    uint32_t d0[32], d1[32];
    const uint32_t tD = (half ? tD_v : tD_m) + lane_off;
    tmem_ld32(tD, d0);
    tmem_ld32(tD + 32, d1);
    tmem_ld_wait();
    float* R = (half ? prm.Rv : prm.Rm) + blockIdx.y * prm.split_stride;
    const int gb = b0 + rloc;
    if (gb < P) {
#pragma unroll
      for (int k = 0; k < 64; ++k)
        if (k < prm.r) R[static_cast<int64_t>(k) * P + gb] = __uint_as_float(k < 32 ? d0[k] : d1[k - 32]);
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 1) tmem_dealloc(tmem_base, kTcTmemCols);
}

static inline size_t align256(size_t x) { return (x + 255) & ~size_t(255); }

}  // namespace sowb

using namespace sowb;

static long long* g_tt_dbg = nullptr;

extern "C" {

// debug aid (not part of the product ABI): 64*8 int64 clock64 stamps of CTA (0,0) of the next tt_adam2_step launches
int tt_adam2_debug_timeline(void* buf) {
  g_tt_dbg = static_cast<long long*>(buf);
  return SOWB_OK;
}

// thin-QR scratch of the two (P x r) bases, sized for the largest rank (r <= 64)
static size_t adam2_qr_bytes(size_t P) {
  const int Pi = static_cast<int>(P);
  return align256(std::max(sow_thin_qr_workspace_bytes(Pi, std::min(64, Pi), 2), 2 * 64 * P * sizeof(float)));
}

size_t tt_adam2_workspace_bytes(int mm, int nn) {
  const size_t P = size_t(mm) * nn, P_pad = (P + 127) / 128 * 128;
  const size_t piece_arr = 3 * P_pad * 64 * sizeof(__nv_bfloat16);      // one operand array: 3 pieces of [P_pad x 64]
  return align256(2 * P * 64 * sizeof(float))                            // X{m,v}: first 64 columns of the new moments
         + adam2_qr_bytes(P)                                                    // thin-QR scratch
         + 6 * align256(piece_arr)
         + align256(tt_adam2_fused_workspace_bytes(mm, nn));                    // split partials of R'{m,v}
}

int tt_adam2_step(void* p, const void* g, const float* G1m, const float* G2m, const float* G1v, const float* G2v, int r,
                  float* Qm, float* Qv, float* Rm, float* Rv, int M, int N, int mm, int nn, double beta1, double beta2,
                  double eps, double step_size, double lr_wd, int first_step, int dtype, void* ws, size_t ws_bytes,
                  void* stream_) {
  SOWB_REQUIRE(p && g && Qm && Qv && Rm && Rv && ws, "tt_adam2_step: null pointer argument");
  SOWB_REQUIRE_TT_DTYPE("tt_adam2_step", dtype);
  if (int rc0 = ensure_context_for(g)) return rc0;
  SOWB_REQUIRE(first_step || (G1m && G2m && G1v && G2v), "tt_adam2_step: null core pointer");
  SOWB_REQUIRE(r > 0 && r <= 64, "tt_adam2_step: rank %d unsupported (1..64)", r);
  SOWB_REQUIRE(int64_t(mm) * mm >= M && int64_t(nn) * nn >= N, "tt_adam2_step: mm/nn too small for (M,N)");
  SOWB_REQUIRE(Qv == Qm + size_t(mm) * nn * r, "tt_adam2_step: Qm and Qv must be the two halves of one (2, P, r) array");
  SOWB_REQUIRE((reinterpret_cast<uintptr_t>(ws) & 255) == 0, "tt_adam2_step: workspace must be 256-byte aligned");
  if (ws_bytes < tt_adam2_workspace_bytes(mm, nn))
    return set_error(SOWB_EWORKSPACE, "tt_adam2_step: workspace %zu B < required %zu B", ws_bytes, tt_adam2_workspace_bytes(mm, nn));
  int rc = require_sm100();
  if (rc) return rc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const int P = mm * nn, P_pad = (P + 127) / 128 * 128;
  SOWB_REQUIRE(r <= P, "tt_adam2_step: rank %d exceeds the unfolding row count %d", r, P);
  uint8_t* w = static_cast<uint8_t*>(ws);
  float* X = reinterpret_cast<float*>(w);
  w += align256(2 * size_t(P) * 64 * sizeof(float));
  void* qr_ws = w;
  const size_t qr_ws_bytes = adam2_qr_bytes(size_t(P));
  w += qr_ws_bytes;
  const size_t piece_arr = align256(3 * size_t(P_pad) * 64 * sizeof(__nv_bfloat16));
  __nv_bfloat16* pcs[6];
  for (int i = 0; i < 6; ++i) pcs[i] = reinterpret_cast<__nv_bfloat16*>(w + i * piece_arr);
  w += 6 * piece_arr;
  float* part = reinterpret_cast<float*>(w);
  const size_t part_bytes = tt_adam2_fused_workspace_bytes(mm, nn);

  // 1. first 64 columns of the new moments -> thin QR -> new bases Q'{m,v} (P x r)
  rc = tt_adam2_head(g, G1m, G2m, G1v, G2v, r, X, X + size_t(P) * 64, M, N, mm, nn, beta1, beta2, first_step, dtype, stream_);
  if (rc) return rc;
  rc = sow_thin_qr(X, int64_t(P) * 64, 64, Qm, int64_t(P) * r, P, r, 2, qr_ws, qr_ws_bytes, stream_);
  if (rc) return rc;
  // Kernel choice (measured, 4096x4096 bf16): the tensor-core kernel is rank-independent (~180 us) and wins above
  // rank 16; below, and whenever the 16-byte vector path is unavailable (nn or N not a multiple of 8), the CUDA-core
  // kernel is faster.  SOWB_TT_TC=0/1 forces one of them (tests exercise both).
  bool use_tc = r > 16 && nn % 8 == 0 && N % 8 == 0;
  if (const char* e = getenv("SOWB_TT_TC")) use_tc = atoi(e) != 0;
  if (!use_tc)
    return tt_adam2_fused(p, g, G1m, G2m, G1v, G2v, r, Qm, Qv, Rm, Rv, M, N, mm, nn, beta1, beta2, eps, step_size, lr_wd,
                          first_step, dtype, part, part_bytes, stream_);
  // 2. bf16 pieces of the operands: G1 [P x r] -> [3][P_pad][64]; G2 [r x P] -> [3][64][P_pad]; Q' like G1
  SplitJobs jobs = {};
  int n_jobs = 0;
  auto split = [&](const float* src, int rows, int cols, int ld, __nv_bfloat16* dst, int rows_pad, int cols_pad) {
    jobs.src[n_jobs] = src, jobs.dst[n_jobs] = dst, jobs.rows[n_jobs] = rows, jobs.cols[n_jobs] = cols, jobs.ld[n_jobs] = ld;
    jobs.rows_pad[n_jobs] = rows_pad, jobs.cols_pad[n_jobs] = cols_pad;
    ++n_jobs;
  };
  if (!first_step) {
    split(G1m, P, r, r, pcs[0], P_pad, 64);
    split(G1v, P, r, r, pcs[1], P_pad, 64);
    split(G2m, r, P, P, pcs[2], 64, P_pad);
    split(G2v, r, P, P, pcs[3], 64, P_pad);
  }
  split(Qm, P, r, r, pcs[4], P_pad, 64);
  split(Qv, P, r, r, pcs[5], P_pad, 64);
  {
    const int64_t n = int64_t(P_pad) * 64;      // every job has P_pad * 64 elements
    const int blocks = static_cast<int>(std::min<int64_t>((n + 255) / 256, int64_t(num_sms()) * 2));
    SOWB_CHECK_CUDA(launch_pdl(tt_split3_kernel, dim3(blocks, n_jobs), dim3(256), 0, stream, jobs));
  }

  // 3. tensor maps: row-stacked pieces.  G1 / Q': [3*P_pad rows, 64 cols], box 64 x 128; G2: [3*64 rows, P_pad cols], box 64 x 64
  CUtensorMap tmG1m, tmG1v, tmG2m, tmG2v, tmQm, tmQv;
  const __nv_bfloat16* g1m_src = first_step ? pcs[4] : pcs[0];   // unused maps still need a valid base address
  const __nv_bfloat16* g1v_src = first_step ? pcs[5] : pcs[1];
  rc = make_tensor_map_2d(&tmG1m, g1m_src, 64, uint64_t(3) * P_pad, 128, 64, 128, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16);
  if (rc) return rc;
  rc = make_tensor_map_2d(&tmG1v, g1v_src, 64, uint64_t(3) * P_pad, 128, 64, 128, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16);
  if (rc) return rc;
  rc = make_tensor_map_2d(&tmG2m, pcs[2], P_pad, 3 * 64, uint64_t(P_pad) * 2, 64, 64, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16);
  if (rc) return rc;
  rc = make_tensor_map_2d(&tmG2v, pcs[3], P_pad, 3 * 64, uint64_t(P_pad) * 2, 64, 64, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16);
  if (rc) return rc;
  rc = make_tensor_map_2d(&tmQm, pcs[4], 64, uint64_t(3) * P_pad, 128, 64, 128, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16);
  if (rc) return rc;
  rc = make_tensor_map_2d(&tmQv, pcs[5], 64, uint64_t(3) * P_pad, 128, 64, 128, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16);
  if (rc) return rc;

  TcParams prm;
  prm.M = M, prm.N = N, prm.mm = mm, prm.nn = nn, prm.P = P, prm.P_pad = P_pad, prm.r = r;
  prm.beta1 = float(beta1), prm.omb1 = float(1.0 - beta1), prm.beta2 = float(beta2), prm.omb2 = float(1.0 - beta2);
  prm.eps = float(eps), prm.step_size = float(step_size), prm.lr_wd = float(lr_wd);
  prm.first_step = first_step;
  prm.dbg = g_tt_dbg;
  const int n_tiles = ceil_div(P, kTcTile);
  int splits = std::max(1, num_sms() / n_tiles);            // one CTA per SM (192 KB of shared memory each)
  splits = std::min(splits, n_tiles);
  prm.tiles_per_cta = ceil_div(n_tiles, splits);
  splits = ceil_div(n_tiles, prm.tiles_per_cta);            // every row-range is non-empty: every partial is written
  // row-range splits store partials of R'{m,v}; sum_splits_kernel adds them in range order (bit-reproducible)
  const int64_t rp = int64_t(r) * P;
  prm.Rm = Rm, prm.Rv = Rv, prm.split_stride = 0;
  if (splits > 1) {
    SOWB_REQUIRE(size_t(2) * splits * rp * sizeof(float) <= part_bytes, "tt_adam2_step: partial scratch too small");
    prm.Rm = part, prm.Rv = part + splits * rp, prm.split_stride = rp;
  }
  dim3 grid(n_tiles, splits);
  if (dtype == SOWB_BF16) {
    auto k = tt_adam2_tc_kernel<__nv_bfloat16>;
    SOWB_CHECK_CUDA(set_max_smem_once(k, size_t(kTcSmem)));
    SOWB_CHECK_CUDA(launch_pdl(k, grid, dim3(kTcThreads), size_t(kTcSmem), stream, tmG1m, tmG1v, tmG2m, tmG2v, tmQm, tmQv,
                               static_cast<__nv_bfloat16*>(p), static_cast<const __nv_bfloat16*>(g), prm));
  } else if (dtype == SOWB_F32) {
    auto k = tt_adam2_tc_kernel<float>;
    SOWB_CHECK_CUDA(set_max_smem_once(k, size_t(kTcSmem)));
    SOWB_CHECK_CUDA(launch_pdl(k, grid, dim3(kTcThreads), size_t(kTcSmem), stream, tmG1m, tmG1v, tmG2m, tmG2v, tmQm, tmQv,
                               static_cast<float*>(p), static_cast<const float*>(g), prm));
  } else {
    return set_error(SOWB_EINVAL, "tt_adam2_step: unknown dtype %d", dtype);
  }
  SOWB_CHECK_CUDA(cudaGetLastError());
  if (splits > 1) return launch_sum_splits(part, splits, rp, splits * rp, Rm, Rv - Rm, rp, 2, stream);
  return SOWB_OK;
}

}  // extern "C"
