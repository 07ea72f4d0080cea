// C-ABI entry points for the SoW linear forward / backward (include/sow_b200.h) on top of the tcgen05 GEMM (gemm.cuh)
// and the fused dt + dB pass (k2.cuh).  The unit of work is a GROUP of projections that read the same input
// (q/k/v, gate/up; a lone projection is a group of one): one packed factor operand, one skinny GEMM for all t's, one
// split-K GEMM for all dA's, one dX GEMM over all members' W.
#include "common.cuh"
#include "gemm.cuh"
#include "k2.cuh"

#include <algorithm>
#include <mutex>
#include <stdlib.h>

namespace sowb {

constexpr int kMaxGroup = 4;   // members per group (dX fuses at most kMaxSeg - 1 of them into one launch)

// ------------------------------------------------------------------------------------------------
// small helper kernels
// ------------------------------------------------------------------------------------------------
// A_i (in, r_i) for i < n  ->  A_cat (in, R) = [A_0 | 0 | A_1 | 0 | ...], every member zero-padded to a multiple of 64
// columns: gives the factors a TMA-legal row pitch and one operand for the shared down-projection.  A bit copy of 16-bit
// elements (0x0000 is +0 in bf16 and fp16): serves both 16-bit types.
struct PackArgs {
  const uint16_t* A[kMaxGroup];
  int r[kMaxGroup];
  int off[kMaxGroup + 1];   // first column of member i in A_cat; off[n] = R
  int n;
};
__global__ void pack_factors_kernel(const PackArgs a, uint16_t* __restrict__ A_cat, int in, int R) {
  const int64_t total = static_cast<int64_t>(in) * (R >> 1);      // one 16-bit pair per thread
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int row = static_cast<int>(i / (R >> 1));
    const int col = static_cast<int>(i % (R >> 1)) * 2;
    int m = 0;
    while (m + 1 < a.n && col >= a.off[m + 1]) ++m;
    const int c = col - a.off[m];
    const uint16_t* src = a.A[m] + static_cast<int64_t>(row) * a.r[m];
    const uint32_t lo = (c < a.r[m]) ? src[c] : 0u;
    const uint32_t hi = (c + 1 < a.r[m]) ? src[c + 1] : 0u;
    *reinterpret_cast<uint32_t*>(A_cat + static_cast<int64_t>(row) * R + col) = lo | (hi << 16);
  }
}

// fp32 split PARTIALS -> 16-bit (bf16 / fp16) gradients in the reference layouts, summed over the splits in a fixed order (so the
// factor gradients are bit-reproducible run to run).  A job sums `splits` partial matrices [rows x ld_src] and writes
// the first `cols` columns either as they are (dA: dst[row, col]) or transposed (dB: partial is dB^T, dst[col, row]).
struct FinJob {
  const float* src;
  int64_t split_stride;
  uint16_t* dst;
  int splits, rows, cols, ld_src, ld_dst, transpose, blk_begin, col_tiles;
};
constexpr int kMaxFinJobs = 8;
struct FinJobs {
  FinJob j[kMaxFinJobs];
  int n;
};
template <bool F16>
__device__ __forceinline__ uint16_t to16(float f) {
  return static_cast<uint16_t>(pack16x2<F16>(f, 0.f) & 0xffffu);
}

template <bool F16>
__global__ void finalize_jobs_kernel(const FinJobs jobs) {
  __shared__ float tile[32][33];
  int ji = 0;
  while (ji + 1 < jobs.n && static_cast<int>(blockIdx.x) >= jobs.j[ji + 1].blk_begin) ++ji;
  const FinJob& J = jobs.j[ji];
  const int b = blockIdx.x - J.blk_begin;
  const int r0 = (b / J.col_tiles) * 32, c0 = (b % J.col_tiles) * 32;
  const int row = r0 + threadIdx.y, col = c0 + threadIdx.x;
  float s = 0.f;
  if (row < J.rows && col < J.cols) {
    const float* p = J.src + static_cast<int64_t>(row) * J.ld_src + col;
    // fixed summation order 0..splits-1; the loads of 8 splits are issued together (the partials come from DRAM: the
    // kernels that wrote them streamed hundreds of MB through L2 since)
    int k = 0;
    for (; k + 8 <= J.splits; k += 8) {
      float v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = __ldcs(p + (k + u) * J.split_stride);
#pragma unroll
      for (int u = 0; u < 8; ++u) s += v[u];
    }
    for (; k < J.splits; ++k) s += __ldcs(p + k * J.split_stride);
  }
  if (!J.transpose) {
    if (row < J.rows && col < J.cols) J.dst[static_cast<int64_t>(row) * J.ld_dst + col] = to16<F16>(s);
    return;
  }
  tile[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  const int orow = r0 + threadIdx.x, ocol = c0 + threadIdx.y;   // orow: partial row (out index), ocol: rank index
  if (orow < J.rows && ocol < J.cols)
    J.dst[static_cast<int64_t>(ocol) * J.ld_dst + orow] = to16<F16>(tile[threadIdx.x][threadIdx.y]);
}

// v -> hi = bf16(v), lo = bf16(v - hi): operand pieces of the bf16x3 products (fp32 modules)
__global__ void split_bf16x2_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ hi,
                                    __nv_bfloat16* __restrict__ lo, int64_t n4) {
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const float4 v = reinterpret_cast<const float4*>(src)[i];
    const float f[4] = {v.x, v.y, v.z, v.w};
    __nv_bfloat16 h[4], l[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      h[j] = __float2bfloat16(f[j]);
      l[j] = __float2bfloat16(f[j] - __bfloat162float(h[j]));
    }
    reinterpret_cast<uint2*>(hi)[i] = make_uint2(pack_bf16x2(__bfloat162float(h[0]), __bfloat162float(h[1])),
                                                 pack_bf16x2(__bfloat162float(h[2]), __bfloat162float(h[3])));
    reinterpret_cast<uint2*>(lo)[i] = make_uint2(pack_bf16x2(__bfloat162float(l[0]), __bfloat162float(l[1])),
                                                 pack_bf16x2(__bfloat162float(l[2]), __bfloat162float(l[3])));
  }
}
__global__ void split_bf16x2_tail_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ hi,
                                         __nv_bfloat16* __restrict__ lo, int64_t begin, int64_t n) {
  const int64_t i = begin + blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i < n) {
    const __nv_bfloat16 h = __float2bfloat16(src[i]);
    hi[i] = h;
    lo[i] = __float2bfloat16(src[i] - __bfloat162float(h));
  }
}

// dbias[o] = sum_t dY[t, o]: block = 64 columns x 4 row-lanes, grid.y splits T; every block writes its partial row,
// the conversion kernel sums the partial rows in a fixed order (bit-reproducible).
template <bool F16>
__global__ void colsum_kernel(const uint16_t* __restrict__ dy, float* __restrict__ part, int64_t T, int out) {
  __shared__ float red[4][64];
  const int col = blockIdx.x * 64 + threadIdx.x;
  const int64_t rows_per = (T + gridDim.y - 1) / gridDim.y;
  const int64_t t0 = blockIdx.y * rows_per, t1 = min(T, t0 + rows_per);
  float s = 0.f;
  if (col < out)
    for (int64_t t = t0 + threadIdx.y; t < t1; t += blockDim.y) s += lo16_to_f32<F16>(dy[t * out + col]);
  red[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.y == 0 && col < out)
    part[static_cast<int64_t>(blockIdx.y) * out + col] = (red[0][threadIdx.x] + red[1][threadIdx.x]) + (red[2][threadIdx.x] + red[3][threadIdx.x]);
}
template <bool F16>
__global__ void sum_partials_to_16_kernel(const float* __restrict__ part, uint16_t* __restrict__ dst, int n, int parts) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    float s = 0.f;
    for (int k = 0; k < parts; ++k) s += part[static_cast<int64_t>(k) * n + i];
    dst[i] = to16<F16>(s);
  }
}

// ------------------------------------------------------------------------------------------------
// GEMM launcher
// ------------------------------------------------------------------------------------------------
struct Operand {
  const void* ptr;
  uint64_t rows, cols;  // as stored in global memory, row-major, `cols` contiguous
  uint64_t pitch_elems;
};
struct Segment {
  Operand A, B;
  int K;
};

// resident clusters of the CTA-pair GEMM (sow_gemm_pair_kernel) on the current device; every instantiation has the same
// resources, so one query serves all of them
static int pair_max_clusters() {
  static std::mutex mu;
  static int cache[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;
  std::lock_guard<std::mutex> lk(mu);
  if (cache[dev] == 0) {
    int n = 0;
    set_max_smem_once(sow_gemm_pair_kernel<true, false>, size_t(GemmPairSmem::kTotal));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * num_sms());
    cfg.blockDim = dim3(kGemmThreads);
    cfg.dynamicSmemBytes = GemmPairSmem::kTotal;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    if (cudaOccupancyMaxActiveClusters(&n, sow_gemm_pair_kernel<true, false>, &cfg) != cudaSuccess || n <= 0) {
      cudaGetLastError();
      n = std::max(1, num_sms() / 2);
    }
    cache[dev] = n;
  }
  return cache[dev];
}

// Operand A of D = A.B: logical [M, K].  K-major  <=> stored [M rows, K cols];  MN-major <=> stored [K rows, M cols].
// Operand B of D = A.B: logical [K, N].  K-major  <=> stored [N rows, K cols];  MN-major <=> stored [K rows, N cols].
// f16: the 16-bit operands (and a 16-bit C / bias) are fp16, else bf16.
// PAIR: the work item is a 256 x 256 tile computed by a cluster of two CTAs (sow_gemm_pair_kernel); BN = 256, MT = 1,
// A K-major, EPI_BF16_TMA only.
template <int BN, bool A_MN, bool B_MN, int EPI, int MT = 1, bool PAIR = false>
static int launch_gemm(const Segment* segs, int nseg, void* C_bf16, float* C_f32, int ldc, int M, int N,
                       const float* alpha_blocks, int n_alpha, const void* bias, bool split_k, bool f16, cudaStream_t stream,
                       int prof_class, double alg_flops, int* splits_out = nullptr) {
  using S = GemmSmem<BN, MT>;
  static_assert(!PAIR || (BN == 256 && MT == 1 && !A_MN && EPI == EPI_BF16_TMA), "pair tiles: 256 wide, A K-major, 16-bit out");
  if (nseg < 1 || nseg > kMaxSeg) return set_error(SOWB_EINVAL, "launch_gemm: %d segments (max %d)", nseg, kMaxSeg);
  GemmMaps maps;
  GemmParams p;
  int rc;
  int kb = 0;
  const CUtensorMapDataType t16 = map_type16(f16);
  for (int s = 0; s < kMaxSeg; ++s) {
    const Segment& sg = segs[s < nseg ? s : 0];
    rc = make_tensor_map_2d(&maps.a[s], sg.A.ptr, sg.A.cols, sg.A.rows, sg.A.pitch_elems * 2, 64, A_MN ? 64 : kBM, t16);
    if (rc) return rc;
    rc = make_tensor_map_2d(&maps.b[s], sg.B.ptr, sg.B.cols, sg.B.rows, sg.B.pitch_elems * 2, 64, B_MN ? 64 : (PAIR ? BN / 2 : BN), t16);
    if (rc) return rc;
    if (s < nseg) kb += ceil_div(sg.K, kBK);
    p.kb_end[s] = kb;
  }
  maps.c = maps.a[0];
  if (EPI == EPI_BF16_TMA) {
    rc = make_tensor_map_2d(&maps.c, C_bf16, N, M, static_cast<uint64_t>(ldc) * 2, kStoreBoxCols, kBM, t16);
    if (rc) return rc;
  } else if (EPI == EPI_F32_TMA) {
    rc = make_tensor_map_2d(&maps.c, C_f32, N, M, static_cast<uint64_t>(ldc) * 4, 32, kBM, CU_TENSOR_MAP_DATA_TYPE_FLOAT32);
    if (rc) return rc;
  }
  p.M = M;
  p.N = N;
  p.nseg = nseg;
  p.m_tiles = ceil_div(M, kBM * MT * (PAIR ? 2 : 1));      // work rows: MT tiles of 128 rows each (two CTAs' for PAIR)
  p.n_tiles = ceil_div(N, BN);
  const int kb_total = kb;
  const int sms = num_sms();
  int splits = 1;
  if (split_k) {
    splits = sms / (p.m_tiles * p.n_tiles);
    if (splits < 1) splits = 1;
    if (splits > kb_total) splits = kb_total;
  }
  p.kb_per_split = ceil_div(kb_total, std::max(1, splits));
  p.splits = ceil_div(kb_total, std::max(1, p.kb_per_split));
  p.alpha_blocks = (n_alpha > 1) ? std::min(n_alpha, kMaxAlphaBlocks) : 0;
  for (int i = 0; i < kMaxAlphaBlocks; ++i) p.alpha[i] = (i < n_alpha) ? alpha_blocks[i] : alpha_blocks[std::max(0, n_alpha - 1)];
  p.bias = (EPI == EPI_BF16_TMA) ? static_cast<const uint16_t*>(bias) : nullptr;
  p.bias_f32 = (EPI == EPI_F32_TMA) ? static_cast<const float*>(bias) : nullptr;
  p.out_f32 = C_f32;
  p.split_stride = static_cast<int64_t>(M) * ldc;
  p.ldc = ldc;
  if (splits_out) *splits_out = p.splits;
  const int total = p.m_tiles * p.n_tiles * p.splits;
  if (total <= 0 || kb_total <= 0) return SOWB_OK;
  if constexpr (PAIR) {
    auto kern = f16 ? sow_gemm_pair_kernel<B_MN, true> : sow_gemm_pair_kernel<B_MN, false>;
    SOWB_CHECK_CUDA(set_max_smem_once(kern, size_t(GemmPairSmem::kTotal)));
    const int clusters = std::min(total, pair_max_clusters());
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * clusters);
    cfg.blockDim = dim3(kGemmThreads);
    cfg.dynamicSmemBytes = GemmPairSmem::kTotal;
    cfg.stream = stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    ProfileScope prof(stream, prof_class, alg_flops);
    SOWB_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, maps, p));
    return SOWB_OK;
  }
  auto kern = sow_gemm_kernel<BN, A_MN, B_MN, EPI, MT, false>;
  if constexpr (EPI != EPI_F32_TMA) {   // the bf16x3 path of fp32 modules has bf16 operands only
    if (f16) kern = sow_gemm_kernel<BN, A_MN, B_MN, EPI, MT, true>;
  }
  SOWB_CHECK_CUDA(set_max_smem_once(kern, size_t(S::kTotal)));
  const int grid = total < sms ? total : sms;
  ProfileScope prof(stream, prof_class, alg_flops);   // algorithmic flops: un-padded ranks (SURVEY.md 8d)
  kern<<<grid, kGemmThreads, S::kTotal, stream>>>(maps, p);
  SOWB_CHECK_CUDA(cudaGetLastError());
  return SOWB_OK;
}

static inline size_t align256(size_t x) { return (x + 255) & ~size_t(255); }

// 256 x 256 CTA tiles (MT = 2) cut the L2 -> SM operand traffic per MAC by a third, but they halve the number of work items
// (wave quantisation) and expose the epilogue (no second TMEM stage).  Measured at T = 32768 / 8192 (tools/bench_group.py,
// SOWB_BIG_TILES=0/1): Llama-7B gate/up forward 590 -> 514 us (1441 TFLOP/s) and its dX 1006 -> 980 us; Llama-350M gate/up
// forward 155.5 -> 151.9 us; but q/k/v forward 60.7 -> 67.6 us (512 items = 3.46 waves) and down dX 140.6 -> 152.7 us
// (17 k-blocks: the exposed epilogue costs more than the traffic saves).  Hence: only when the last wave is >= 93 % full
// AND the K loop is long enough (>= 32 k-blocks) to amortise the epilogue.
static bool use_big_tiles(int M, int N, int kb_total) {
  static const int knob = []() {
    const char* e = getenv("SOWB_BIG_TILES");   // tuning knob: 0 never, 1 always, unset = by wave efficiency
    return e ? atoi(e) : -1;
  }();
  if (knob >= 0) return knob != 0;
  const int items = ceil_div(M, 2 * kBM) * ceil_div(N, 256);
  const int sms = num_sms();
  const int waves = ceil_div(items, sms);
  return kb_total >= 32 && items >= 2 * sms && double(items) / (double(waves) * sms) >= 0.93;
}

// CTA-pair 256 x 256 tiles (sow_gemm_pair_kernel) take every 16-bit forward y_i and group dX that the rules above leave on the
// 128 x 256 tile.  They keep the same number of SMs busy as the 128 x 256 tiles (a pair tile is two CTAs) with a third less
// operand traffic per MAC, so they are used at every size (small T was not timed separately).  Measured at T = 32768
// (tools/bench_group.py): 7-18 % less time per launch for every Llama-350M forward and dX.  SOWB_GEMM_PAIR=0 restores the
// 128 x 256 tile (for A/B runs).
static bool use_pair_tiles() {
  static const bool on = []() {
    const char* e = getenv("SOWB_GEMM_PAIR");
    return e == nullptr || atoi(e) != 0;
  }();
  return on;
}

// number of split-K partials launch_gemm<BN, ..., EPI_F32_PARTIAL> produces for an [M x N] output contracted over K
static int splitk_count(int M, int N, int BN, int K) {
  const int tiles = ceil_div(M, kBM) * ceil_div(N, BN), kb_total = ceil_div(K, kBK);
  int splits = num_sms() / std::max(1, tiles);
  splits = std::max(1, std::min(splits, kb_total));
  const int per = ceil_div(kb_total, splits);
  return ceil_div(kb_total, per);
}
constexpr int kBiasParts = 64;

// tile width of the skinny GEMMs over the concatenated rank dimension R (a multiple of 64)
static int skinny_bn(int R) { return R >= 256 ? 256 : R; }

template <bool A_MN, bool B_MN, int EPI>
static int launch_skinny(int R, const Segment* seg, int nseg, void* C_bf16, float* C_f32, int ldc, int M,
                         const float* alpha, int n_alpha, bool split_k, bool f16, cudaStream_t stream, int prof_class,
                         double alg_flops, int* splits_out = nullptr) {
  switch (skinny_bn(R)) {
    case 64:
      return launch_gemm<64, A_MN, B_MN, EPI>(seg, nseg, C_bf16, C_f32, ldc, M, R, alpha, n_alpha, nullptr, split_k, f16, stream, prof_class, alg_flops, splits_out);
    case 128:
      return launch_gemm<128, A_MN, B_MN, EPI>(seg, nseg, C_bf16, C_f32, ldc, M, R, alpha, n_alpha, nullptr, split_k, f16, stream, prof_class, alg_flops, splits_out);
    case 192:
      return launch_gemm<192, A_MN, B_MN, EPI>(seg, nseg, C_bf16, C_f32, ldc, M, R, alpha, n_alpha, nullptr, split_k, f16, stream, prof_class, alg_flops, splits_out);
    default:
      return launch_gemm<256, A_MN, B_MN, EPI>(seg, nseg, C_bf16, C_f32, ldc, M, R, alpha, n_alpha, nullptr, split_k, f16, stream, prof_class, alg_flops, splits_out);
  }
}

// K2 decomposition of one projection: clusters of G CTAs (one column group each), n_clusters of them walking the T-chunks
struct K2Plan {
  int G, bpg, n_clusters, n_chunks, n_launch, blk_per_launch, out_pad;
};
static int k2_max_clusters(int G) {
  static std::mutex mu;
  static int cache[64][kK2MaxG + 1] = {{0}};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;
  std::lock_guard<std::mutex> lk(mu);
  if (cache[dev][G] == 0) {
    int n = 0;
    // the fp16 instantiation has the same resources: one query serves both
    set_max_smem_once(sow_k2_kernel<false>, size_t(kK2SmemTotal));
    if (G > 8) cudaFuncSetAttribute(sow_k2_kernel<false>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(G * 64);
    cfg.blockDim = dim3(kK2Threads);
    cfg.dynamicSmemBytes = kK2SmemTotal;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = G;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    if (cudaOccupancyMaxActiveClusters(&n, sow_k2_kernel<false>, &cfg) != cudaSuccess || n <= 0) {
      cudaGetLastError();
      n = std::max(1, (num_sms() / G) * 3 / 4);      // conservative guess if the query is unavailable
    }
    cache[dev][G] = n;
  }
  return cache[dev][G];
}
static K2Plan k2_plan(int64_t T, int out) {
  K2Plan pl;
  const int nblk = ceil_div(out, 128);
  pl.n_launch = ceil_div(nblk, kK2MaxG * kK2MaxBpg);
  pl.blk_per_launch = ceil_div(nblk, pl.n_launch);
  pl.G = 1;
  while (pl.G * kK2MaxBpg < pl.blk_per_launch) pl.G *= 2;
  pl.bpg = ceil_div(pl.blk_per_launch, pl.G);
  pl.n_chunks = static_cast<int>((T + 127) / 128);
  const int cap = pl.G == 1 ? num_sms() : k2_max_clusters(pl.G);
  pl.n_clusters = std::max(1, std::min(cap, pl.n_chunks));
  pl.out_pad = round_up(out, 128);
  return pl;
}

struct GroupLayout {
  int n, R;
  int off[kMaxGroup + 1];
  int rpad[kMaxGroup];
};

static int group_layout(const char* fn, const sowb_group_member* m, int n, int64_t T, int in, int dtype, const void* any,
                        GroupLayout* L) {
  if (any != nullptr) {
    const int rc0 = ensure_context_for(any);   // backward runs on autograd's worker thread
    if (rc0) return rc0;
  }
  if (dtype != SOWB_BF16 && dtype != SOWB_F32 && dtype != SOWB_F16) return set_error(SOWB_EINVAL, "%s: unknown dtype %d", fn, dtype);
  if (m == nullptr || n < 1 || n > kMaxGroup) return set_error(SOWB_EINVAL, "%s: group size %d (1..%d)", fn, n, kMaxGroup);
  if (T <= 0 || in <= 0) return set_error(SOWB_EINVAL, "%s: non-positive dimension", fn);
  if (T >= (int64_t(1) << 31)) return set_error(SOWB_EINVAL, "%s: T too large", fn);
  if (in % 8 != 0) return set_error(SOWB_EINVAL, "%s: in=%d must be a multiple of 8 (16-byte TMA row pitch)", fn, in);
  L->n = n;
  int off = 0;
  for (int i = 0; i < n; ++i) {
    if (m[i].out <= 0 || m[i].r <= 0) return set_error(SOWB_EINVAL, "%s: member %d has a non-positive dimension", fn, i);
    if (m[i].out % 8 != 0)
      return set_error(SOWB_EINVAL, "%s: out=%d must be a multiple of 8 (16-byte TMA row pitch)", fn, m[i].out);
    if (m[i].A == nullptr || m[i].B == nullptr) return set_error(SOWB_EINVAL, "%s: member %d has a null factor", fn, i);
    L->off[i] = off;
    L->rpad[i] = round_up(m[i].r, kBK);
    off += L->rpad[i];
  }
  L->off[n] = off;
  L->R = off;
  if (L->R / 64 > kMaxAlphaBlocks)
    return set_error(SOWB_EINVAL, "%s: concatenated rank %d exceeds %d", fn, L->R, 64 * kMaxAlphaBlocks);
  return require_sm100();
}

static size_t group_bwd_ws(const sowb_group_member* m, const GroupLayout& L, int64_t T, int in, size_t* off_partA,
                           size_t* off_partB /*[n]*/, size_t* off_bias) {
  size_t o = 0;
  const int sa = splitk_count(in, L.R, skinny_bn(L.R), static_cast<int>(T));
  if (off_partA) *off_partA = o;
  o += align256(size_t(sa) * in * L.R * 4);
  for (int i = 0; i < L.n; ++i) {
    const K2Plan pl = k2_plan(T, m[i].out);
    if (off_partB) off_partB[i] = o;
    o += align256(size_t(pl.n_clusters) * pl.out_pad * L.rpad[i] * 4);
  }
  if (off_bias) *off_bias = o;
  int max_out = 0;
  for (int i = 0; i < L.n; ++i) max_out = std::max(max_out, m[i].out);
  o += align256(size_t(kBiasParts) * max_out * 4);
  return o;
}

}  // namespace sowb

using namespace sowb;

static long long* g_k2_ts = nullptr;   // debug timeline buffer (device), see sow_k2_debug_timeline

extern "C" {

// Debug aid (not part of the product ABI): device buffer of 64*16 int64 that CTA 0 of the next K2 launches fills with
// clock64 stamps per T-chunk; pass NULL to switch off.
int sow_k2_debug_timeline(void* buf) {
  g_k2_ts = static_cast<long long*>(buf);
  return SOWB_OK;
}

int sow_rank_pad(int r) { return round_up(r, kBK); }

size_t sow_group_workspace_bytes(int op, int64_t T, int in, const sowb_group_member* m, int n) {
  if (op != SOWB_OP_LINEAR_BWD || m == nullptr || n < 1 || n > kMaxGroup || T <= 0) return 0;
  GroupLayout L;
  L.n = n;
  int off = 0;
  for (int i = 0; i < n; ++i) {
    L.off[i] = off;
    L.rpad[i] = round_up(m[i].r, kBK);
    off += L.rpad[i];
  }
  L.off[n] = L.R = off;
  return group_bwd_ws(m, L, T, in, nullptr, nullptr, nullptr);
}

int sow_split_bf16x2(const float* src, void* hi, void* lo, int64_t n, void* stream_) {
  if (n <= 0) return SOWB_OK;
  SOWB_REQUIRE(src && hi && lo, "sow_split_bf16x2: null pointer argument");
  if (int rc0 = ensure_context_for(src)) return rc0;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const int64_t n4 = ((reinterpret_cast<uintptr_t>(src) & 15) == 0 && (reinterpret_cast<uintptr_t>(hi) & 7) == 0 &&
                      (reinterpret_cast<uintptr_t>(lo) & 7) == 0) ? n / 4 : 0;
  if (n4 > 0) {
    const int blocks = static_cast<int>(std::min<int64_t>((n4 + 255) / 256, int64_t(num_sms()) * 16));
    split_bf16x2_kernel<<<blocks, 256, 0, stream>>>(src, static_cast<__nv_bfloat16*>(hi), static_cast<__nv_bfloat16*>(lo), n4);
    SOWB_CHECK_CUDA(cudaGetLastError());
  }
  if (n4 * 4 < n) {
    const int64_t rem = n - n4 * 4;
    split_bf16x2_tail_kernel<<<static_cast<int>((rem + 255) / 256), 256, 0, stream>>>(
        src, static_cast<__nv_bfloat16*>(hi), static_cast<__nv_bfloat16*>(lo), n4 * 4, n);
    SOWB_CHECK_CUDA(cudaGetLastError());
  }
  return SOWB_OK;
}

int sow_group_fwd(const void* x, const void* x_lo, const sowb_group_member* m, int n, void* A_cat, void* t_cat, int64_t T,
                  int in, int dtype, void* stream_) {
  GroupLayout L;
  int rc = group_layout("sow_group_fwd", m, n, T, in, dtype, x, &L);
  if (rc) return rc;
  SOWB_REQUIRE(x && A_cat && t_cat, "sow_group_fwd: null pointer argument");
  const bool f32 = dtype == SOWB_F32, f16 = dtype == SOWB_F16;
  SOWB_REQUIRE(!f32 || x_lo != nullptr, "sow_group_fwd: SOWB_F32 needs the low piece of x");
  SOWB_REQUIRE(!f16 || x_lo == nullptr, "sow_group_fwd: SOWB_F16 takes no x_lo");
  for (int i = 0; i < n; ++i) SOWB_REQUIRE(!f16 || m[i].W_lo == nullptr, "sow_group_fwd: SOWB_F16 takes no W_lo (member %d)", i);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const int R = L.R;
  {
    PackArgs pa;
    pa.n = n;
    for (int i = 0; i < kMaxGroup; ++i) {
      pa.A[i] = static_cast<const uint16_t*>(m[i < n ? i : 0].A);
      pa.r[i] = m[i < n ? i : 0].r;
      pa.off[i] = L.off[i < n ? i : n];
    }
    pa.off[kMaxGroup] = R;
    for (int i = n; i <= kMaxGroup; ++i) pa.off[i] = R;
    const int64_t total = int64_t(in) * (R / 2);
    const int blocks = static_cast<int>(std::min<int64_t>((total + 255) / 256, 2048));
    pack_factors_kernel<<<blocks, 256, 0, stream>>>(pa, static_cast<uint16_t*>(A_cat), in, R);
    SOWB_CHECK_CUDA(cudaGetLastError());
  }
  // t_cat [T, R] = scale_i * x . A_cat      (one pass over x for every member of the group)
  {
    float alpha[kMaxAlphaBlocks];
    int nb = 0;
    for (int i = 0; i < n; ++i)
      for (int b = 0; b < L.rpad[i] / 64; ++b) alpha[nb++] = m[i].scale;
    Segment sg[2] = {{Operand{x, uint64_t(T), uint64_t(in), uint64_t(in)},
                      Operand{A_cat, uint64_t(in), uint64_t(R), uint64_t(R)}, in},   // B operand [K=in rows, N=R cols]
                     {Operand{x_lo, uint64_t(T), uint64_t(in), uint64_t(in)},
                      Operand{A_cat, uint64_t(in), uint64_t(R), uint64_t(R)}, in}};
    int rsum = 0;
    for (int i = 0; i < n; ++i) rsum += m[i].r;
    rc = launch_skinny<false, true, EPI_BF16_TMA>(R, sg, f32 ? 2 : 1, t_cat, nullptr, R, static_cast<int>(T), alpha, nb, false,
                                                  f16, stream, PROF_GEMM_SKINNY, 2.0 * double(T) * double(in) * double(rsum));
    if (rc) return rc;
  }
  // y_i = x . W_i + t_i . B_i (+ bias_i)
  const float one = 1.0f;
  for (int i = 0; i < n; ++i) {
    SOWB_REQUIRE(m[i].y != nullptr, "sow_group_fwd: member %d has no output buffer", i);
    const uint16_t* t_i = static_cast<const uint16_t*>(t_cat) + L.off[i];
    Segment segs[4];
    int ns = 0;
    if (m[i].W != nullptr) {
      const Operand opX{x, uint64_t(T), uint64_t(in), uint64_t(in)};
      const Operand opW{m[i].W, uint64_t(in), uint64_t(m[i].out), uint64_t(m[i].out)};
      segs[ns++] = Segment{opX, opW, in};
      if (f32) {
        SOWB_REQUIRE(m[i].W_lo != nullptr, "sow_group_fwd: SOWB_F32 needs the low piece of W (member %d)", i);
        const Operand opXl{x_lo, uint64_t(T), uint64_t(in), uint64_t(in)};
        const Operand opWl{m[i].W_lo, uint64_t(in), uint64_t(m[i].out), uint64_t(m[i].out)};
        segs[ns++] = Segment{opX, opWl, in};
        segs[ns++] = Segment{opXl, opW, in};
      }
    }
    // rows >= r of B read as zero through the tensor-map bounds
    segs[ns++] = Segment{Operand{t_i, uint64_t(T), uint64_t(L.rpad[i]), uint64_t(R)},
                         Operand{m[i].B, uint64_t(m[i].r), uint64_t(m[i].out), uint64_t(m[i].out)}, L.rpad[i]};
    const double fl = 2.0 * double(T) * double(m[i].out) * (double(m[i].W != nullptr ? in : 0) + double(m[i].r));
    if (f32)
      rc = launch_gemm<256, false, true, EPI_F32_TMA>(segs, ns, nullptr, static_cast<float*>(m[i].y), m[i].out,
                                                      static_cast<int>(T), m[i].out, &one, 1, m[i].bias, false, false,
                                                      stream, PROF_GEMM_FWD, fl);
    else if (use_big_tiles(static_cast<int>(T), m[i].out, ceil_div(in, kBK) * (m[i].W != nullptr) + L.rpad[i] / kBK))
      rc = launch_gemm<256, false, true, EPI_BF16_TMA, 2>(segs, ns, m[i].y, nullptr, m[i].out, static_cast<int>(T), m[i].out,
                                                          &one, 1, m[i].bias, false, f16, stream, PROF_GEMM_FWD, fl);
    else if (use_pair_tiles())
      rc = launch_gemm<256, false, true, EPI_BF16_TMA, 1, true>(segs, ns, m[i].y, nullptr, m[i].out, static_cast<int>(T), m[i].out,
                                                                &one, 1, m[i].bias, false, f16, stream, PROF_GEMM_FWD, fl);
    else
      rc = launch_gemm<256, false, true, EPI_BF16_TMA>(segs, ns, m[i].y, nullptr, m[i].out, static_cast<int>(T), m[i].out,
                                                       &one, 1, m[i].bias, false, f16, stream, PROF_GEMM_FWD, fl);
    if (rc) return rc;
  }
  return SOWB_OK;
}

int sow_group_bwd(const void* x, const void* A_cat, const void* t_cat, const sowb_group_member* m, int n, void* dt_cat,
                  void* dx, int64_t T, int in, int dtype, void* ws, size_t ws_bytes, void* stream_) {
  GroupLayout L;
  int rc = group_layout("sow_group_bwd", m, n, T, in, dtype, x, &L);
  if (rc) return rc;
  SOWB_REQUIRE(x && A_cat && t_cat && dt_cat && ws, "sow_group_bwd: null pointer argument");
  size_t oA, oB[kMaxGroup], oBias;
  const size_t need = group_bwd_ws(m, L, T, in, &oA, oB, &oBias);
  if (ws_bytes < need)
    return set_error(SOWB_EWORKSPACE, "sow_group_bwd: workspace %zu B < required %zu B", ws_bytes, need);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  uint8_t* wsp = static_cast<uint8_t*>(ws);
  const int R = L.R;
  const int Ti = static_cast<int>(T);
  const bool f16 = dtype == SOWB_F16;
  const CUtensorMapDataType t16 = map_type16(f16);
  for (int i = 0; i < n; ++i)
    SOWB_REQUIRE(!f16 || (m[i].W_lo == nullptr && m[i].dy_lo == nullptr), "sow_group_bwd: SOWB_F16 takes no W_lo / dy_lo (member %d)", i);

  // ---- K2: one pass over every dY_i -> dt_i (into dt_cat) and the split partials of dB_i^T -------------
  auto k2_kernel = f16 ? sow_k2_kernel<true> : sow_k2_kernel<false>;
  SOWB_CHECK_CUDA(set_max_smem_once(k2_kernel, size_t(kK2SmemTotal)));
  K2Plan plans[kMaxGroup];
  bool uniform = true;
  for (int i = 0; i < n; ++i) {
    SOWB_REQUIRE(m[i].dy != nullptr, "sow_group_bwd: member %d has no upstream gradient", i);
    plans[i] = k2_plan(T, m[i].out);
    if (plans[i].G > 8)
      SOWB_CHECK_CUDA(cudaFuncSetAttribute(k2_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    uniform = uniform && plans[i].G == plans[0].G && plans[i].n_launch == plans[0].n_launch && L.rpad[i] == L.rpad[0];
  }
  // members that share the cluster size go into ONE launch with the clusters partitioned among them
  const int n_batches = uniform ? 1 : n;
  for (int bt = 0; bt < n_batches; ++bt) {
    const int i0 = uniform ? 0 : bt, cnt = uniform ? n : 1;
    const K2Plan& pl0 = plans[i0];
    const int cap = pl0.G == 1 ? num_sms() : k2_max_clusters(pl0.G);
    const int total_clusters = std::max(cnt, std::min(cap, cnt * pl0.n_chunks));
    int cl_begin[kK2MaxMembers + 1];
    cl_begin[0] = 0;
    for (int j = 0; j < cnt; ++j) {
      int share = (total_clusters * (j + 1)) / cnt - (total_clusters * j) / cnt;
      share = std::max(1, std::min(share, pl0.n_chunks));
      // same makespan with fewer clusters = fewer dB^T split partials
      share = ceil_div(pl0.n_chunks, ceil_div(pl0.n_chunks, share));
      plans[i0 + j].n_clusters = share;
      cl_begin[j + 1] = cl_begin[j] + share;
    }
    for (int ch = 0; ch < L.rpad[i0] / 64; ++ch) {
      for (int ln = 0; ln < pl0.n_launch; ++ln) {
        K2Maps maps;
        K2Params p;
        p.T = Ti;
        p.G = pl0.G;
        p.n_members = cnt;
        p.n_chunks = pl0.n_chunks;
        p.ldt = R;
        p.dbg = g_k2_ts;
        double flops = 0;
        for (int j = 0; j <= kK2MaxMembers; ++j) p.cl_begin[j] = cl_begin[std::min(j, cnt)];
        for (int j = 0; j < kK2MaxMembers; ++j) {
          const int i = i0 + std::min(j, cnt - 1);
          const K2Plan& pl = plans[i];
          K2MemberMaps& mm = maps.m[j];
          rc = make_tensor_map_2d(&mm.dy, m[i].dy, m[i].out, T, uint64_t(m[i].out) * 2, 64, 128, t16);
          if (rc) return rc;
          const int rows_b = std::min(64, m[i].r - ch * 64);
          rc = make_tensor_map_2d(&mm.b, static_cast<const uint16_t*>(m[i].B) + size_t(ch) * 64 * m[i].out, m[i].out,
                                  rows_b, uint64_t(m[i].out) * 2, 64, 64, t16);
          if (rc) return rc;
          rc = make_tensor_map_2d(&mm.t, static_cast<const uint16_t*>(t_cat) + L.off[i] + ch * 64, 64, T,
                                  uint64_t(R) * 2, 64, 128, t16);
          if (rc) return rc;
          float* dB_part = reinterpret_cast<float*>(wsp + oB[i]) + size_t(ch) * pl.n_clusters * pl.out_pad * 64;
          rc = make_tensor_map_2d(&mm.dbp, dB_part, 64, uint64_t(pl.n_clusters) * pl.out_pad, 64 * 4, 32, 32, CU_TENSOR_MAP_DATA_TYPE_FLOAT32);
          if (rc) return rc;
          K2Member& km = p.m[j];
          const int nblk = ceil_div(m[i].out, 128);
          km.out = m[i].out;
          km.out_pad = pl.out_pad;
          km.bpg = pl.bpg;
          km.blk_first = ln * pl.blk_per_launch;
          km.blk_end = std::min(nblk, km.blk_first + pl.blk_per_launch);
          km.dt_accumulate = ln > 0;
          km.scale = m[i].scale;
          km.dt = static_cast<uint16_t*>(dt_cat) + L.off[i] + ch * 64;
          // algorithmic flops: dt and dB, un-padded r (SURVEY.md 8d)
          if (j < cnt && ln == 0) flops += 4.0 * double(T) * double(m[i].out) * double(rows_b);
        }
        ProfileScope prof(stream, PROF_GEMM_K2, flops);
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(pl0.G * cl_begin[cnt]);
        cfg.blockDim = dim3(kK2Threads);
        cfg.dynamicSmemBytes = kK2SmemTotal;
        cfg.stream = stream;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = pl0.G;
        at[0].val.clusterDim.y = 1;
        at[0].val.clusterDim.z = 1;
        cfg.attrs = at;
        cfg.numAttrs = pl0.G > 1 ? 1 : 0;
        SOWB_CHECK_CUDA(cudaLaunchKernelEx(&cfg, k2_kernel, maps, p));
      }
    }
  }

  // ---- dA_cat [in, R] = x^T . dt_cat: split-K over T into fp32 partials ------------------------------------
  float* partA = reinterpret_cast<float*>(wsp + oA);
  int splitsA = 1;
  bool need_dA = false;
  for (int i = 0; i < n; ++i) need_dA = need_dA || m[i].dA != nullptr;
  if (need_dA) {
    const float one = 1.0f;
    Segment sg{Operand{x, uint64_t(T), uint64_t(in), uint64_t(in)},         // A operand MN-major: [K=T rows, M=in cols]
               Operand{dt_cat, uint64_t(T), uint64_t(R), uint64_t(R)}, Ti};  // B operand MN-major: [K=T rows, N=R cols]
    int rsum = 0;
    for (int i = 0; i < n; ++i) rsum += m[i].r;
    rc = launch_skinny<true, true, EPI_F32_PARTIAL>(R, &sg, 1, nullptr, partA, R, in, &one, 1, true, f16, stream, PROF_GEMM_SPLITK,
                                                    2.0 * double(T) * double(in) * double(rsum), &splitsA);
    if (rc) return rc;
    if (splitsA > splitk_count(in, R, skinny_bn(R), Ti))
      return set_error(SOWB_EWORKSPACE, "sow_group_bwd: split-K count exceeds the workspace plan");
  }

  // ---- partials -> 16-bit dA_i (in, r_i), dB_i (r_i, out_i) ------------------------------------------------------
  {
    FinJobs jobs;
    jobs.n = 0;
    int blocks = 0;
    auto flush = [&]() -> int {
      if (jobs.n == 0) return SOWB_OK;
      if (f16) finalize_jobs_kernel<true><<<blocks, dim3(32, 32), 0, stream>>>(jobs);
      else finalize_jobs_kernel<false><<<blocks, dim3(32, 32), 0, stream>>>(jobs);
      SOWB_CHECK_CUDA(cudaGetLastError());
      jobs.n = 0;
      blocks = 0;
      return SOWB_OK;
    };
    auto add = [&](const float* src, int64_t stride, int splits, int rows, int cols, int ld_src, uint16_t* dst,
                   int ld_dst, int transpose) -> int {
      if (jobs.n == kMaxFinJobs) {
        const int rcf = flush();
        if (rcf) return rcf;
      }
      FinJob& J = jobs.j[jobs.n++];
      J.src = src;
      J.split_stride = stride;
      J.dst = dst;
      J.splits = splits;
      J.rows = rows;
      J.cols = cols;
      J.ld_src = ld_src;
      J.ld_dst = ld_dst;
      J.transpose = transpose;
      J.blk_begin = blocks;
      J.col_tiles = ceil_div(cols, 32);
      blocks += ceil_div(rows, 32) * J.col_tiles;
      return SOWB_OK;
    };
    for (int i = 0; i < n; ++i) {
      if (m[i].dA != nullptr) {
        rc = add(partA + L.off[i], int64_t(in) * R, splitsA, in, m[i].r, R, static_cast<uint16_t*>(m[i].dA), m[i].r, 0);
        if (rc) return rc;
      }
      if (m[i].dB != nullptr) {
        for (int ch = 0; ch < L.rpad[i] / 64; ++ch) {
          const int rows_b = std::min(64, m[i].r - ch * 64);
          const float* src = reinterpret_cast<float*>(wsp + oB[i]) + size_t(ch) * plans[i].n_clusters * plans[i].out_pad * 64;
          rc = add(src, int64_t(plans[i].out_pad) * 64, plans[i].n_clusters, m[i].out, rows_b, 64,
                   static_cast<uint16_t*>(m[i].dB) + size_t(ch) * 64 * m[i].out, m[i].out, 1);
          if (rc) return rc;
        }
      }
    }
    rc = flush();
    if (rc) return rc;
  }

  // ---- dbias_i = sum_T dY_i ---------------------------------------------------------------------------------------
  for (int i = 0; i < n; ++i) {
    if (m[i].dbias == nullptr) continue;
    float* partBias = reinterpret_cast<float*>(wsp + oBias);
    dim3 grid(ceil_div(m[i].out, 64), static_cast<unsigned>(std::min<int64_t>(kBiasParts, (T + 255) / 256)));
    const uint16_t* dy = static_cast<const uint16_t*>(m[i].dy);
    uint16_t* db = static_cast<uint16_t*>(m[i].dbias);
    if (f16) colsum_kernel<true><<<grid, dim3(64, 4), 0, stream>>>(dy, partBias, T, m[i].out);
    else colsum_kernel<false><<<grid, dim3(64, 4), 0, stream>>>(dy, partBias, T, m[i].out);
    SOWB_CHECK_CUDA(cudaGetLastError());
    if (f16) sum_partials_to_16_kernel<true><<<ceil_div(m[i].out, 256), 256, 0, stream>>>(partBias, db, m[i].out, int(grid.y));
    else sum_partials_to_16_kernel<false><<<ceil_div(m[i].out, 256), 256, 0, stream>>>(partBias, db, m[i].out, int(grid.y));
    SOWB_CHECK_CUDA(cudaGetLastError());
  }

  // ---- dX [T, in] = sum_i dY_i . W_i^T + dt_cat . A_cat^T: ONE launch, K-concatenated segments -------------------------
  if (dx != nullptr) {
    const float one = 1.0f;
    Segment segs[kMaxSeg];
    int ns = 0;
    // W (in,out) is K-major for this product: [N=in rows, K=out cols]
    const bool f32 = dtype == SOWB_F32;
    Segment tail{Operand{dt_cat, uint64_t(T), uint64_t(R), uint64_t(R)},
                 Operand{A_cat, uint64_t(in), uint64_t(R), uint64_t(R)}, R};   // [N=in rows, K=R cols]
    int nW = 0;
    for (int i = 0; i < n; ++i) nW += m[i].W != nullptr;
    if (nW * (f32 ? 3 : 1) + 1 > kMaxSeg)
      return set_error(SOWB_EINVAL, "sow_group_bwd: %d members with a dense W exceed one dX launch", nW);
    for (int i = 0; i < n; ++i) {
      if (m[i].W == nullptr) continue;
      const Operand opDY{m[i].dy, uint64_t(T), uint64_t(m[i].out), uint64_t(m[i].out)};
      const Operand opW{m[i].W, uint64_t(in), uint64_t(m[i].out), uint64_t(m[i].out)};
      segs[ns++] = Segment{opDY, opW, m[i].out};
      if (f32) {
        SOWB_REQUIRE(m[i].W_lo && m[i].dy_lo, "sow_group_bwd: SOWB_F32 needs the low pieces of W and dY (member %d)", i);
        segs[ns++] = Segment{opDY, Operand{m[i].W_lo, uint64_t(in), uint64_t(m[i].out), uint64_t(m[i].out)}, m[i].out};
        segs[ns++] = Segment{Operand{m[i].dy_lo, uint64_t(T), uint64_t(m[i].out), uint64_t(m[i].out)}, opW, m[i].out};
      }
    }
    segs[ns++] = tail;
    double kalg = 0;
    for (int i = 0; i < n; ++i) kalg += double(m[i].W != nullptr ? m[i].out : 0) + double(m[i].r);
    if (f32)
      rc = launch_gemm<256, false, false, EPI_F32_TMA>(segs, ns, nullptr, static_cast<float*>(dx), in, Ti, in, &one, 1, nullptr,
                                                       false, false, stream, PROF_GEMM_DX, 2.0 * double(T) * double(in) * kalg);
    else if (use_big_tiles(Ti, in, static_cast<int>(kalg) / kBK))
      rc = launch_gemm<256, false, false, EPI_BF16_TMA, 2>(segs, ns, dx, nullptr, in, Ti, in, &one, 1, nullptr, false, f16, stream,
                                                           PROF_GEMM_DX, 2.0 * double(T) * double(in) * kalg);
    else if (use_pair_tiles())
      rc = launch_gemm<256, false, false, EPI_BF16_TMA, 1, true>(segs, ns, dx, nullptr, in, Ti, in, &one, 1, nullptr, false, f16,
                                                                 stream, PROF_GEMM_DX, 2.0 * double(T) * double(in) * kalg);
    else
      rc = launch_gemm<256, false, false, EPI_BF16_TMA>(segs, ns, dx, nullptr, in, Ti, in, &one, 1, nullptr, false, f16, stream,
                                                        PROF_GEMM_DX, 2.0 * double(T) * double(in) * kalg);
    if (rc) return rc;
  }
  return SOWB_OK;
}

}  // extern "C"
