// Tensor-train path: truncated-QR decomposition pieces, reconstruction and the fused TT-Adam update.
//
// The reference's "TT-SVD" is a left-to-right sweep of COMPLETE Householder QR + truncation
// (tn_gradient/tt.py:127-136).  Keeping Q[:, :r] and R[:r, :] of a complete QR of L is exactly the orthogonal
// projection of L onto span(L[:, :r]):  Q_r = thin-QR(L[:, :r]),  R_r = Q_r^T L   (SURVEY.md section 7, verified
// to 1.9e-07), so the m x m orthogonal factor is never formed:
//     sow_thin_qr  : Q_r  (CGS2 -- classical Gram-Schmidt with re-orthogonalisation, fp32)
//     tt_project   : R_r = Q_r^T L   (fp32 FMA accumulate; TF32/bf16 would break the 1e-5 reconstruction bound)
// Reconstruction results are gauge-invariant, so parity is defined on reconstruct()/to_matrix(), never on cores.
#include "common.cuh"

#include <algorithm>

namespace sowb {

// ------------------------------------------------------------------------------------------------
// thin QR (batched; one CTA per matrix)
// ------------------------------------------------------------------------------------------------
constexpr int kQrThreads = 512;
constexpr int kQrWarps = kQrThreads / 32;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// CGS2 on a COLUMN-MAJOR work copy Wt[k][i] (r x m): every sweep is thread-per-row, so with this layout the 32
// lanes of a warp touch 32 consecutive floats of one column (one 128-byte wavefront) for every k.  (On the
// row-major layout the same sweeps cost one wavefront per element: measured 20 ms instead of < 1 ms for 4096x64.)
// Prologue / epilogue transpose X[:, :r] -> Wt and Wt -> Q through per-warp 32x33 smem tiles.
__device__ __forceinline__ void qr_transpose_in(const float* __restrict__ X, int ldx, float* __restrict__ Wt, int m,
                                                int r, float (*tile)[33], int warp, int lane) {
  const int tiles_i = (m + 31) / 32, tiles_k = (r + 31) / 32;
  for (int t = warp; t < tiles_i * tiles_k; t += kQrWarps) {
    const int i0 = (t / tiles_k) * 32, k0 = (t % tiles_k) * 32;
    for (int ii = 0; ii < 32; ++ii) {
      const int i = i0 + ii, k = k0 + lane;
      tile[ii][lane] = (i < m && k < r) ? X[static_cast<int64_t>(i) * ldx + k] : 0.f;
    }
    __syncwarp();
    for (int kk = 0; kk < 32; ++kk) {
      const int k = k0 + kk, i = i0 + lane;
      if (k < r && i < m) Wt[static_cast<int64_t>(k) * m + i] = tile[lane][kk];
    }
    __syncwarp();
  }
}
__device__ __forceinline__ void qr_transpose_out(const float* __restrict__ Wt, float* __restrict__ Q, int m, int r,
                                                 float (*tile)[33], int warp, int lane) {
  const int tiles_i = (m + 31) / 32, tiles_k = (r + 31) / 32;
  for (int t = warp; t < tiles_i * tiles_k; t += kQrWarps) {
    const int i0 = (t / tiles_k) * 32, k0 = (t % tiles_k) * 32;
    for (int kk = 0; kk < 32; ++kk) {
      const int k = k0 + kk, i = i0 + lane;
      tile[kk][lane] = (k < r && i < m) ? Wt[static_cast<int64_t>(k) * m + i] : 0.f;
    }
    __syncwarp();
    for (int ii = 0; ii < 32; ++ii) {
      const int i = i0 + ii, k = k0 + lane;
      if (i < m && k < r) Q[static_cast<int64_t>(i) * r + k] = tile[lane][ii];
    }
    __syncwarp();
  }
}

__global__ void __launch_bounds__(kQrThreads, 1)
thin_qr_kernel(const float* __restrict__ X, int64_t x_bs, int ldx, float* __restrict__ Q, int64_t q_bs,
               float* __restrict__ work, int m, int r) {
  extern __shared__ float qr_smem[];
  float* c = qr_smem;                 // [r]      projection coefficients
  float* red = qr_smem + r;           // [kQrWarps * 64] cross-warp partials
  float (*tiles)[33] = reinterpret_cast<float (*)[33]>(red + kQrWarps * 64);   // [kQrWarps][32][33]
  __shared__ float s_norm;
  const float* Xb = X + blockIdx.x * x_bs;
  float* Qb = Q + blockIdx.x * q_bs;
  float* Wt = work + static_cast<int64_t>(blockIdx.x) * m * r;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  qr_transpose_in(Xb, ldx, Wt, m, r, tiles + warp * 32, warp, lane);
  __syncthreads();

  for (int j = 0; j < r; ++j) {
    float* colj = Wt + static_cast<int64_t>(j) * m;
    for (int pass = 0; pass < 2 && j > 0; ++pass) {
      // c[k] = sum_i Wt[k][i] * Wt[j][i], k < j, in chunks of 32 coefficients held in registers
      for (int k0 = 0; k0 < j; k0 += 32) {
        const int kn = min(32, j - k0);
        float part[32];
#pragma unroll
        for (int k = 0; k < 32; ++k) part[k] = 0.f;
        for (int i = tid; i < m; i += kQrThreads) {
          const float v = colj[i];
#pragma unroll
          for (int k = 0; k < 32; ++k)
            if (k < kn) part[k] = fmaf(Wt[static_cast<int64_t>(k0 + k) * m + i], v, part[k]);
        }
#pragma unroll
        for (int k = 0; k < 32; ++k) {
          if (k < kn) {
            const float s = warp_sum(part[k]);
            if (lane == 0) red[warp * 64 + k] = s;
          }
        }
        __syncthreads();
        if (tid < kn) {
          float s = 0.f;
#pragma unroll
          for (int w = 0; w < kQrWarps; ++w) s += red[w * 64 + tid];
          c[k0 + tid] = s;
        }
        __syncthreads();
      }
      // Wt[j][i] -= sum_k Wt[k][i] c[k]
      for (int i = tid; i < m; i += kQrThreads) {
        float acc = 0.f;
        for (int k = 0; k < j; ++k) acc = fmaf(Wt[static_cast<int64_t>(k) * m + i], c[k], acc);
        colj[i] -= acc;
      }
      __syncthreads();
    }
    // normalise
    float ss = 0.f;
    for (int i = tid; i < m; i += kQrThreads) {
      const float v = colj[i];
      ss = fmaf(v, v, ss);
    }
    ss = warp_sum(ss);
    if (lane == 0) red[warp] = ss;
    __syncthreads();
    if (tid == 0) {
      float s = 0.f;
      for (int w = 0; w < kQrWarps; ++w) s += red[w];
      s_norm = s;
    }
    __syncthreads();
    const float nrm2 = s_norm;
    const float inv = (nrm2 > 1e-37f) ? rsqrtf(nrm2) : 0.f;   // rank-deficient column -> zero vector
    for (int i = tid; i < m; i += kQrThreads) colj[i] *= inv;
    __syncthreads();
  }
  qr_transpose_out(Wt, Qb, m, r, tiles + warp * 32, warp, lane);
}

// ------------------------------------------------------------------------------------------------
// Cholesky-QR for r <= 64 (the TT ranks 8-64 and the SoW rank 50): three fully parallel passes instead of one CTA
// walking the columns.  All intermediate arithmetic is fp64, so a single pass keeps |Q^T Q - I| at fp32 rounding
// level up to cond(X) ~ 1e6 (Gram error ~ cond^2 * 2^-53):
//     G = X^T X (fp64, all SMs)  ->  G = L L^T (one CTA)  ->  q_row . L^T = x_row by forward substitution (all SMs)
// R = L^T has a positive diagonal: same sign convention as the CGS2 kernel.  A column whose pivot vanishes
// (d_j <= 1e-12 * G_jj: linearly dependent on the previous ones) yields a ZERO column of Q, like CGS2's zero-norm rule.
// Orthogonality degrades as cond(X)^2 * 2^-53 = 2^-53 / min_j(d_j / G_jj): when a surviving pivot ratio drops below
// 1e-8 (cond >~ 1e4 -- e.g. the all-positive, nearly rank-one leading columns of a TT-Adam second-moment unfolding) the
// Cholesky kernel raises the matrix's flag and a SECOND Cholesky-QR pass over Q (CholeskyQR2, same three kernels, still
// fp64 inside) restores |Q^T Q - I| to rounding level without moving the subspace (a re-orthogonalised fp32 Gram-Schmidt
// would keep Q orthonormal but tilt its span by eps32 * cond).  For well-conditioned inputs the three extra launches exit
// at their first instruction.
// ------------------------------------------------------------------------------------------------
constexpr int kCqMaxR = 64;
constexpr int kCqRows = 128;
constexpr int kCqGramRows = 64;    // rows per Gram block: the fp64 pipe is narrow, so the work is spread over more SMs
// per-matrix factor block: L (64 x 64, lower) | dinv (64) | W = L^-T (64 x 64, upper: the operand of the tensor-core solve)
constexpr int kCqFac = 2 * kCqMaxR * kCqMaxR + kCqMaxR;
constexpr size_t kCqWsPerBatch = kCqFac * sizeof(double);

// Gram partials: CTA (x, b) accumulates X_b[rows]^T X_b[rows] in fp64 over the 128-row blocks x, x + gridDim.x, ... (fixed
// order) and stores the lower triangle compactly, part[(b * gridDim.x + x)][i * r + j].  cq_sum_kernel adds the
// partials in block order, so the whole factorisation is bit-reproducible (no fp64 atomics).
// RT = ceil(r / 16): a thread owns the RT x RT entries G[ty + 16a][tx + 16c] (r = 8: one fp64 FMA and two conversions per
// row instead of 16 + 8 -- the f32 -> f64 conversions, not the FMAs, bound the untemplated loop)
template <int RT>
__global__ void __launch_bounds__(256)
cq_gram_kernel(const float* __restrict__ X, int64_t x_bs, int ldx, double* __restrict__ part, int m, int r,
               const int* __restrict__ only_if) {
  pdl_trigger();
  pdl_wait();
  if (only_if != nullptr && only_if[blockIdx.y] == 0) return;      // second pass: flagged matrices only
  __shared__ float sx[kCqGramRows][kCqMaxR + 1];
  const float* Xb = X + blockIdx.y * x_bs;
  double* G = part + (static_cast<int64_t>(blockIdx.y) * gridDim.x + blockIdx.x) * (r * r);
  const int tid = threadIdx.x;
  const int ty = tid >> 4, tx = tid & 15;   // G[ty + 16a][tx + 16c]
  double acc[RT][RT];
#pragma unroll
  for (int a = 0; a < RT; ++a)
#pragma unroll
    for (int c = 0; c < RT; ++c) acc[a][c] = 0.0;
  for (int row0 = blockIdx.x * kCqGramRows; row0 < m; row0 += gridDim.x * kCqGramRows) {
    const int rows = min(kCqGramRows, m - row0);
    __syncthreads();
    for (int idx = tid; idx < rows * r; idx += 256) {
      const int i = idx / r, k = idx - i * r;
      sx[i][k] = Xb[static_cast<int64_t>(row0 + i) * ldx + k];
    }
    __syncthreads();
    for (int i = 0; i < rows; ++i) {
      double xa[RT], xc[RT];
#pragma unroll
      for (int a = 0; a < RT; ++a) xa[a] = (ty + 16 * a < r) ? static_cast<double>(sx[i][ty + 16 * a]) : 0.0;
#pragma unroll
      for (int c = 0; c < RT; ++c) xc[c] = (tx + 16 * c < r) ? static_cast<double>(sx[i][tx + 16 * c]) : 0.0;
#pragma unroll
      for (int a = 0; a < RT; ++a)
#pragma unroll
        for (int c = 0; c < RT; ++c) acc[a][c] = fma(xa[a], xc[c], acc[a][c]);
    }
  }
#pragma unroll
  for (int a = 0; a < RT; ++a)
#pragma unroll
    for (int c = 0; c < RT; ++c) {
      const int i = ty + 16 * a, j = tx + 16 * c;
      if (i < r && j < r && j <= i) G[i * r + j] = acc[a][c];   // lower triangle is enough
    }
}

// G[i][j] (lower triangle of the matrix's 64 x 64 block) = sum of its Gram partials in block order: one entry per thread,
// the loads of eight partials in flight at a time.  grid (ceil(r*r / 256), batch)
__global__ void __launch_bounds__(256)
cq_sum_kernel(const double* __restrict__ part, int n_part, int r, double* __restrict__ ws, const int* __restrict__ only_if) {
  pdl_trigger();
  pdl_wait();
  if (only_if != nullptr && only_if[blockIdx.y] == 0) return;
  const int e = blockIdx.x * 256 + threadIdx.x;
  const int rr = r * r;
  if (e >= rr) return;
  const int i = e / r, j = e - i * r;
  if (j > i) return;
  const double* pp = part + static_cast<int64_t>(blockIdx.y) * n_part * rr + e;
  double g = 0.0;
  int q = 0;
  for (; q + 8 <= n_part; q += 8) {
    double v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) v[u] = pp[static_cast<int64_t>(q + u) * rr];
#pragma unroll
    for (int u = 0; u < 8; ++u) g += v[u];
  }
  for (; q < n_part; ++q) g += pp[static_cast<int64_t>(q) * rr];
  ws[blockIdx.y * kCqFac + i * kCqMaxR + j] = g;
}

// In place: lower triangle of G -> L; dinv[j] = 1 / L_jj (0 for a dependent column).  1024 threads, 4 entries each.
// Right-looking Cholesky with the column scaling deferred: step j only needs the pivot d_j = A[j][j] and the unscaled
// column j, A[i][k] -= A[i][j] A[k][j] / d_j, so there is ONE barrier per step; L = A . diag(d)^-1/2 at the end.
__global__ void __launch_bounds__(1024)
cq_chol_kernel(double* __restrict__ ws, const double* __restrict__ part, int n_part, int r, int* __restrict__ flags,
               const int* __restrict__ only_if, int want_inv) {
  pdl_trigger();
  pdl_wait();
  if (only_if != nullptr && only_if[blockIdx.x] == 0) return;
  extern __shared__ __align__(16) double chol_smem[];
  double (*A)[kCqMaxR + 1] = reinterpret_cast<double (*)[kCqMaxR + 1]>(chol_smem);
  double (*Li)[kCqMaxR + 1] = A + kCqMaxR;                          // L^-1 (want_inv)
  double* g0 = reinterpret_cast<double*>(Li + kCqMaxR);
  double* dfin = g0 + kCqMaxR;          // final pivots (0 for a dependent column)
  double* G = ws + blockIdx.x * kCqFac;
  double* dinv = G + kCqMaxR * kCqMaxR;
  const int tid = threadIdx.x;
  const int i = tid >> 4, kb = tid & 15;
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const int k = kb + 16 * c;
    double g = 0.0;
    if (i < r && k <= i) {
      if (part == nullptr) {
        g = G[i * kCqMaxR + k];
      } else {
        // small ranks: the fixed-order sum of the Gram partials happens here (no separate cq_sum_kernel launch)
        const int rr = r * r;
        const double* pp = part + static_cast<int64_t>(blockIdx.x) * n_part * rr + i * r + k;
        int q = 0;
        for (; q + 8 <= n_part; q += 8) {
          double v[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) v[u] = pp[static_cast<int64_t>(q + u) * rr];
#pragma unroll
          for (int u = 0; u < 8; ++u) g += v[u];
        }
        for (; q < n_part; ++q) g += pp[static_cast<int64_t>(q) * rr];
      }
    }
    A[i][k] = g;
  }
  __syncthreads();
  if (tid < kCqMaxR) g0[tid] = A[tid][tid];
  __syncthreads();
  bool weak = false;                                                // thread 0: some surviving pivot ratio < 1e-9
  for (int j = 0; j < r; ++j) {
    const double d = A[j][j];                                       // final after step j-1 (broadcast read)
    const bool alive = (g0[j] > 1e-300) && (d > 1e-12 * g0[j]);
    if (tid == 0) {
      dfin[j] = alive ? d : 0.0;
      weak = weak || (alive && d < 1e-8 * g0[j]);
    }
    if (alive && i > j && i < r) {
      const double f = A[i][j] * __drcp_rn(d);     // reciprocal + multiply: the fp64 divide is the longest link of the 64-step chain
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int k = kb + 16 * c;
        if (k > j && k <= i) A[i][k] -= f * A[k][j];
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const int k = kb + 16 * c;
    if (i < r && k <= i) {
      const double d = dfin[k];
      const double s = d > 0.0 ? rsqrt(d) : 0.0;
      const double lv = (k == i) ? (d > 0.0 ? sqrt(d) : 1.0) : A[i][k] * s;      // dependent column: L_jj = 1, rest 0
      G[i * kCqMaxR + k] = lv;
      A[i][k] = lv;                                                               // own entry: L stays in smem for the inverse
    }
  }
  if (tid < r) {
    const double d = dfin[tid];
    const double di = d > 0.0 ? rsqrt(d) : 0.0;
    dinv[tid] = di;
    g0[tid] = di;                                                                 // g0 is dead: dinv for the inverse below
  }
  if (tid == 0 && flags != nullptr) flags[blockIdx.x] = weak ? 1 : 0;
  if (!want_inv) return;
  // The tensor-core solve is a forward substitution blocked by 8 columns: it needs L and the inverses of the eight 8 x 8
  // diagonal blocks of L only (an explicit 64 x 64 inverse is a 64-step chain of dependent fp64 operations: 30 us).
  // Thread (b, c), tid < 64: column c of inv(L_bb), eight unrolled steps; stored transposed as W[8b + c][8b + j], j >= c.
  __syncthreads();
  if (tid < kCqMaxR) {
    const int b8 = (tid >> 3) * 8, c = tid & 7;
    double y[8];
#pragma unroll
    for (int i2 = 0; i2 < 8; ++i2) {
      double sum = 0.0;
#pragma unroll
      for (int k = 0; k < 8; ++k)
        if (k >= c && k < i2) sum = fma(A[b8 + i2][b8 + k], y[k], sum);
      y[i2] = (i2 < c) ? 0.0 : (i2 == c ? g0[b8 + c] : -sum * g0[b8 + i2]);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) Li[b8 + c][b8 + j] = y[j];          // Li[k][j] = inv(L_bb)[j][k]: already transposed
  }
  __syncthreads();
  double* Wg = G + kCqMaxR * kCqMaxR + kCqMaxR;
  for (int idx = tid; idx < kCqMaxR * kCqMaxR; idx += 1024) {
    const int k = idx >> 6, j = idx & 63;
    Wg[idx] = ((k >> 3) == (j >> 3) && k <= j && j < r) ? Li[k][j] : 0.0;
  }
}

// ---- tensor-core (fp64 mma.sync m8n8k4) Gram and solve for ranks above 16 ------------------------------------------------
// The CUDA-core fp64 rate bounds the scalar kernels (2 x 4096 x 64: Gram 21 us, solve 32 us); the same products on the fp64
// tensor path.  Shared tiles are doubles with a 68-element pitch: both fragment patterns (row = lane & 3, column = base +
// (lane >> 2), and row = base + (lane >> 2), column = lane & 3) then hit every bank pair exactly twice.
constexpr int kCqLd = 68;
__device__ __forceinline__ void dmma_8x8x4(double (&c)[2], double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
               : "+d"(c[0]), "+d"(c[1])
               : "d"(a), "d"(b));
}

// part[(b * gridDim.x + x)][i * r + j] (lower triangle) = X_b[rows]^T X_b[rows] over the 64-row blocks x, x + gridDim.x, ...
__global__ void __launch_bounds__(256)
cq_gram_mma_kernel(const float* __restrict__ X, int64_t x_bs, int ldx, double* __restrict__ part, int m, int r,
                   const int* __restrict__ only_if) {
  pdl_trigger();
  pdl_wait();
  if (only_if != nullptr && only_if[blockIdx.y] == 0) return;
  extern __shared__ __align__(16) double cq_mma_smem[];
  double* sX = cq_mma_smem;                                  // [64 rows][kCqLd]
  const float* Xb = X + blockIdx.y * x_bs;
  double* G = part + (static_cast<int64_t>(blockIdx.y) * gridDim.x + blockIdx.x) * (r * r);
  const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31;
  const int r8 = (r + 7) & ~7, rb = r8 >> 3;
  const int fr = lane & 3, fc = lane >> 2;
  double acc[8][2];
#pragma unroll
  for (int jb = 0; jb < 8; ++jb) acc[jb][0] = acc[jb][1] = 0.0;
  for (int row0 = blockIdx.x * kCqGramRows; row0 < m; row0 += gridDim.x * kCqGramRows) {
    __syncthreads();
    for (int idx = tid; idx < kCqGramRows * r8; idx += 256) {
      const int i = idx / r8, k = idx - i * r8;
      sX[i * kCqLd + k] = (row0 + i < m && k < r) ? static_cast<double>(Xb[static_cast<int64_t>(row0 + i) * ldx + k]) : 0.0;
    }
    __syncthreads();
    if (w < rb) {
#pragma unroll 4
      for (int ks = 0; ks < kCqGramRows / 4; ++ks) {
        const double* rowp = sX + (4 * ks + fr) * kCqLd + fc;
        const double a = rowp[8 * w];
#pragma unroll
        for (int jb = 0; jb < 8; ++jb)
          if (jb <= w) dmma_8x8x4(acc[jb], a, rowp[8 * jb]);
      }
    }
  }
  if (w < rb) {
#pragma unroll
    for (int jb = 0; jb < 8; ++jb) {
      if (jb > w) continue;
      const int i = 8 * w + fc;
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int j = 8 * jb + 2 * fr + e;
        if (i < r && j <= i) G[i * r + j] = acc[jb][e];
      }
    }
  }
}

// Q = X . L^-T as a forward substitution blocked by 8 columns, 64 rows per CTA, a warp owns 8 rows:
//   Y_j = X_j - sum_{b < j} Q_b . L[j-block, b-block]^T   (2 j MMAs on one accumulator),   Q_j = Y_j . inv(L_jj)^T   (2 MMAs)
// Y_j and Q_j go back to the warp's rows of the shared X tile (the accumulator layout is not the A-operand layout), so only
// __syncwarp separates the stages.
__global__ void __launch_bounds__(256)
cq_solve_mma_kernel(const float* __restrict__ X, int64_t x_bs, int ldx, float* __restrict__ Q, int64_t q_bs,
                    const double* __restrict__ ws, int m, int r, const int* __restrict__ only_if) {
  pdl_trigger();
  pdl_wait();
  if (only_if != nullptr && only_if[blockIdx.y] == 0) return;
  extern __shared__ __align__(16) double cq_mma_smem[];
  double* sX = cq_mma_smem;                                  // [64 rows][kCqLd]: x, then y, then q
  double* sL = sX + 64 * kCqLd;                              // [64 j][kCqLd]: L[j][k]
  double* sD = sL + 64 * kCqLd;                              // [64 k][kCqLd]: inv(L_bb)^T blocks (W of the Cholesky kernel)
  const double* Gg = ws + blockIdx.y * kCqFac;
  const double* Wg = Gg + kCqMaxR * kCqMaxR + kCqMaxR;
  const float* Xb = X + blockIdx.y * x_bs;
  float* Qb = Q + blockIdx.y * q_bs;
  const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31;
  const int r8 = (r + 7) & ~7, rb = r8 >> 3;
  const int fr = lane & 3, fc = lane >> 2;
  const int row0 = blockIdx.x * 64;
  for (int idx = tid; idx < r8 * r8; idx += 256) {
    const int j = idx / r8, k = idx - j * r8;
    sL[j * kCqLd + k] = (j < r && k <= j) ? Gg[j * kCqMaxR + k] : 0.0;
    sD[j * kCqLd + k] = Wg[j * kCqMaxR + k];
  }
  for (int idx = tid; idx < 64 * r8; idx += 256) {
    const int i = idx / r8, k = idx - i * r8;
    sX[i * kCqLd + k] = (row0 + i < m && k < r) ? static_cast<double>(Xb[static_cast<int64_t>(row0 + i) * ldx + k]) : 0.0;
  }
  __syncthreads();
  double* xw = sX + (8 * w) * kCqLd;                          // this warp's 8 rows
  const int row = row0 + 8 * w + fc;
  for (int jb = 0; jb < rb; ++jb) {
    double acc[2];
    acc[0] = xw[fc * kCqLd + 8 * jb + 2 * fr];
    acc[1] = xw[fc * kCqLd + 8 * jb + 2 * fr + 1];
    // Y_j: minus the finished blocks; A = -Q[:, k0..k0+3], B[kk][jj] = L[8 jb + jj][k0 + kk]
    for (int ks = 0; ks < 2 * jb; ++ks) {
      const double a = -xw[fc * kCqLd + 4 * ks + fr];
      const double bq = sL[(8 * jb + fc) * kCqLd + 4 * ks + fr];
      dmma_8x8x4(acc, a, bq);
    }
    __syncwarp();
    xw[fc * kCqLd + 8 * jb + 2 * fr] = acc[0];
    xw[fc * kCqLd + 8 * jb + 2 * fr + 1] = acc[1];
    __syncwarp();
    // Q_j = Y_j . inv(L_jj)^T: B[kk][jj] = sD[8 jb + k0 + kk][8 jb + jj]
    double q[2] = {0.0, 0.0};
#pragma unroll
    for (int s2 = 0; s2 < 2; ++s2) {
      const double a = xw[fc * kCqLd + 8 * jb + 4 * s2 + fr];
      const double bq = sD[(8 * jb + 4 * s2 + fr) * kCqLd + 8 * jb + fc];
      dmma_8x8x4(q, a, bq);
    }
    __syncwarp();
    xw[fc * kCqLd + 8 * jb + 2 * fr] = q[0];
    xw[fc * kCqLd + 8 * jb + 2 * fr + 1] = q[1];
    __syncwarp();
    if (row < m) {
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int j = 8 * jb + 2 * fr + e;
        if (j < r) Qb[static_cast<int64_t>(row) * r + j] = static_cast<float>(q[e]);
      }
    }
  }
}

// Q[row, :] = x_row . R^-1 with R = L^T:  q_j = (x_j - sum_{k<j} q_k L_jk) * dinv_j, one row per thread, fp64.
// RQ = r rounded up to 8 / 16 / 32 / 64 bounds the unrolled substitution (the r = 8 instance is 28 FMAs, not a walk through
// the 2016-FMA code of the r = 64 one).
template <int RQ>
__global__ void __launch_bounds__(kCqRows)
cq_solve_kernel(const float* __restrict__ X, int64_t x_bs, int ldx, float* __restrict__ Q, int64_t q_bs,
                const double* __restrict__ ws, int m, int r, const int* __restrict__ only_if) {
  pdl_trigger();
  pdl_wait();
  if (only_if != nullptr && only_if[blockIdx.y] == 0) return;
  extern __shared__ double cq_smem[];
  double (*sL)[kCqMaxR + 1] = reinterpret_cast<double (*)[kCqMaxR + 1]>(cq_smem);   // sL[k][j] = L_jk (broadcast reads)
  double* sdinv = cq_smem + kCqMaxR * (kCqMaxR + 1);
  float (*sx)[kCqMaxR + 1] = reinterpret_cast<float (*)[kCqMaxR + 1]>(sdinv + kCqMaxR);
  const double* G = ws + blockIdx.y * kCqFac;
  const float* Xb = X + blockIdx.y * x_bs;
  float* Qb = Q + blockIdx.y * q_bs;
  const int tid = threadIdx.x;
  const int row0 = blockIdx.x * kCqRows;
  const int rows = min(kCqRows, m - row0);
  for (int idx = tid; idx < r * r; idx += kCqRows) {
    const int j = idx / r, k = idx - j * r;
    sL[k][j] = (k <= j) ? G[j * kCqMaxR + k] : 0.0;
  }
  if (tid < r) sdinv[tid] = G[kCqMaxR * kCqMaxR + tid];
  for (int idx = tid; idx < rows * r; idx += kCqRows) {
    const int i = idx / r, k = idx - i * r;
    sx[i][k] = Xb[static_cast<int64_t>(row0 + i) * ldx + k];
  }
  __syncthreads();
  if (tid < rows) {
    double q[RQ];
#pragma unroll
    for (int j = 0; j < RQ; ++j) {
      q[j] = 0.0;
      if (j < r) {
        // four independent partial sums: the fp64 FMA chain is latency-bound with one row per thread
        double a0 = static_cast<double>(sx[tid][j]), a1 = 0.0, a2 = 0.0, a3 = 0.0;
#pragma unroll
        for (int k = 0; k < j; ++k) {
          if ((k & 3) == 0) a0 = fma(-q[k], sL[k][j], a0);
          else if ((k & 3) == 1) a1 = fma(-q[k], sL[k][j], a1);
          else if ((k & 3) == 2) a2 = fma(-q[k], sL[k][j], a2);
          else a3 = fma(-q[k], sL[k][j], a3);
        }
        q[j] = ((a0 + a1) + (a2 + a3)) * sdinv[j];
      }
    }
#pragma unroll
    for (int j = 0; j < RQ; ++j)
      if (j < r) sx[tid][j] = static_cast<float>(q[j]);
  }
  __syncthreads();
  for (int idx = tid; idx < rows * r; idx += kCqRows) {
    const int i = idx / r, k = idx - i * r;
    Qb[static_cast<int64_t>(row0 + i) * r + k] = sx[i][k];
  }
}

// Measured and dropped: a variant blocked by 8 columns (finished q_k in shared memory, dynamic loop over the finished columns,
// only the 8 x 8 triangle unrolled; 64 rows per CTA).  Same 32 us for 2 x 4096 x 64 and 0.91 ms instead of 0.69 ms for the
// 168 x 2736 x 50 re-initialisation batch: the fp64 FMA rate of the CUDA cores bounds both, not instruction fetch.

// ------------------------------------------------------------------------------------------------
// projection R[r, n] = Q[m, r]^T L[m, n]    (fp32, register-tiled; split over m into per-split partials that
// sum_splits_kernel adds in split order: bit-reproducible, no atomics)
// ------------------------------------------------------------------------------------------------
// dst[b][i] = sum_s part[b][s][i], s ascending (fixed order).  grid (blocks, batch)
__global__ void sum_splits_kernel(const float* __restrict__ part, int splits, int64_t split_stride, int64_t part_bs,
                                  float* __restrict__ dst, int64_t dst_bs, int64_t n) {
  pdl_trigger();
  pdl_wait();
  const float* pb = part + blockIdx.y * part_bs;
  float* db = dst + blockIdx.y * dst_bs;
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
    float s = pb[i];
#pragma unroll 4
    for (int k = 1; k < splits; ++k) s += pb[k * split_stride + i];
    db[i] = s;
  }
}

int launch_sum_splits(const float* part, int splits, int64_t split_stride, int64_t part_bs, float* dst, int64_t dst_bs,
                      int64_t n, int batch, cudaStream_t stream) {
  const int blocks = static_cast<int>(std::min<int64_t>((n + 255) / 256, int64_t(num_sms()) * 8));
  SOWB_CHECK_CUDA(launch_pdl(sum_splits_kernel, dim3(blocks, batch), dim3(256), 0, stream, part, splits, split_stride, part_bs, dst, dst_bs, n));
  return SOWB_OK;
}

constexpr int kPjTN = 128;   // columns of L per CTA
constexpr int kPjTM = 32;    // rows of L per smem stage
constexpr int kPjThreads = 256;
constexpr int kPjRT = 64;    // rank tile

// thread layout: 16 (r) x 16 (n); each thread owns 4 (r) x (4 + 4) (n) outputs of a 64 x 128 tile: rank rows
// tr*4..+3, columns tn*4..+3 and 64+tn*4..+3, so that every shared-memory operand is one conflict-free 16-byte load
// (3 LDS.128 per 32 FMA: FMA-bound, not LDS-bound).  The next K stage is prefetched into registers during the FMAs.
__global__ void __launch_bounds__(kPjThreads)
tt_project_kernel(const float* __restrict__ L, int64_t l_bs, const float* __restrict__ Q, int64_t q_bs,
                  float* __restrict__ R, int64_t r_bs, int64_t split_stride, int m, int n, int r, int m_per_split) {
  __shared__ __align__(16) float sL[kPjTM][kPjTN];
  __shared__ __align__(16) float sQ[kPjTM][kPjRT];
  const int b = blockIdx.z;
  const float* Lb = L + b * l_bs;
  const float* Qb = Q + b * q_bs;
  float* Rb = R + b * r_bs + blockIdx.y * split_stride;   // split s stores its own partial (split_stride 0: one split)
  const int n0 = blockIdx.x * kPjTN;
  const int m_begin = blockIdx.y * m_per_split;
  const int m_end = min(m, m_begin + m_per_split);
  const int tid = threadIdx.x;
  const int tr = tid / 16, tn = tid % 16;
  const bool vec = ((n & 3) == 0) && ((reinterpret_cast<uintptr_t>(Lb) & 15) == 0);
  // staging assignment: L tile = 32 rows x 32 float4 -> 4 float4 per thread; Q tile = 32 x 64 floats -> 8 per thread
  float4 pl[4];
  float pq[8];
  for (int r0 = 0; r0 < r; r0 += kPjRT) {
    float acc[4][8];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int c = 0; c < 8; ++c) acc[a][c] = 0.f;
    auto fetch = [&](int mm0) {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int idx = tid + u * kPjThreads;          // 0..1023
        const int i = idx >> 5, c4 = (idx & 31) * 4;
        const int gi = mm0 + i, gc = n0 + c4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (gi < m_end) {
          const float* src = Lb + static_cast<int64_t>(gi) * n + gc;
          if (vec && gc + 3 < n) {
            v = *reinterpret_cast<const float4*>(src);
          } else {
            if (gc < n) v.x = src[0];
            if (gc + 1 < n) v.y = src[1];
            if (gc + 2 < n) v.z = src[2];
            if (gc + 3 < n) v.w = src[3];
          }
        }
        pl[u] = v;
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int idx = tid + u * kPjThreads;          // 0..2047
        const int i = idx >> 6, k = idx & 63;
        const int gi = mm0 + i, gk = r0 + k;
        pq[u] = (gi < m_end && gk < r) ? Qb[static_cast<int64_t>(gi) * r + gk] : 0.f;
      }
    };
    auto stash = [&]() {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int idx = tid + u * kPjThreads;
        *reinterpret_cast<float4*>(&sL[idx >> 5][(idx & 31) * 4]) = pl[u];
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int idx = tid + u * kPjThreads;
        sQ[idx >> 6][idx & 63] = pq[u];
      }
    };
    if (m_begin < m_end) fetch(m_begin);
    for (int mm0 = m_begin; mm0 < m_end; mm0 += kPjTM) {
      stash();
      __syncthreads();
      if (mm0 + kPjTM < m_end) fetch(mm0 + kPjTM);
#pragma unroll 8
      for (int i = 0; i < kPjTM; ++i) {
        const float4 q = *reinterpret_cast<const float4*>(&sQ[i][tr * 4]);
        const float4 l0 = *reinterpret_cast<const float4*>(&sL[i][tn * 4]);
        const float4 l1 = *reinterpret_cast<const float4*>(&sL[i][64 + tn * 4]);
        const float qv[4] = {q.x, q.y, q.z, q.w};
        const float lv[8] = {l0.x, l0.y, l0.z, l0.w, l1.x, l1.y, l1.z, l1.w};
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int c = 0; c < 8; ++c) acc[a][c] = fmaf(qv[a], lv[c], acc[a][c]);
      }
      __syncthreads();
    }
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      const int gr = r0 + tr * 4 + a;
      if (gr >= r) continue;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const int gc = n0 + (c < 4 ? tn * 4 + c : 64 + tn * 4 + (c - 4));
        if (gc < n) Rb[static_cast<int64_t>(gr) * n + gc] = acc[a][c];
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// pad + interleave / de-interleave for arbitrary order (tt.py:58,65,33 ; tt.py:242-247, utils.py:86-87)
//   interleaved index: digits (i1,o1,i2,o2,...,id,od), i_k base mm, o_k base nn
//   matrix index     : row = (i1..id) base mm, col = (o1..od) base nn
// ------------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ float load_as_f32(const T* p, int64_t i);
template <>
__device__ __forceinline__ float load_as_f32<float>(const float* p, int64_t i) { return p[i]; }
template <>
__device__ __forceinline__ float load_as_f32<__nv_bfloat16>(const __nv_bfloat16* p, int64_t i) {
  return __bfloat162float(p[i]);
}
template <typename T>
__device__ __forceinline__ void store_from_f32(T* p, int64_t i, float v);
template <>
__device__ __forceinline__ void store_from_f32<float>(float* p, int64_t i, float v) { p[i] = v; }
template <>
__device__ __forceinline__ void store_from_f32<__nv_bfloat16>(__nv_bfloat16* p, int64_t i, float v) {
  p[i] = __float2bfloat16(v);
}

// 4 consecutive elements at an index that is a multiple of 4 (8-byte bf16 / 16-byte fp32 accesses)
template <typename T>
__device__ __forceinline__ void load4_as_f32(const T* p, int64_t i, float (&v)[4]);
template <>
__device__ __forceinline__ void load4_as_f32<float>(const float* p, int64_t i, float (&v)[4]) {
  const float4 t = *reinterpret_cast<const float4*>(p + i);
  v[0] = t.x, v[1] = t.y, v[2] = t.z, v[3] = t.w;
}
template <>
__device__ __forceinline__ void load4_as_f32<__nv_bfloat16>(const __nv_bfloat16* p, int64_t i, float (&v)[4]) {
  const uint2 t = *reinterpret_cast<const uint2*>(p + i);
  v[0] = __uint_as_float(t.x << 16), v[1] = __uint_as_float(t.x & 0xffff0000u);
  v[2] = __uint_as_float(t.y << 16), v[3] = __uint_as_float(t.y & 0xffff0000u);
}
template <typename T>
__device__ __forceinline__ void store4_from_f32(T* p, int64_t i, const float (&v)[4]);
template <>
__device__ __forceinline__ void store4_from_f32<float>(float* p, int64_t i, const float (&v)[4]) {
  *reinterpret_cast<float4*>(p + i) = make_float4(v[0], v[1], v[2], v[3]);
}
template <>
__device__ __forceinline__ void store4_from_f32<__nv_bfloat16>(__nv_bfloat16* p, int64_t i, const float (&v)[4]) {
  __nv_bfloat162 lo = __floats2bfloat162_rn(v[0], v[1]), hi = __floats2bfloat162_rn(v[2], v[3]);
  uint2 t;
  t.x = *reinterpret_cast<uint32_t*>(&lo);
  t.y = *reinterpret_cast<uint32_t*>(&hi);
  *reinterpret_cast<uint2*>(p + i) = t;
}

// Division of a 32-bit index by a run-time constant d (>= 1) without the ~25-instruction software divide:
// q = (mulhi(n, M) + n) >> s with s = ceil(log2 d), M = floor(2^32 * (2^s - d) / d) + 1 (exact for all 32-bit n).
struct FastDiv {
  uint32_t d, M, s;
};
static inline FastDiv make_fastdiv(uint32_t d) {
  FastDiv f;
  f.d = d;
  uint32_t s = 0;
  while ((uint64_t(1) << s) < d) ++s;
  f.s = s;
  f.M = static_cast<uint32_t>(((uint64_t(1) << 32) * ((uint64_t(1) << s) - d)) / d + 1);
  return f;
}
__device__ __forceinline__ uint32_t fdiv(uint32_t n, const FastDiv& f) {
  return static_cast<uint32_t>((static_cast<uint64_t>(__umulhi(n, f.M)) + n) >> f.s);
}

__device__ __forceinline__ void decode_interleaved(uint32_t idx, const FastDiv& fm, const FastDiv& fn, int order,
                                                   int64_t& row, int64_t& col) {
  // idx = ((((i1*nn + o1)*mm + i2)*nn + o2) ... ); peel digits from the least significant end
  int64_t rmul = 1, cmul = 1;
  row = 0;
  col = 0;
  for (int k = 0; k < order; ++k) {
    uint32_t q = fdiv(idx, fn);
    const uint32_t o = idx - q * fn.d;
    idx = q;
    q = fdiv(idx, fm);
    const uint32_t i = idx - q * fm.d;
    idx = q;
    row += i * rmul;
    col += o * cmul;
    rmul *= fm.d;
    cmul *= fn.d;
  }
}

// generic (64-bit index) variant for tensors with >= 2^32 padded elements
__device__ __forceinline__ void decode_interleaved64(int64_t idx, int mm, int nn, int order, int64_t& row, int64_t& col) {
  int64_t rmul = 1, cmul = 1;
  row = 0;
  col = 0;
  for (int k = 0; k < order; ++k) {
    const int o = static_cast<int>(idx % nn);
    idx /= nn;
    const int i = static_cast<int>(idx % mm);
    idx /= mm;
    row += i * rmul;
    col += o * cmul;
    rmul *= mm;
    cmul *= nn;
  }
}

template <typename T>
__global__ void tt_interleave_kernel(const T* __restrict__ src, int M, int N, FastDiv fm, FastDiv fn, int order,
                                     float* __restrict__ out, int64_t total) {
  const bool small = total < (int64_t(1) << 32);
  for (int64_t idx = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    int64_t row, col;
    if (small) decode_interleaved(static_cast<uint32_t>(idx), fm, fn, order, row, col);
    else decode_interleaved64(idx, fm.d, fn.d, order, row, col);
    out[idx] = (row < M && col < N) ? load_as_f32<T>(src, row * N + col) : 0.f;
  }
}

template <typename T>
__global__ void tt_deinterleave_kernel(const float* __restrict__ src, int M, int N, FastDiv fm, FastDiv fn, int order,
                                       T* __restrict__ out, int64_t total) {
  const bool small = total < (int64_t(1) << 32);
  for (int64_t idx = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    int64_t row, col;
    if (small) decode_interleaved(static_cast<uint32_t>(idx), fm, fn, order, row, col);
    else decode_interleaved64(idx, fm.d, fn.d, order, row, col);
    if (row < M && col < N) store_from_f32<T>(out, row * N + col, src[idx]);
  }
}

// ------------------------------------------------------------------------------------------------
// Order-2 TT of a matrix WITHOUT materialising the padded + interleaved unfolding (tt.py:48-67 builds it with pad,
// reshape and permute = three passes over M.N): element (ga, gb) of the P x P unfolding, ga = i1*nn + o1, gb = i2*nn + o2,
// is source element (i1*mm + i2, o1*nn + o2) (zero outside (M, N)), so the kernels below address the source directly.
//   tt_gather2   : X[P, ncols]  = first ncols columns of the unfolding     (input of the thin QR)
//   tt_project2  : R[r, P]      = Q[P, r]^T . unfolding                    (one pass over the source)
//   tt_reconstruct2 : dst[M, N] = (G1 . G2) de-interleaved and un-padded   (TensorTrain.to_matrix, tt.py:242-247)
// ------------------------------------------------------------------------------------------------
constexpr int kRkTile = 64;

template <typename T>
__global__ void tt_gather2_kernel(const T* __restrict__ src, int M, int N, int mm, int nn, float* __restrict__ X, int ncols) {
  const int P = mm * nn;
  const int64_t total = static_cast<int64_t>(P) * ncols;
  for (int64_t idx = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int ga = static_cast<int>(idx / ncols), gb = static_cast<int>(idx - static_cast<int64_t>(ga) * ncols);
    const int i1 = ga / nn, o1 = ga - i1 * nn, i2 = gb / nn, o2 = gb - i2 * nn;
    const int64_t row = static_cast<int64_t>(i1) * mm + i2, col = static_cast<int64_t>(o1) * nn + o2;
    X[idx] = (gb < P && row < M && col < N) ? load_as_f32<T>(src, row * N + col) : 0.f;
  }
}

// Same tiling as tt_project_kernel (64 x 128 tile, 4 x (4 + 4) outputs per thread, 16-byte shared-memory operands,
// register prefetch of the next K stage); only the fetch differs: the unfolding is read through the index map.
template <typename T>
__global__ void __launch_bounds__(kPjThreads)
tt_project2_kernel(const T* __restrict__ src, int M, int N, int mm, int nn, const float* __restrict__ Q,
                   float* __restrict__ R, int64_t split_stride, int r, int m_per_split) {
  __shared__ __align__(16) float sL[kPjTM][kPjTN];
  __shared__ __align__(16) float sQ[kPjTM][kPjRT];
  __shared__ int64_t s_colpart[kPjTN];
  float* Rs = R + blockIdx.y * split_stride;   // split s stores its own partial (split_stride 0: one split)
  __shared__ int s_coli2[kPjTN], s_colo2[kPjTN];
  const int P = mm * nn;
  const int n0 = blockIdx.x * kPjTN;
  const int m_begin = blockIdx.y * m_per_split;
  const int m_end = min(P, m_begin + m_per_split);
  const int tid = threadIdx.x;
  const int tr = tid / 16, tn = tid % 16;
  if (tid < kPjTN) {
    const int gb = n0 + tid;
    const int i2 = gb / nn, o2 = gb - i2 * nn;
    s_coli2[tid] = (gb < P) ? i2 : (1 << 28);
    s_colo2[tid] = o2;
    s_colpart[tid] = static_cast<int64_t>(i2) * N + o2;
  }
  __syncthreads();
  float pl[16];
  float pq[8];
  for (int r0 = 0; r0 < r; r0 += kPjRT) {
    float acc[4][8];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int c = 0; c < 8; ++c) acc[a][c] = 0.f;
    auto fetch = [&](int mm0) {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int idx = tid + u * kPjThreads;          // 0..1023: row i, column group c4
        const int i = idx >> 5, c4 = (idx & 31) * 4;
        const int ga = mm0 + i;
        const int i1 = ga / nn, o1 = ga - i1 * nn;
        const int64_t rowbase = static_cast<int64_t>(i1) * mm * N + static_cast<int64_t>(o1) * nn;
        const int rlim = (ga < m_end) ? M - i1 * mm : 0;
        const int clim = N - o1 * nn;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int c = c4 + e;
          const bool ok = s_coli2[c] < rlim && s_colo2[c] < clim;
          pl[u * 4 + e] = ok ? load_as_f32<T>(src, rowbase + s_colpart[c]) : 0.f;
        }
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int idx = tid + u * kPjThreads;          // 0..2047
        const int i = idx >> 6, k = idx & 63;
        const int gi = mm0 + i, gk = r0 + k;
        pq[u] = (gi < m_end && gk < r) ? Q[static_cast<int64_t>(gi) * r + gk] : 0.f;
      }
    };
    auto stash = [&]() {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int idx = tid + u * kPjThreads;
        *reinterpret_cast<float4*>(&sL[idx >> 5][(idx & 31) * 4]) = make_float4(pl[u * 4], pl[u * 4 + 1], pl[u * 4 + 2], pl[u * 4 + 3]);
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int idx = tid + u * kPjThreads;
        sQ[idx >> 6][idx & 63] = pq[u];
      }
    };
    if (m_begin < m_end) fetch(m_begin);
    for (int mm0 = m_begin; mm0 < m_end; mm0 += kPjTM) {
      stash();
      __syncthreads();
      if (mm0 + kPjTM < m_end) fetch(mm0 + kPjTM);
#pragma unroll 8
      for (int i = 0; i < kPjTM; ++i) {
        const float4 q = *reinterpret_cast<const float4*>(&sQ[i][tr * 4]);
        const float4 l0 = *reinterpret_cast<const float4*>(&sL[i][tn * 4]);
        const float4 l1 = *reinterpret_cast<const float4*>(&sL[i][64 + tn * 4]);
        const float qv[4] = {q.x, q.y, q.z, q.w};
        const float lv[8] = {l0.x, l0.y, l0.z, l0.w, l1.x, l1.y, l1.z, l1.w};
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int c = 0; c < 8; ++c) acc[a][c] = fmaf(qv[a], lv[c], acc[a][c]);
      }
      __syncthreads();
    }
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      const int gr = r0 + tr * 4 + a;
      if (gr >= r) continue;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const int gc = n0 + (c < 4 ? tn * 4 + c : 64 + tn * 4 + (c - 4));
        if (gc < P) Rs[static_cast<int64_t>(gr) * P + gc] = acc[a][c];
      }
    }
  }
}

// C = G1 [P, r] . G2 [r, P], written straight to dst[M, N] through the index map (only the (M, N) window is stored).
template <typename T>
__global__ void __launch_bounds__(256)
tt_reconstruct2_kernel(const float* __restrict__ G1, const float* __restrict__ G2, int r, T* __restrict__ dst, int M, int N,
                       int mm, int nn) {
  __shared__ float sA[kRkTile][kRkTile + 1];  // [row][k]
  __shared__ float sB[kRkTile][kRkTile];      // [k][col]
  const int P = mm * nn;
  const int m0 = blockIdx.y * kRkTile, n0 = blockIdx.x * kRkTile;
  const int tid = threadIdx.x, ty = tid / 16, tx = tid % 16;
  float acc[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[a][c] = 0.f;
  for (int k0 = 0; k0 < r; k0 += kRkTile) {
    for (int idx = tid; idx < kRkTile * kRkTile; idx += 256) {
      const int i = idx / kRkTile, k = idx % kRkTile;
      sA[i][k] = (m0 + i < P && k0 + k < r) ? G1[static_cast<int64_t>(m0 + i) * r + k0 + k] : 0.f;
      const int kk = idx / kRkTile, c = idx % kRkTile;
      sB[kk][c] = (k0 + kk < r && n0 + c < P) ? G2[static_cast<int64_t>(k0 + kk) * P + n0 + c] : 0.f;
    }
    __syncthreads();
    const int kn = min(kRkTile, r - k0);
    for (int k = 0; k < kn; ++k) {
      float av[4], bv[4];
#pragma unroll
      for (int a = 0; a < 4; ++a) av[a] = sA[ty * 4 + a][k];
#pragma unroll
      for (int c = 0; c < 4; ++c) bv[c] = sB[k][tx + 16 * c];
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[a][c] = fmaf(av[a], bv[c], acc[a][c]);
    }
    __syncthreads();
  }
  int ci2[4], co2[4];
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const int gb = n0 + tx + 16 * c;
    ci2[c] = gb / nn;
    co2[c] = gb - ci2[c] * nn;
    if (gb >= P) ci2[c] = 1 << 28;
  }
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    const int ga = m0 + ty * 4 + a;
    if (ga >= P) continue;
    const int i1 = ga / nn, o1 = ga - i1 * nn;
    const int rlim = M - i1 * mm, clim = N - o1 * nn;
    const int64_t rowbase = static_cast<int64_t>(i1) * mm * N + static_cast<int64_t>(o1) * nn;
#pragma unroll
    for (int c = 0; c < 4; ++c)
      if (ci2[c] < rlim && co2[c] < clim) store_from_f32<T>(dst, rowbase + static_cast<int64_t>(ci2[c]) * N + co2[c], acc[a][c]);
  }
}

// ------------------------------------------------------------------------------------------------
// small-K fp32 matmul  C[m, n] = A[m, r] . B[r, n]   (TT reconstruction chain, tt.py:213-237)
// 64 x 64 output tile per CTA, 4 x 4 per thread, whole K (= r <= 64 per pass) in smem.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
tt_matmul_rk_kernel(const float* __restrict__ A, const float* __restrict__ B, float* __restrict__ C, int m, int n, int r) {
  __shared__ float sA[kRkTile][kRkTile + 1];  // [row][k]
  __shared__ float sB[kRkTile][kRkTile];      // [k][col]
  const int m0 = blockIdx.y * kRkTile, n0 = blockIdx.x * kRkTile;
  const int tid = threadIdx.x, ty = tid / 16, tx = tid % 16;
  float acc[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[a][c] = 0.f;
  for (int k0 = 0; k0 < r; k0 += kRkTile) {
    for (int idx = tid; idx < kRkTile * kRkTile; idx += 256) {
      const int i = idx / kRkTile, k = idx % kRkTile;
      sA[i][k] = (m0 + i < m && k0 + k < r) ? A[static_cast<int64_t>(m0 + i) * r + k0 + k] : 0.f;
      const int kk = idx / kRkTile, c = idx % kRkTile;
      sB[kk][c] = (k0 + kk < r && n0 + c < n) ? B[static_cast<int64_t>(k0 + kk) * n + n0 + c] : 0.f;
    }
    __syncthreads();
    const int kn = min(kRkTile, r - k0);
    for (int k = 0; k < kn; ++k) {
      float av[4], bv[4];
#pragma unroll
      for (int a = 0; a < 4; ++a) av[a] = sA[ty * 4 + a][k];
#pragma unroll
      for (int c = 0; c < 4; ++c) bv[c] = sB[k][tx + 16 * c];
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[a][c] = fmaf(av[a], bv[c], acc[a][c]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    const int gi = m0 + ty * 4 + a;
    if (gi >= m) continue;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int gc = n0 + tx + 16 * c;
      if (gc < n) C[static_cast<int64_t>(gi) * n + gc] = acc[a][c];
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Order-2 reconstruction fused with the TT-Adam update (see include/sow_b200.h: tt_adam_fused2)
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
tt_adam_fused2_kernel(T* __restrict__ p, const T* __restrict__ g, const float* __restrict__ G1m,
                      const float* __restrict__ G2m, const float* __restrict__ G1v, const float* __restrict__ G2v,
                      int r, float* __restrict__ m_out, float* __restrict__ v_out, int M, int N, int mm, int nn,
                      float beta1, float omb1, float beta2, float omb2, float eps, float step_size, float lr_wd, int first_step) {
  extern __shared__ __align__(16) float fs[];
  const int P = mm * nn;  // interleaved matrix is P x P
  // smem, all k-major so that every operand of the inner product is one 16-byte load:
  //   s1m/s1v [r][64] = G1[a0 + i][k] transposed,  s2m/s2v [r][64] = G2[k][b0 + c]
  float* s1m = fs;
  float* s1v = s1m + r * 64;
  float* s2m = s1v + r * 64;
  float* s2v = s2m + r * 64;
  const int a0 = blockIdx.y * 64, b0 = blockIdx.x * 64;
  const int tid = threadIdx.x, ty = tid / 16, tx = tid % 16;   // thread owns rows ty*4..+3, columns tx*4..+3
  float am[4][4], av[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int c = 0; c < 4; ++c) am[a][c] = av[a][c] = 0.f;
  if (!first_step) {
    for (int idx = tid; idx < 64 * r; idx += 256) {
      const int i = idx / r, k = idx % r;
      const bool ok = a0 + i < P;
      s1m[k * 64 + i] = ok ? G1m[static_cast<int64_t>(a0 + i) * r + k] : 0.f;
      s1v[k * 64 + i] = ok ? G1v[static_cast<int64_t>(a0 + i) * r + k] : 0.f;
      const int kk = idx / 64, c = idx % 64;
      const bool ok2 = b0 + c < P;
      s2m[kk * 64 + c] = ok2 ? G2m[static_cast<int64_t>(kk) * P + b0 + c] : 0.f;
      s2v[kk * 64 + c] = ok2 ? G2v[static_cast<int64_t>(kk) * P + b0 + c] : 0.f;
    }
    __syncthreads();
#pragma unroll 4
    for (int k = 0; k < r; ++k) {
      const float4 a1m = *reinterpret_cast<const float4*>(s1m + k * 64 + ty * 4);
      const float4 a1v = *reinterpret_cast<const float4*>(s1v + k * 64 + ty * 4);
      const float4 b2m = *reinterpret_cast<const float4*>(s2m + k * 64 + tx * 4);
      const float4 b2v = *reinterpret_cast<const float4*>(s2v + k * 64 + tx * 4);
      const float x1m[4] = {a1m.x, a1m.y, a1m.z, a1m.w}, x1v[4] = {a1v.x, a1v.y, a1v.z, a1v.w};
      const float x2m[4] = {b2m.x, b2m.y, b2m.z, b2m.w}, x2v[4] = {b2v.x, b2v.y, b2v.z, b2v.w};
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          am[a][c] = fmaf(x1m[a], x2m[c], am[a][c]);
          av[a][c] = fmaf(x1v[a], x2v[c], av[a][c]);
        }
    }
  }
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    const int ga = a0 + ty * 4 + a;
    if (ga >= P) continue;
    const int i1 = ga / nn, o1 = ga % nn;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int gb = b0 + tx * 4 + c;
      if (gb >= P) continue;
      const int i2 = gb / nn, o2 = gb % nn;
      const int64_t row = static_cast<int64_t>(i1) * mm + i2, col = static_cast<int64_t>(o1) * nn + o2;
      float mo = 0.f, vo = 0.f;
      if (row < M && col < N) {
        const int64_t e = row * N + col;
        const float gv = load_as_f32<T>(g, e);
        float pv = load_as_f32<T>(p, e);
        const float mp = am[a][c];
        const float vp = fmaxf(av[a][c], 0.f);                     // ttadam.py:84
        mo = beta1 * mp + omb1 * gv;                      // ttadam.py:92
        vo = beta2 * vp + omb2 * gv * gv;                 // ttadam.py:93
        pv -= step_size * (mo / (sqrtf(vo) + eps));                // ttadam.py:94,103,108
        if (lr_wd > 0.f) pv -= lr_wd * pv;                         // ttadam.py:110-111
        store_from_f32<T>(p, e, pv);
      }
      m_out[static_cast<int64_t>(ga) * P + gb] = mo;
      v_out[static_cast<int64_t>(ga) * P + gb] = vo;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Order-2 TT-Adam with the re-compression fused in (no dense moment ever reaches HBM).
//
//   new moments  m' = b1 * (G1m . G2m) + (1-b1) g,   v' = b2 * max(G1v . G2v, 0) + (1-b2) g^2   (P x P, interleaved)
//   new cores    Q' = thin-QR(first r columns of m' / v'),   R' = Q'^T m' / Q'^T v'
//
// HEAD : the first 64 columns of m', v' (P x 64 each) -> X, the input of the thin QR.  p is NOT touched.
// FULL : CTA = (strip of 64 columns, range of 64-row tiles).  Per tile: reconstruct the old moments from the cores
//        (register-tiled rank-R product), Adam on p, stash m', v' in shared memory, accumulate R'[:, strip] +=
//        Q'[tile rows]^T . tile in registers; the accumulators are stored once per CTA as its row-range's partial (summed in range order afterwards).
// Traffic per step: g once + p read/write + cores (vs. + 16 B/element for dense fp32 moments written and re-read).
// R = rank padded to 8/16/32/64 (cores and bases are zero-padded in shared memory).
// ------------------------------------------------------------------------------------------------
template <typename T, int R, bool HEAD>
__global__ void __launch_bounds__(256, (R <= 16 ? 4 : (R <= 32 ? 3 : 2)))
tt_adam2_kernel(T* __restrict__ p, const T* __restrict__ g, const float* __restrict__ G1m, const float* __restrict__ G2m,
                const float* __restrict__ G1v, const float* __restrict__ G2v, int r, const float* __restrict__ Qm,
                const float* __restrict__ Qv, float* __restrict__ Rm, float* __restrict__ Rv, float* __restrict__ Xm,
                float* __restrict__ Xv, int M, int N, int mm, int nn, float beta1, float omb1, float beta2, float omb2,
                float eps, float step_size, float lr_wd, int first_step, int tiles_per_cta, int64_t split_stride) {
  extern __shared__ __align__(16) float fs[];
  const int P = mm * nn;
  float* s2m = fs;                 // [R][64]  G2m[k][b0 + c]
  pdl_trigger();
  pdl_wait();
  float* s2v = s2m + R * 64;
  float* s1m = s2v + R * 64;       // [64][R]  G1m[a0 + i][k]
  float* s1v = s1m + R * 64;
  float* sQm = s1v + R * 64;       // [64][R]  Q'm[a0 + i][k]
  float* sQv = sQm + 64 * R;
  // [64][64] m' / v' tiles; at R = 64 they alias s1m / s1v (dead once the tile is reconstructed): 96 KB -> 2 CTAs per SM
  constexpr bool kAlias = (R == 64);
  float* sMt = kAlias ? s1m : sQv + 64 * R;
  float* sVt = sMt + 64 * 64;
  const int tid = threadIdx.x, ty = tid / 16, tx = tid % 16;   // phase 1: rows ty*4..+3, columns tx*4..+3
  const int b0 = HEAD ? 0 : blockIdx.x * 64;
  const int n_tiles = (P + 63) / 64;
  const int t_begin = HEAD ? blockIdx.x : blockIdx.y * tiles_per_cta;
  const int t_end = HEAD ? blockIdx.x + 1 : min(n_tiles, t_begin + tiles_per_cta);
  // phase 2 mapping: column pcol of the strip, quarter kpart of the padded rank
  const int pcol = tid & 63, kpart = tid >> 6;
  constexpr int KQ = R / 4;
  float accm[KQ], accv[KQ];
#pragma unroll
  for (int k = 0; k < KQ; ++k) accm[k] = accv[k] = 0.f;
  // element (ga, gb) of the interleaved matrix is (row, col) = (i1*mm + i2, o1*nn + o2) with ga = i1*nn + o1 and
  // gb = i2*nn + o2: the column part depends on the strip only, so it is decoded once per CTA
  int ci2[4], co2[4];
  int64_t colbase[4];
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const int gb = b0 + tx * 4 + c;
    ci2[c] = gb / nn;
    co2[c] = gb - ci2[c] * nn;
    colbase[c] = static_cast<int64_t>(ci2[c]) * N + co2[c];
    if (gb >= P) ci2[c] = 1 << 28;   // fails the row bound below
  }
  const bool cols_contig = (ci2[0] == ci2[3]);

  if (!first_step) {
    for (int idx = tid; idx < R * 64; idx += 256) {
      const int kk = idx / 64, c = idx % 64;
      const bool ok = kk < r && b0 + c < P;
      s2m[idx] = ok ? G2m[static_cast<int64_t>(kk) * P + b0 + c] : 0.f;
      s2v[idx] = ok ? G2v[static_cast<int64_t>(kk) * P + b0 + c] : 0.f;
    }
  }
  for (int t = t_begin; t < t_end; ++t) {
    const int a0 = t * 64;
    __syncthreads();   // previous tile's phase 2 is done with sQ / sMt; first iteration: s2 staged
    // staging: constant trip counts, so all global loads of a tile are in flight before the first shared store
    constexpr int kStage = 64 * R / 256;
    if (!first_step) {
      float t1m[kStage], t1v[kStage];
#pragma unroll
      for (int u = 0; u < kStage; ++u) {
        const int idx = tid + u * 256;
        const int i = idx / R, k = idx % R;
        const bool ok = a0 + i < P && k < r;
        t1m[u] = ok ? G1m[static_cast<int64_t>(a0 + i) * r + k] : 0.f;
        t1v[u] = ok ? G1v[static_cast<int64_t>(a0 + i) * r + k] : 0.f;
      }
#pragma unroll
      for (int u = 0; u < kStage; ++u) {
        s1m[tid + u * 256] = t1m[u];      // row-major [64][R], like G1 itself
        s1v[tid + u * 256] = t1v[u];
      }
    }
    if (!HEAD) {
      float tqm[kStage], tqv[kStage];
#pragma unroll
      for (int u = 0; u < kStage; ++u) {
        const int idx = tid + u * 256;
        const int i = idx / R, k = idx % R;
        const bool ok = a0 + i < P && k < r;
        tqm[u] = ok ? Qm[static_cast<int64_t>(a0 + i) * r + k] : 0.f;
        tqv[u] = ok ? Qv[static_cast<int64_t>(a0 + i) * r + k] : 0.f;
      }
#pragma unroll
      for (int u = 0; u < kStage; ++u) {
        sQm[tid + u * 256] = tqm[u];
        sQv[tid + u * 256] = tqv[u];
      }
    }
    __syncthreads();
    float am[4][4], av[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int c = 0; c < 4; ++c) am[a][c] = av[a][c] = 0.f;
    if (!first_step) {
#pragma unroll 2
      for (int k0 = 0; k0 < R; k0 += 4) {
        float x1m[4][4], x1v[4][4], x2m[4][4], x2v[4][4];   // [row a | k j][k j | col c]
#pragma unroll
        for (int a = 0; a < 4; ++a) {
          const float4 tm = *reinterpret_cast<const float4*>(s1m + (ty * 4 + a) * R + k0);
          const float4 tv = *reinterpret_cast<const float4*>(s1v + (ty * 4 + a) * R + k0);
          x1m[a][0] = tm.x, x1m[a][1] = tm.y, x1m[a][2] = tm.z, x1m[a][3] = tm.w;
          x1v[a][0] = tv.x, x1v[a][1] = tv.y, x1v[a][2] = tv.z, x1v[a][3] = tv.w;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 tm = *reinterpret_cast<const float4*>(s2m + (k0 + j) * 64 + tx * 4);
          const float4 tv = *reinterpret_cast<const float4*>(s2v + (k0 + j) * 64 + tx * 4);
          x2m[j][0] = tm.x, x2m[j][1] = tm.y, x2m[j][2] = tm.z, x2m[j][3] = tm.w;
          x2v[j][0] = tv.x, x2v[j][1] = tv.y, x2v[j][2] = tv.z, x2v[j][3] = tv.w;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
          for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              am[a][c] = fmaf(x1m[a][j], x2m[j][c], am[a][c]);
              av[a][c] = fmaf(x1v[a][j], x2v[j][c], av[a][c]);
            }
      }
    }
    if (kAlias && !HEAD) __syncthreads();   // every thread is done reading s1m / s1v before the tile overwrites them
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      const int ga = a0 + ty * 4 + a;
      const int i1 = ga / nn, o1 = ga - i1 * nn;
      const int64_t rowbase = static_cast<int64_t>(i1) * mm * N + static_cast<int64_t>(o1) * nn;
      const int rlim = (ga < P) ? M - i1 * mm : 0;     // valid iff i2 < rlim
      const int clim = N - o1 * nn;                    // valid iff o2 < clim
      float mo4[4] = {0.f, 0.f, 0.f, 0.f}, vo4[4] = {0.f, 0.f, 0.f, 0.f};
      bool ok[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) ok[c] = ci2[c] < rlim && co2[c] < clim;
      const int64_t e0 = rowbase + colbase[0];
      float gv[4] = {0.f, 0.f, 0.f, 0.f}, pv[4] = {0.f, 0.f, 0.f, 0.f};
      const bool vec = cols_contig && ok[0] && ok[3] && ((e0 & 3) == 0);
      if (vec) {
        load4_as_f32<T>(g, e0, gv);
        if (!HEAD) load4_as_f32<T>(p, e0, pv);
      } else {
#pragma unroll
        for (int c = 0; c < 4; ++c)
          if (ok[c]) {
            gv[c] = load_as_f32<T>(g, rowbase + colbase[c]);
            if (!HEAD) pv[c] = load_as_f32<T>(p, rowbase + colbase[c]);
          }
      }
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        if (ok[c]) {
          const float mp = am[a][c];
          const float vp = fmaxf(av[a][c], 0.f);                       // ttadam.py:84
          const float mo = beta1 * mp + omb1 * gv[c];                  // ttadam.py:92
          const float vo = beta2 * vp + omb2 * gv[c] * gv[c];          // ttadam.py:93
          if (!HEAD) {
            pv[c] -= step_size * (mo / (sqrtf(vo) + eps));             // ttadam.py:94,103,108
            if (lr_wd > 0.f) pv[c] -= lr_wd * pv[c];                   // ttadam.py:110-111
          }
          mo4[c] = mo;
          vo4[c] = vo;
        }
      }
      if (!HEAD) {
        if (vec) {
          store4_from_f32<T>(p, e0, pv);
        } else {
#pragma unroll
          for (int c = 0; c < 4; ++c)
            if (ok[c]) store_from_f32<T>(p, rowbase + colbase[c], pv[c]);
        }
      }
      if (HEAD) {
        if (ga < P) {
          *reinterpret_cast<float4*>(Xm + static_cast<int64_t>(ga) * 64 + tx * 4) = make_float4(mo4[0], mo4[1], mo4[2], mo4[3]);
          *reinterpret_cast<float4*>(Xv + static_cast<int64_t>(ga) * 64 + tx * 4) = make_float4(vo4[0], vo4[1], vo4[2], vo4[3]);
        }
      } else {
        *reinterpret_cast<float4*>(sMt + (ty * 4 + a) * 64 + tx * 4) = make_float4(mo4[0], mo4[1], mo4[2], mo4[3]);
        *reinterpret_cast<float4*>(sVt + (ty * 4 + a) * 64 + tx * 4) = make_float4(vo4[0], vo4[1], vo4[2], vo4[3]);
      }
    }
    if (!HEAD) {
      __syncthreads();
      // phase 2: R'[k, b0 + pcol] += sum_i Q'[a0 + i, k] * tile[i, pcol]
#pragma unroll 8
      for (int i = 0; i < 64; ++i) {
        const float mv = sMt[i * 64 + pcol], vv = sVt[i * 64 + pcol];
        float qm[KQ], qv[KQ];
        if constexpr (KQ >= 4) {
#pragma unroll
          for (int k4 = 0; k4 < KQ / 4; ++k4) {
            const float4 a4 = *reinterpret_cast<const float4*>(sQm + i * R + kpart * KQ + 4 * k4);
            const float4 b4 = *reinterpret_cast<const float4*>(sQv + i * R + kpart * KQ + 4 * k4);
            qm[4 * k4] = a4.x, qm[4 * k4 + 1] = a4.y, qm[4 * k4 + 2] = a4.z, qm[4 * k4 + 3] = a4.w;
            qv[4 * k4] = b4.x, qv[4 * k4 + 1] = b4.y, qv[4 * k4 + 2] = b4.z, qv[4 * k4 + 3] = b4.w;
          }
        } else {
          const float2 a2 = *reinterpret_cast<const float2*>(sQm + i * R + kpart * KQ);
          const float2 b2 = *reinterpret_cast<const float2*>(sQv + i * R + kpart * KQ);
          qm[0] = a2.x, qm[1] = a2.y, qv[0] = b2.x, qv[1] = b2.y;
        }
#pragma unroll
        for (int k = 0; k < KQ; ++k) {
          accm[k] = fmaf(qm[k], mv, accm[k]);
          accv[k] = fmaf(qv[k], vv, accv[k]);
        }
      }
    }
  }
  if (!HEAD && b0 + pcol < P) {
#pragma unroll
    for (int k = 0; k < KQ; ++k) {
      const int gk = kpart * KQ + k;
      if (gk < r) {
        // row-range split blockIdx.y stores its own partial (split_stride 0: one split, Rm / Rv are the results)
        Rm[blockIdx.y * split_stride + static_cast<int64_t>(gk) * P + b0 + pcol] = accm[k];
        Rv[blockIdx.y * split_stride + static_cast<int64_t>(gk) * P + b0 + pcol] = accv[k];
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// FULL step for ranks <= 16 with the projection accumulated in REGISTERS (tt_adam2_reg_kernel).
//
// The kernel above stashes every m' / v' tile in shared memory and re-reads it column by column for the projection
// (256 shared loads per 256 FMAs per thread and tile: the shared-memory pipe bounds it, ~4500 cycles per 64 x 64 tile).
// Here a thread keeps its (RTH rows x CT columns) micro-tile of m', v' in registers after the Adam update and multiplies
// it straight into its own accumulators acc[k][c] += Q'[row, k] . m'[row, c] for ALL k, over every tile of the CTA's
// row range; the TY threads that share a column group are summed once, through shared memory, when the range is done
// (fixed order).  Shared loads per tile: the G1 / Q' rows (warp-broadcast LDS.128) and the G2 strip (CT-wide) only.
//   R =  8: CT = 4 (TY = 16, RTH = 2) ; R = 16: CT = 2 (TY = 8, RTH = 4)   [R = 32, CT = 1 measured 260 us at 4096^2
//   against 185 us for the tensor-core kernel: not instantiated]
//   -> 2 . R . CT = 64 accumulators per thread in every configuration; tile = 32 rows x 64 columns.
// G1 / Q' tiles are staged by cp.async, three buffers deep (one barrier per tile); g and p of the tile are requested
// before the barrier and consumed after the reconstruction FMAs.
// Measured and dropped: serving rows whose offset is not a multiple of four elements (4096 x 11008: nn = 105, three rows in
// four) with two aligned halves or element / pair / element instead of four element accesses -- 0.38 -> 0.51 ms per step at
// r = 8 (a third raw register per row and a three-way unpack / store per row cost more than the saved accesses).
// ------------------------------------------------------------------------------------------------
template <typename T, int CT>
struct RawVec;
template <>
struct RawVec<__nv_bfloat16, 4> { using type = uint2; };
template <>
struct RawVec<__nv_bfloat16, 2> { using type = uint32_t; };
template <>
struct RawVec<__nv_bfloat16, 1> { using type = unsigned short; };
template <>
struct RawVec<float, 4> { using type = float4; };
template <>
struct RawVec<float, 2> { using type = float2; };
template <>
struct RawVec<float, 1> { using type = float; };

template <typename T, int CT>
__device__ __forceinline__ void raw_unpack(const typename RawVec<T, CT>::type& raw, float (&v)[CT]) {
  T tmp[CT];
  memcpy(tmp, &raw, sizeof(tmp));
#pragma unroll
  for (int c = 0; c < CT; ++c) v[c] = load_as_f32<T>(tmp, c);
}
template <typename T, int CT>
__device__ __forceinline__ typename RawVec<T, CT>::type raw_pack(const float (&v)[CT]) {
  T tmp[CT];
#pragma unroll
  for (int c = 0; c < CT; ++c) store_from_f32<T>(tmp, c, v[c]);
  typename RawVec<T, CT>::type raw;
  memcpy(&raw, tmp, sizeof(tmp));
  return raw;
}

__device__ __forceinline__ void cp_async16(float* smem_dst, const float* src, bool valid) {
  const uint32_t dst = static_cast<uint32_t>(__cvta_generic_to_shared(smem_dst));
  const int bytes = valid ? 16 : 0;   // src-size 0: the 16 bytes are zero-filled, the source is not read
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

template <int CT>
__device__ __forceinline__ void lds_ct(const float* s, float (&v)[CT]) {
  if constexpr (CT == 4) {
    const float4 t = *reinterpret_cast<const float4*>(s);
    v[0] = t.x, v[1] = t.y, v[2] = t.z, v[3] = t.w;
  } else if constexpr (CT == 2) {
    const float2 t = *reinterpret_cast<const float2*>(s);
    v[0] = t.x, v[1] = t.y;
  } else {
    v[0] = s[0];
  }
}
template <int CT>
__device__ __forceinline__ void sts_ct(float* s, const float (&v)[CT]) {
  if constexpr (CT == 4) *reinterpret_cast<float4*>(s) = make_float4(v[0], v[1], v[2], v[3]);
  else if constexpr (CT == 2) *reinterpret_cast<float2*>(s) = make_float2(v[0], v[1]);
  else s[0] = v[0];
}

constexpr int kRegTileRows = 32;
constexpr size_t reg_kernel_smem(int R) { return std::max<size_t>(size_t(2048) * R, 32768); }
// projection-only instance: three Q' stage buffers; the final reduction scratch is TY * R * 64 floats = 1024 * CT * R bytes
constexpr size_t reg_proj_smem(int R, int CT) { return std::max<size_t>(size_t(384) * R, size_t(1024) * CT * R); }
// row-range splits of the register-accumulating kernels: two resident CTAs per SM, two waves
static int reg_kernel_splits(int P, int* per) {
  const int n_strips = ceil_div(P, 64), n_rt = ceil_div(P, kRegTileRows);
  int splits = std::max(1, (2 * 2 * num_sms()) / n_strips);
  splits = std::min(splits, n_rt);
  *per = ceil_div(n_rt, splits);
  return ceil_div(n_rt, *per);
}

// PROJ: projection only -- R'[r, P] = Q'^T . unfolding(g) (tt_project2: no cores, no Adam, p untouched, one moment).
template <typename T, int R, int CT, bool PROJ = false>
__global__ void __launch_bounds__(256, 2)
tt_adam2_reg_kernel(T* __restrict__ p, const T* __restrict__ g, const float* __restrict__ G1m, const float* __restrict__ G2m,
                    const float* __restrict__ G1v, const float* __restrict__ G2v, int r, const float* __restrict__ Qm,
                    const float* __restrict__ Qv, float* __restrict__ Rm, float* __restrict__ Rv, int M, int N, int mm, int nn,
                    float beta1, float omb1, float beta2, float omb2, float eps, float step_size, float lr_wd, int first_step,
                    int tiles_per_cta, int64_t split_stride) {
  pdl_trigger();
  pdl_wait();
  constexpr int TX = 64 / CT, TY = 256 / TX, RTH = kRegTileRows / TY;
  constexpr int KS = (CT == 4) ? 2 : 4;       // k-step of the reconstruction: 2 . KS . CT operand registers
  static_assert((PROJ ? 1 : 2) * R * CT <= 64, "accumulator registers");
  constexpr int kArr = kRegTileRows * R;        // floats of one staged array (32 rows x R)
  constexpr int kNArr = PROJ ? 1 : 4;           // G1m | G1v | Q'm | Q'v   (PROJ: Q' only)
  constexpr int kQm = PROJ ? 0 : 2, kQv = 3;
  constexpr int kBuf = kNArr * kArr;
  using Raw = typename RawVec<T, CT>::type;
  extern __shared__ __align__(16) float fs[];
  float* s2m = fs;                 // [R][64]  G2m[k][b0 + c]   (absent in PROJ)
  float* s2v = s2m + (PROJ ? 0 : R * 64);
  float* stage = s2v + (PROJ ? 0 : R * 64);     // [3][kNArr][32][R]
  const int P = mm * nn;
  const int tid = threadIdx.x, ty = tid / TX, tx = tid % TX;
  const int b0 = blockIdx.x * 64;
  const int n_tiles = (P + kRegTileRows - 1) / kRegTileRows;
  const int t_begin = blockIdx.y * tiles_per_cta;
  const int t_end = min(n_tiles, t_begin + tiles_per_cta);

  constexpr int RV = PROJ ? 1 : R;
  float accm[R][CT], accv[RV][CT];
#pragma unroll
  for (int k = 0; k < R; ++k)
#pragma unroll
    for (int c = 0; c < CT; ++c) accm[k][c] = 0.f;
#pragma unroll
  for (int k = 0; k < RV; ++k)
#pragma unroll
    for (int c = 0; c < CT; ++c) accv[k][c] = 0.f;

  // column part of the index map (strip-constant): gb = i2 * nn + o2 -> source (row offset i2, column offset o2).
  // A thread's CT columns cross at most one i2 boundary (nn >= CT is required by the launcher): columns c >= cut sit
  // in the next i2 block, i.e. one source row further down and nn columns to the left.
  const int gb0 = b0 + tx * CT;
  const int ci2 = gb0 / nn, co2 = gb0 - ci2 * nn;
  const int cut = nn - co2;                                    // >= CT: no boundary inside the thread's columns
  const int ncols = min(CT, P - gb0);                          // columns c < ncols exist in the unfolding (<= 0: none)
  const bool vec_base = cut >= CT && ncols >= CT &&
                        ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g)) % sizeof(Raw)) == 0;

  // rows (a0 + i) of the four [P x r] arrays -> stage buffer; cp.async when the rows are whole 16-byte chunks
  const bool fast = (r == R) && (((reinterpret_cast<uintptr_t>(Qm) | reinterpret_cast<uintptr_t>(Qv) |
                                   reinterpret_cast<uintptr_t>(G1m) | reinterpret_cast<uintptr_t>(G1v)) & 15) == 0);
  auto stage_tile = [&](int t, float* buf) {
    const int a0 = t * kRegTileRows;
    constexpr int kChunks = kBuf / 4;            // 16-byte chunks of one buffer
    if (fast) {
#pragma unroll
      for (int q = tid; q < kChunks; q += 256) {
        const int arr = q / (kArr / 4), w = q - arr * (kArr / 4);
        const int i = w / (R / 4), k4 = w - i * (R / 4);
        if (!PROJ && first_step && arr < 2) continue;
        const float* base = PROJ ? Qm : (arr == 0 ? G1m : (arr == 1 ? G1v : (arr == 2 ? Qm : Qv)));
        const bool ok = a0 + i < P;
        cp_async16(buf + arr * kArr + i * R + k4 * 4, ok ? base + static_cast<int64_t>(a0 + i) * r + k4 * 4 : base, ok);
      }
    } else {
      for (int q = tid; q < kBuf; q += 256) {
        const int arr = q / kArr, w = q - arr * kArr;
        const int i = w / R, k = w - i * R;
        if (!PROJ && first_step && arr < 2) continue;
        const float* base = PROJ ? Qm : (arr == 0 ? G1m : (arr == 1 ? G1v : (arr == 2 ? Qm : Qv)));
        buf[q] = (a0 + i < P && k < r) ? base[static_cast<int64_t>(a0 + i) * r + k] : 0.f;
      }
    }
  };

  if (t_begin < t_end) stage_tile(t_begin, stage);
  cp_async_commit();
  if (!PROJ && !first_step) {
    for (int idx = tid; idx < R * 64; idx += 256) {
      const int kk = idx / 64, c = idx % 64;
      const bool ok = kk < r && b0 + c < P;
      s2m[idx] = ok ? G2m[static_cast<int64_t>(kk) * P + b0 + c] : 0.f;
      s2v[idx] = ok ? G2v[static_cast<int64_t>(kk) * P + b0 + c] : 0.f;
    }
  }

  for (int t = t_begin; t < t_end; ++t) {
    const int a0 = t * kRegTileRows;
    float* buf = stage + ((t - t_begin) % 3) * kBuf;
    if (t + 1 < t_end) stage_tile(t + 1, stage + ((t + 1 - t_begin) % 3) * kBuf);
    cp_async_commit();

    // ---- g, p of this thread's RTH x CT elements: requested now, consumed after the reconstruction ----
    // row ga = i1 * nn + o1 -> source row i1 * mm + i2, column o1 * nn + o2 (zero outside (M, N))
    const int ga_first = a0 + ty * RTH;
    int i1 = ga_first / nn, o1 = ga_first - i1 * nn;
    // 32-bit element offsets (the launcher guarantees (M + 1) * N < 2^31).  vecbits: row a is one aligned vector inside
    // (M, N); okbits: element (a, c) of a non-vector row is inside (M, N).  Column c >= cut sits in the next i2 block:
    // one source row down, nn columns to the left (+ hop elements).
    int eoff[RTH];
    uint32_t vecbits = 0, okbits = 0;
    Raw graw[RTH], praw[RTH];
    const int hop = N - nn;
#pragma unroll
    for (int a = 0; a < RTH; ++a) {
      const bool row_ok = ga_first + a < P;
      const int row = i1 * mm + ci2, col = o1 * nn + co2;
      eoff[a] = row * N + col;
      if (vec_base && row_ok && row < M && col + CT <= N && (eoff[a] % CT) == 0) {
        vecbits |= 1u << a;
        graw[a] = *reinterpret_cast<const Raw*>(g + eoff[a]);
        if constexpr (!PROJ) praw[a] = *reinterpret_cast<const Raw*>(p + eoff[a]);
      } else {
        // unaligned / boundary rows: element loads, packed like the vector (zeros outside)
        T tg[CT], tp[CT];
#pragma unroll
        for (int c = 0; c < CT; ++c) {
          const int over = c >= cut ? 1 : 0;
          const bool ok = row_ok && c < ncols && row + over < M && col + c - over * nn < N;
          const int e = eoff[a] + c + over * hop;
          okbits |= (ok ? 1u : 0u) << (a * CT + c);
          tg[c] = ok ? g[e] : T(0.f);
          if constexpr (!PROJ) tp[c] = ok ? p[e] : T(0.f);
        }
        memcpy(&graw[a], tg, sizeof(Raw));
        if constexpr (!PROJ) memcpy(&praw[a], tp, sizeof(Raw));
      }
      if (++o1 == nn) o1 = 0, ++i1;
    }

    cp_async_wait<1>();     // this tile's stage group has landed (the next tile's may still be in flight)
    __syncthreads();

    // ---- reconstruct the old moments of the micro-tile ----
    float am[RTH][CT], av[RTH][CT];
#pragma unroll
    for (int a = 0; a < RTH; ++a)
#pragma unroll
      for (int c = 0; c < CT; ++c) am[a][c] = av[a][c] = 0.f;
    if (!PROJ && !first_step) {
      const float* s1m = buf + (ty * RTH) * R;
      const float* s1v = buf + kArr + (ty * RTH) * R;
#pragma unroll
      for (int k0 = 0; k0 < R; k0 += KS) {
        float x2m[KS][CT], x2v[KS][CT];
#pragma unroll
        for (int j = 0; j < KS; ++j) {
          lds_ct<CT>(s2m + (k0 + j) * 64 + tx * CT, x2m[j]);
          lds_ct<CT>(s2v + (k0 + j) * 64 + tx * CT, x2v[j]);
        }
#pragma unroll
        for (int a = 0; a < RTH; ++a) {
          float x1m[KS], x1v[KS];
          lds_ct<KS>(s1m + a * R + k0, x1m);
          lds_ct<KS>(s1v + a * R + k0, x1v);
#pragma unroll
          for (int j = 0; j < KS; ++j)
#pragma unroll
            for (int c = 0; c < CT; ++c) {
              am[a][c] = fmaf(x1m[j], x2m[j][c], am[a][c]);
              av[a][c] = fmaf(x1v[j], x2v[j][c], av[a][c]);
            }
        }
      }
    }

    // ---- Adam on p; am / av become the new moments m' / v' (zero outside (M, N)) ----
    // sqrt.approx / rcp.approx (MUFU, <= 2 ulp each) instead of the IEEE sequences: the update term is scaled by the
    // step size before it meets p, far inside the 2e-5 trajectory bound (tests/test_tt_gpu.py)
    auto adam1 = [&](float& m_io, float& v_io, float gval, float& pval) {
      const float mo = fmaf(beta1, m_io, omb1 * gval);                         // ttadam.py:92
      const float vo = fmaf(beta2, fmaxf(v_io, 0.f), omb2 * gval * gval);      // ttadam.py:84,93
      float sq, rc;
      asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(sq) : "f"(vo));
      asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rc) : "f"(sq + eps));
      pval = fmaf(-step_size, mo * rc, pval);                                  // ttadam.py:94,103,108
      pval = fmaf(-lr_wd, pval, pval);                                         // ttadam.py:110-111 (lr_wd = 0: no-op)
      m_io = mo, v_io = vo;
    };
    if constexpr (PROJ) {
      // the "moment" is the source element itself (zeros outside (M, N) came with the loads)
#pragma unroll
      for (int a = 0; a < RTH; ++a) raw_unpack<T, CT>(graw[a], am[a]);
    } else if (vecbits == (1u << RTH) - 1u) {        // the common case: every row of the micro-tile is one aligned vector
#pragma unroll
      for (int a = 0; a < RTH; ++a) {
        float gv[CT], pv[CT];
        raw_unpack<T, CT>(graw[a], gv);
        raw_unpack<T, CT>(praw[a], pv);
#pragma unroll
        for (int c = 0; c < CT; ++c) adam1(am[a][c], av[a][c], gv[c], pv[c]);
        *reinterpret_cast<Raw*>(p + eoff[a]) = raw_pack<T, CT>(pv);
      }
    } else {
#pragma unroll
      for (int a = 0; a < RTH; ++a) {
        float gv[CT], pv[CT];
        raw_unpack<T, CT>(graw[a], gv);
        raw_unpack<T, CT>(praw[a], pv);
#pragma unroll
        for (int c = 0; c < CT; ++c) adam1(am[a][c], av[a][c], gv[c], pv[c]);
        if ((vecbits >> a) & 1u) {
          *reinterpret_cast<Raw*>(p + eoff[a]) = raw_pack<T, CT>(pv);
        } else {
#pragma unroll
          for (int c = 0; c < CT; ++c) {
            if ((okbits >> (a * CT + c)) & 1u) store_from_f32<T>(p, eoff[a] + c + (c >= cut ? hop : 0), pv[c]);
            else am[a][c] = av[a][c] = 0.f;
          }
        }
      }
    }

    // ---- projection: acc[k][c] += Q'[row a, k] . m'[a][c] ----
    {
      const float* sQm = buf + kQm * kArr + (ty * RTH) * R;
      const float* sQv = buf + (PROJ ? 0 : kQv) * kArr + (ty * RTH) * R;
#pragma unroll
      for (int a = 0; a < RTH; ++a)
#pragma unroll
        for (int k4 = 0; k4 < R / 4; ++k4) {
          const float4 qm = *reinterpret_cast<const float4*>(sQm + a * R + 4 * k4);
          const float qms[4] = {qm.x, qm.y, qm.z, qm.w};
#pragma unroll
          for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int c = 0; c < CT; ++c) accm[4 * k4 + j][c] = fmaf(qms[j], am[a][c], accm[4 * k4 + j][c]);
          if constexpr (!PROJ) {
            const float4 qv = *reinterpret_cast<const float4*>(sQv + a * R + 4 * k4);
            const float qvs[4] = {qv.x, qv.y, qv.z, qv.w};
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
              for (int c = 0; c < CT; ++c) accv[4 * k4 + j][c] = fmaf(qvs[j], av[a][c], accv[4 * k4 + j][c]);
          }
        }
    }
  }

  // ---- sum the TY row groups of every column (fixed order) and store this row range's partial of R' ----
  cp_async_wait<0>();
  float* red = fs;                  // [TY][R][64] floats (32 KB; PROJ: up to 64 KB), over the (dead) staging area
#pragma unroll
  for (int pass = 0; pass < (PROJ ? 1 : 2); ++pass) {
    __syncthreads();
#pragma unroll
    for (int k = 0; k < R; ++k) {
      if (pass == 0) sts_ct<CT>(red + (ty * R + k) * 64 + tx * CT, accm[k]);
      else if constexpr (!PROJ) sts_ct<CT>(red + (ty * R + k) * 64 + tx * CT, accv[k]);
    }
    __syncthreads();
    float* dst = (pass == 0 ? Rm : Rv) + blockIdx.y * split_stride;
#pragma unroll
    for (int u = 0; u < R * 64 / 256; ++u) {
      const int o = tid + u * 256;
      const int k = o / 64, col = o % 64;
      float s = 0.f;
#pragma unroll
      for (int y = 0; y < TY; ++y) s += red[(y * R + k) * 64 + col];
      if (k < r && b0 + col < P) dst[static_cast<int64_t>(k) * P + b0 + col] = s;
    }
  }
}

// Reconstruction only, same structure: dst[M, N] = (G1 [P, r] . G2 [r, P]) read back through the index map.  A thread owns
// 4 rows x 4 columns of a 64 x 64 tile (2 R shared loads per 16 R FMAs, against 8 per 16 in tt_reconstruct2_kernel), the G2
// strip stays in shared memory for the CTA's whole row range, G1 tiles arrive by cp.async three buffers deep, and the
// (M, N) window is written with one vector store per row wherever the index map allows it.
template <typename T, int R>
__global__ void __launch_bounds__(256, 3)
tt_reconstruct2_reg_kernel(const float* __restrict__ G1, const float* __restrict__ G2, int r, T* __restrict__ dst, int M, int N,
                           int mm, int nn, int tiles_per_cta) {
  pdl_trigger();
  pdl_wait();
  constexpr int CT = 4, TX = 16, RTH = 4, ROWS = 64;
  constexpr int kArr = ROWS * R;
  using Raw = typename RawVec<T, CT>::type;
  extern __shared__ __align__(16) float fs[];
  float* s2 = fs;                  // [R][64]  G2[k][b0 + c]
  float* stage = s2 + R * 64;      // [3][64][R]
  const int P = mm * nn;
  const int tid = threadIdx.x, ty = tid / TX, tx = tid % TX;
  const int b0 = blockIdx.x * 64;
  const int n_tiles = (P + ROWS - 1) / ROWS;
  const int t_begin = blockIdx.y * tiles_per_cta;
  const int t_end = min(n_tiles, t_begin + tiles_per_cta);
  const int gb0 = b0 + tx * CT;
  const int ci2 = gb0 / nn, co2 = gb0 - ci2 * nn;
  const int cut = nn - co2;
  const int ncols = min(CT, P - gb0);
  const bool vec_base = cut >= CT && ncols >= CT && (reinterpret_cast<uintptr_t>(dst) % sizeof(Raw)) == 0;
  const int hop = N - nn;
  const bool fast = (r == R) && ((reinterpret_cast<uintptr_t>(G1) & 15) == 0);
  auto stage_tile = [&](int t, float* buf) {
    const int a0 = t * ROWS;
    if (fast) {
      for (int q = tid; q < kArr / 4; q += 256) {
        const int i = q / (R / 4), k4 = q - i * (R / 4);
        const bool ok = a0 + i < P;
        cp_async16(buf + i * R + k4 * 4, ok ? G1 + static_cast<int64_t>(a0 + i) * r + k4 * 4 : G1, ok);
      }
    } else {
      for (int q = tid; q < kArr; q += 256) {
        const int i = q / R, k = q - i * R;
        buf[q] = (a0 + i < P && k < r) ? G1[static_cast<int64_t>(a0 + i) * r + k] : 0.f;
      }
    }
  };
  if (t_begin < t_end) stage_tile(t_begin, stage);
  cp_async_commit();
  for (int idx = tid; idx < R * 64; idx += 256) {
    const int kk = idx / 64, c = idx % 64;
    s2[idx] = (kk < r && b0 + c < P) ? G2[static_cast<int64_t>(kk) * P + b0 + c] : 0.f;
  }
  for (int t = t_begin; t < t_end; ++t) {
    float* buf = stage + ((t - t_begin) % 3) * kArr;
    if (t + 1 < t_end) stage_tile(t + 1, stage + ((t + 1 - t_begin) % 3) * kArr);
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
    float acc[RTH][CT];
#pragma unroll
    for (int a = 0; a < RTH; ++a)
#pragma unroll
      for (int c = 0; c < CT; ++c) acc[a][c] = 0.f;
    const float* s1 = buf + (ty * RTH) * R;
#pragma unroll
    for (int k0 = 0; k0 < R; k0 += 4) {
      float x2[4][CT];
#pragma unroll
      for (int j = 0; j < 4; ++j) lds_ct<CT>(s2 + (k0 + j) * 64 + tx * CT, x2[j]);
#pragma unroll
      for (int a = 0; a < RTH; ++a) {
        float x1[4];
        lds_ct<4>(s1 + a * R + k0, x1);
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
          for (int c = 0; c < CT; ++c) acc[a][c] = fmaf(x1[j], x2[j][c], acc[a][c]);
      }
    }
    // row ga = i1 * nn + o1 -> source row i1 * mm + i2, column o1 * nn + o2; only the (M, N) window is stored
    const int ga_first = t * ROWS + ty * RTH;
    int i1 = ga_first / nn, o1 = ga_first - i1 * nn;
#pragma unroll
    for (int a = 0; a < RTH; ++a) {
      const bool row_ok = ga_first + a < P;
      const int row = i1 * mm + ci2, col = o1 * nn + co2;
      const int e0 = row * N + col;
      if (vec_base && row_ok && row < M && col + CT <= N && (e0 % CT) == 0) {
        *reinterpret_cast<Raw*>(dst + e0) = raw_pack<T, CT>(acc[a]);
      } else {
#pragma unroll
        for (int c = 0; c < CT; ++c) {
          const int over = c >= cut ? 1 : 0;
          if (row_ok && c < ncols && row + over < M && col + c - over * nn < N)
            store_from_f32<T>(dst, e0 + c + over * hop, acc[a][c]);
        }
      }
      if (++o1 == nn) o1 = 0, ++i1;
    }
  }
  cp_async_wait<0>();
}

// Dense relatives of the two kernels above for the order > 2 chains (no index map): same micro-tiles and staging.
//   tt_matmul_rk_reg_kernel : C[m, n] = A[m, r] . B[r, n]                       (r <= 64; reconstruction chain, tt.py:213-237)
//   tt_project_reg_kernel   : R[r, n] (per split) = Q[rows, r]^T . L[rows, n]   (r <= 32; decomposition sweep, tt.py:129-133)
template <int R>
__global__ void __launch_bounds__(256, 3)
tt_matmul_rk_reg_kernel(const float* __restrict__ A, const float* __restrict__ B, int r, float* __restrict__ C, int m, int n,
                        int tiles_per_cta) {
  pdl_trigger();
  pdl_wait();
  constexpr int CT = 4, TX = 16, RTH = 4, ROWS = 64;
  constexpr int kArr = ROWS * R;
  extern __shared__ __align__(16) float fs[];
  float* s2 = fs;                  // [R][64]  B[k][b0 + c]
  float* stage = s2 + R * 64;      // [3][64][R]
  const int tid = threadIdx.x, ty = tid / TX, tx = tid % TX;
  const int b0 = blockIdx.x * 64;
  const int n_tiles = (m + ROWS - 1) / ROWS;
  const int t_begin = blockIdx.y * tiles_per_cta;
  const int t_end = min(n_tiles, t_begin + tiles_per_cta);
  const int gb0 = b0 + tx * CT;
  const int ncols = min(CT, n - gb0);
  const bool vec_base = ncols >= CT && (n % 4 == 0) && (reinterpret_cast<uintptr_t>(C) & 15) == 0;
  const bool fast = (r == R) && ((reinterpret_cast<uintptr_t>(A) & 15) == 0);
  auto stage_tile = [&](int t, float* buf) {
    const int a0 = t * ROWS;
    if (fast) {
      for (int q = tid; q < kArr / 4; q += 256) {
        const int i = q / (R / 4), k4 = q - i * (R / 4);
        const bool ok = a0 + i < m;
        cp_async16(buf + i * R + k4 * 4, ok ? A + static_cast<int64_t>(a0 + i) * r + k4 * 4 : A, ok);
      }
    } else {
      for (int q = tid; q < kArr; q += 256) {
        const int i = q / R, k = q - i * R;
        buf[q] = (a0 + i < m && k < r) ? A[static_cast<int64_t>(a0 + i) * r + k] : 0.f;
      }
    }
  };
  if (t_begin < t_end) stage_tile(t_begin, stage);
  cp_async_commit();
  for (int idx = tid; idx < R * 64; idx += 256) {
    const int kk = idx / 64, c = idx % 64;
    s2[idx] = (kk < r && b0 + c < n) ? B[static_cast<int64_t>(kk) * n + b0 + c] : 0.f;
  }
  for (int t = t_begin; t < t_end; ++t) {
    float* buf = stage + ((t - t_begin) % 3) * kArr;
    if (t + 1 < t_end) stage_tile(t + 1, stage + ((t + 1 - t_begin) % 3) * kArr);
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
    float acc[RTH][CT];
#pragma unroll
    for (int a = 0; a < RTH; ++a)
#pragma unroll
      for (int c = 0; c < CT; ++c) acc[a][c] = 0.f;
    const float* s1 = buf + (ty * RTH) * R;
#pragma unroll
    for (int k0 = 0; k0 < R; k0 += 4) {
      float x2[4][CT];
#pragma unroll
      for (int j = 0; j < 4; ++j) lds_ct<CT>(s2 + (k0 + j) * 64 + tx * CT, x2[j]);
#pragma unroll
      for (int a = 0; a < RTH; ++a) {
        float x1[4];
        lds_ct<4>(s1 + a * R + k0, x1);
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
          for (int c = 0; c < CT; ++c) acc[a][c] = fmaf(x1[j], x2[j][c], acc[a][c]);
      }
    }
#pragma unroll
    for (int a = 0; a < RTH; ++a) {
      const int ga = t * ROWS + ty * RTH + a;
      if (ga >= m) continue;
      float* dst = C + static_cast<int64_t>(ga) * n + gb0;
      if (vec_base) {
        *reinterpret_cast<float4*>(dst) = make_float4(acc[a][0], acc[a][1], acc[a][2], acc[a][3]);
      } else {
#pragma unroll
        for (int c = 0; c < CT; ++c)
          if (c < ncols) dst[c] = acc[a][c];
      }
    }
  }
  cp_async_wait<0>();
}

template <int R, int CT>
__global__ void __launch_bounds__(256, 2)
tt_project_reg_kernel(const float* __restrict__ L, int64_t l_bs, const float* __restrict__ Q, int64_t q_bs, float* __restrict__ Rout,
                      int64_t r_bs, int64_t split_stride, int rows, int n, int r, int tiles_per_cta) {
  pdl_trigger();
  pdl_wait();
  constexpr int TX = 64 / CT, TY = 256 / TX, RTH = kRegTileRows / TY;
  static_assert(R * CT <= 64, "accumulator registers");
  constexpr int kArr = kRegTileRows * R;
  extern __shared__ __align__(16) float fs[];
  float* stage = fs;               // [3][32][R]
  const float* Lb = L + blockIdx.z * l_bs;
  const float* Qb = Q + blockIdx.z * q_bs;
  float* Rb = Rout + blockIdx.z * r_bs + blockIdx.y * split_stride;
  const int tid = threadIdx.x, ty = tid / TX, tx = tid % TX;
  const int b0 = blockIdx.x * 64;
  const int n_tiles = (rows + kRegTileRows - 1) / kRegTileRows;
  const int t_begin = blockIdx.y * tiles_per_cta;
  const int t_end = min(n_tiles, t_begin + tiles_per_cta);
  const int gb0 = b0 + tx * CT;
  const int ncols = min(CT, n - gb0);
  const bool vec = ncols >= CT && (n % CT == 0) && (reinterpret_cast<uintptr_t>(Lb) % (CT * 4)) == 0;
  const bool fast = (r == R) && ((reinterpret_cast<uintptr_t>(Qb) & 15) == 0);
  float acc[R][CT];
#pragma unroll
  for (int k = 0; k < R; ++k)
#pragma unroll
    for (int c = 0; c < CT; ++c) acc[k][c] = 0.f;
  auto stage_tile = [&](int t, float* buf) {
    const int a0 = t * kRegTileRows;
    if (fast) {
      for (int q = tid; q < kArr / 4; q += 256) {
        const int i = q / (R / 4), k4 = q - i * (R / 4);
        const bool ok = a0 + i < rows;
        cp_async16(buf + i * R + k4 * 4, ok ? Qb + static_cast<int64_t>(a0 + i) * r + k4 * 4 : Qb, ok);
      }
    } else {
      for (int q = tid; q < kArr; q += 256) {
        const int i = q / R, k = q - i * R;
        buf[q] = (a0 + i < rows && k < r) ? Qb[static_cast<int64_t>(a0 + i) * r + k] : 0.f;
      }
    }
  };
  if (t_begin < t_end) stage_tile(t_begin, stage);
  cp_async_commit();
  for (int t = t_begin; t < t_end; ++t) {
    float* buf = stage + ((t - t_begin) % 3) * kArr;
    if (t + 1 < t_end) stage_tile(t + 1, stage + ((t + 1 - t_begin) % 3) * kArr);
    cp_async_commit();
    float x[RTH][CT];
#pragma unroll
    for (int a = 0; a < RTH; ++a) {
      const int ga = t * kRegTileRows + ty * RTH + a;
      const float* src = Lb + static_cast<int64_t>(ga) * n + gb0;
#pragma unroll
      for (int c = 0; c < CT; ++c) x[a][c] = 0.f;
      if (ga < rows) {
        if (vec) {
          lds_ct<CT>(src, x[a]);       // plain vector load (the helper is address-space agnostic)
        } else {
#pragma unroll
          for (int c = 0; c < CT; ++c)
            if (c < ncols) x[a][c] = src[c];
        }
      }
    }
    cp_async_wait<1>();
    __syncthreads();
    const float* sQ = buf + (ty * RTH) * R;
#pragma unroll
    for (int a = 0; a < RTH; ++a)
#pragma unroll
      for (int k4 = 0; k4 < R / 4; ++k4) {
        const float4 q = *reinterpret_cast<const float4*>(sQ + a * R + 4 * k4);
        const float qs[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
          for (int c = 0; c < CT; ++c) acc[4 * k4 + j][c] = fmaf(qs[j], x[a][c], acc[4 * k4 + j][c]);
      }
  }
  cp_async_wait<0>();
  __syncthreads();
  float* red = fs;                  // [TY][R][64] floats over the (dead) staging area
#pragma unroll
  for (int k = 0; k < R; ++k) sts_ct<CT>(red + (ty * R + k) * 64 + tx * CT, acc[k]);
  __syncthreads();
#pragma unroll
  for (int u = 0; u < R * 64 / 256; ++u) {
    const int o = tid + u * 256;
    const int k = o / 64, col = o % 64;
    float sum = 0.f;
#pragma unroll
    for (int y = 0; y < TY; ++y) sum += red[(y * R + k) * 64 + col];
    if (k < r && b0 + col < n) Rb[static_cast<int64_t>(k) * n + b0 + col] = sum;
  }
}

// Dense variant for order > 2: m, v are fp32 (M, N) work matrices (already reconstructed + de-interleaved).
template <typename T>
__global__ void tt_adam_dense_kernel(T* __restrict__ p, const T* __restrict__ g, float* __restrict__ m,
                                     float* __restrict__ v, int64_t n, float beta1, float omb1, float beta2, float omb2,
                                     float eps, float step_size, float lr_wd) {
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const float gv = load_as_f32<T>(g, i);
    float pv = load_as_f32<T>(p, i);
    const float mo = beta1 * m[i] + omb1 * gv;
    const float vo = beta2 * fmaxf(v[i], 0.f) + omb2 * gv * gv;
    pv -= step_size * (mo / (sqrtf(vo) + eps));
    if (lr_wd > 0.f) pv -= lr_wd * pv;
    store_from_f32<T>(p, i, pv);
    m[i] = mo;
    v[i] = vo;
  }
}

// Dense TT-Adam for order > 2 on moments kept in the INTERLEAVED layout (the layout the reconstruction chain produces and
// the decomposition sweep consumes): m, v are fp32 tensors of (mm*nn)^order elements in (i1,o1,...,id,od) order, updated
// in place; p and g are addressed through the index map; padded positions get m = v = 0 (the reference crops the
// reconstruction to (M, N) and zero-pads again, ttadam.py:71-84 + tt.py:48-58).  Saves the de-interleave of both
// reconstructed moments and the interleave of both updated moments: four passes over the padded matrix per step.
template <typename T>
__global__ void tt_adam_interleaved_kernel(T* __restrict__ p, const T* __restrict__ g, float* __restrict__ m,
                                           float* __restrict__ v, int M, int N, FastDiv fm, FastDiv fn, int order,
                                           int64_t total, float beta1, float omb1, float beta2, float omb2, float eps,
                                           float step_size, float lr_wd) {
  const bool small = total < (int64_t(1) << 32);
  for (int64_t idx = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    int64_t row, col;
    if (small) decode_interleaved(static_cast<uint32_t>(idx), fm, fn, order, row, col);
    else decode_interleaved64(idx, fm.d, fn.d, order, row, col);
    float mo = 0.f, vo = 0.f;
    if (row < M && col < N) {
      const int64_t e = row * N + col;
      const float gv = load_as_f32<T>(g, e);
      float pv = load_as_f32<T>(p, e);
      mo = beta1 * m[idx] + omb1 * gv;                                   // ttadam.py:92
      vo = beta2 * fmaxf(v[idx], 0.f) + omb2 * gv * gv;                  // ttadam.py:84,93
      pv -= step_size * (mo / (sqrtf(vo) + eps));                        // ttadam.py:94,103,108
      if (lr_wd > 0.f) pv -= lr_wd * pv;                                 // ttadam.py:110-111
      store_from_f32<T>(p, e, pv);
    }
    m[idx] = mo;
    v[idx] = vo;
  }
}

// Four consecutive interleaved positions per thread (nn % 4 == 0: they differ in the last output digit only, so they are
// four consecutive columns of one source row): one index decode per four elements, 16-byte accesses on the interleaved
// side and one vector access on the (M, N) side when N % 4 == 0.  MODE 0: interleave (src -> out4), 1: de-interleave
// (in4 -> dst), 2: the TT-Adam update of tt_adam_interleaved_kernel.
template <typename T, int MODE>
__global__ void __launch_bounds__(256)
tt_interleaved_vec4_kernel(T* __restrict__ p, const T* __restrict__ g, float* __restrict__ m, float* __restrict__ v, int M,
                           int N, FastDiv fm, FastDiv fn, int order, uint32_t total4, float beta1, float omb1, float beta2,
                           float omb2, float eps, float step_size, float lr_wd) {
  using Raw = typename RawVec<T, 4>::type;
  const bool src_vec = (N % 4 == 0) && ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g)) % sizeof(Raw)) == 0;
  for (uint32_t i4 = blockIdx.x * blockDim.x + threadIdx.x; i4 < total4; i4 += gridDim.x * blockDim.x) {
    const uint32_t idx = i4 * 4;
    int64_t row, col;
    decode_interleaved(idx, fm, fn, order, row, col);
    const bool row_ok = row < M;
    const int64_t left = N - col;
    const int ncol = row_ok ? static_cast<int>(left < 4 ? left : 4) : 0;      // valid columns (<= 0: none)
    const int64_t e = row * N + col;
    const bool vec = src_vec && ncol == 4;
    float gv[4] = {0.f, 0.f, 0.f, 0.f}, pv[4] = {0.f, 0.f, 0.f, 0.f};
    if (MODE != 1) {
      if (vec) {
        raw_unpack<T, 4>(*reinterpret_cast<const Raw*>(g + e), gv);
        if (MODE == 2) raw_unpack<T, 4>(*reinterpret_cast<const Raw*>(p + e), pv);
      } else {
#pragma unroll
        for (int c = 0; c < 4; ++c)
          if (c < ncol) {
            gv[c] = load_as_f32<T>(g, e + c);
            if (MODE == 2) pv[c] = load_as_f32<T>(p, e + c);
          }
      }
    }
    if (MODE == 0) {
      *reinterpret_cast<float4*>(m + idx) = make_float4(gv[0], gv[1], gv[2], gv[3]);
      continue;
    }
    const float4 m4 = *reinterpret_cast<const float4*>(m + idx);
    float mo[4] = {m4.x, m4.y, m4.z, m4.w};
    if (MODE == 2) {
      const float4 v4 = *reinterpret_cast<const float4*>(v + idx);
      float vo[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        if (c < ncol) {
          mo[c] = beta1 * mo[c] + omb1 * gv[c];                                   // ttadam.py:92
          vo[c] = beta2 * fmaxf(vo[c], 0.f) + omb2 * gv[c] * gv[c];               // ttadam.py:84,93
          pv[c] -= step_size * (mo[c] / (sqrtf(vo[c]) + eps));                    // ttadam.py:94,103,108
          if (lr_wd > 0.f) pv[c] -= lr_wd * pv[c];                                // ttadam.py:110-111
        } else {
          mo[c] = vo[c] = 0.f;                                                    // padded positions
        }
      }
      *reinterpret_cast<float4*>(m + idx) = make_float4(mo[0], mo[1], mo[2], mo[3]);
      *reinterpret_cast<float4*>(v + idx) = make_float4(vo[0], vo[1], vo[2], vo[3]);
    } else {
#pragma unroll
      for (int c = 0; c < 4; ++c) pv[c] = mo[c];
    }
    if (vec) {
      *reinterpret_cast<Raw*>(p + e) = raw_pack<T, 4>(pv);
    } else {
#pragma unroll
      for (int c = 0; c < 4; ++c)
        if (c < ncol) store_from_f32<T>(p, e + c, pv[c]);
    }
  }
}

// the vec4 kernels apply when the last output digit runs over a multiple of 4 and 32-bit indices suffice
static inline bool interleaved_vec4_ok(int nn, int64_t total, const void* a, const void* b) {
  return nn % 4 == 0 && total < (int64_t(1) << 32) && ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b)) & 15) == 0;
}

static inline int grid_for(int64_t n, int threads) {
  const int64_t b = (n + threads - 1) / threads;
  return static_cast<int>(std::min<int64_t>(b, int64_t(num_sms()) * 16));
}


template <typename T, int R>
static int launch_adam2(bool head, void* p, const void* g, const float* G1m, const float* G2m, const float* G1v,
                        const float* G2v, int r, const float* Qm, const float* Qv, float* Rm, float* Rv, float* Xm,
                        float* Xv, int M, int N, int mm, int nn, float beta1, float omb1, float beta2, float omb2, float eps,
                        float step_size, float lr_wd, int first_step, float* part, size_t part_bytes, cudaStream_t stream) {
  const int P = mm * nn;
  const int n_tiles = ceil_div(P, 64);
  const size_t smem = (size_t(4) * R * 64 + size_t(2) * 64 * R + (R == 64 ? 0 : size_t(2) * 64 * 64)) * sizeof(float);
  if (head) {
    auto k = tt_adam2_kernel<T, R, true>;
    SOWB_CHECK_CUDA(set_max_smem_once(k, size_t(smem)));
    SOWB_CHECK_CUDA(launch_pdl(k, dim3(n_tiles), dim3(256), smem, stream, static_cast<T*>(p), static_cast<const T*>(g), G1m, G2m,
                               G1v, G2v, r, Qm, Qv, Rm, Rv, Xm, Xv, M, N, mm, nn, beta1, omb1, beta2, omb2, eps, step_size,
                               lr_wd, first_step, 1, int64_t(0)));
  } else {
    if constexpr (R <= 16) {
      // ranks <= 16: projection accumulated in registers (tt_adam2_reg_kernel); SOWB_TT_REG=0 keeps the kernel below
      static const bool use_reg = [] { const char* e = getenv("SOWB_TT_REG"); return e == nullptr || atoi(e) != 0; }();
      if (use_reg && nn >= 4 && (int64_t(mm) * mm + 1) * N < (int64_t(1) << 31)) {
        constexpr int CT = 32 / R;
        int per;
        const int splits = reg_kernel_splits(P, &per);
        const int64_t rp = int64_t(r) * P;
        float* dm = Rm;
        float* dv = Rv;
        if (splits > 1) {
          const size_t need = size_t(2) * splits * rp * sizeof(float);
          if (part == nullptr || part_bytes < need)
            return set_error(SOWB_EWORKSPACE, "tt_adam2: workspace %zu B < %zu B for the projection partials", part_bytes, need);
          dm = part, dv = part + splits * rp;
        }
        auto k = tt_adam2_reg_kernel<T, R, CT>;
        constexpr size_t rsmem = reg_kernel_smem(R);
        SOWB_CHECK_CUDA(set_max_smem_once(k, size_t(rsmem)));
        SOWB_CHECK_CUDA(launch_pdl(k, dim3(n_tiles, splits), dim3(256), rsmem, stream, static_cast<T*>(p),
                                   static_cast<const T*>(g), G1m, G2m, G1v, G2v, r, Qm, Qv, dm, dv, M, N, mm, nn, beta1, omb1,
                                   beta2, omb2, eps, step_size, lr_wd, first_step, per, splits > 1 ? rp : int64_t(0)));
        if (splits > 1) return launch_sum_splits(part, splits, rp, splits * rp, Rm, Rv - Rm, rp, 2, stream);
        return SOWB_OK;
      }
    }
    // strips x row-ranges: enough CTAs that every SM holds as many as its shared memory admits (the per-tile chain
    // load -> reconstruct -> update -> project is latency-bound inside one CTA); every CTA stores its [r x 64]
    // accumulators once, as the partial of its row-range, and sum_splits_kernel adds the partials in range order
    const int ctas_per_sm = std::max(1, std::min(R <= 16 ? 4 : (R <= 32 ? 3 : 2), int(size_t(220) * 1024 / smem)));
    int splits = std::max(1, (2 * ctas_per_sm * num_sms()) / n_tiles);
    splits = std::min(splits, n_tiles);
    const int per = ceil_div(n_tiles, splits);
    splits = ceil_div(n_tiles, per);
    const int64_t rp = int64_t(r) * P;
    float* dm = Rm;
    float* dv = Rv;
    if (splits > 1) {
      const size_t need = size_t(2) * splits * rp * sizeof(float);
      if (part == nullptr || part_bytes < need)
        return set_error(SOWB_EWORKSPACE, "tt_adam2: workspace %zu B < %zu B for the projection partials", part_bytes, need);
      dm = part, dv = part + splits * rp;
    }
    auto k = tt_adam2_kernel<T, R, false>;
    SOWB_CHECK_CUDA(set_max_smem_once(k, size_t(smem)));
    SOWB_CHECK_CUDA(launch_pdl(k, dim3(n_tiles, splits), dim3(256), smem, stream, static_cast<T*>(p), static_cast<const T*>(g),
                               G1m, G2m, G1v, G2v, r, Qm, Qv, dm, dv, Xm, Xv, M, N, mm, nn, beta1, omb1, beta2, omb2, eps,
                               step_size, lr_wd, first_step, per, splits > 1 ? rp : int64_t(0)));
    if (splits > 1) return launch_sum_splits(part, splits, rp, splits * rp, Rm, Rv - Rm, rp, 2, stream);
  }
  SOWB_CHECK_CUDA(cudaGetLastError());
  return SOWB_OK;
}

template <typename T>
static int dispatch_adam2(bool head, void* p, const void* g, const float* G1m, const float* G2m, const float* G1v,
                          const float* G2v, int r, const float* Qm, const float* Qv, float* Rm, float* Rv, float* Xm,
                          float* Xv, int M, int N, int mm, int nn, float beta1, float omb1, float beta2, float omb2,
                          float eps, float step_size, float lr_wd, int first_step, float* part, size_t part_bytes,
                          cudaStream_t stream) {
#define SOWB_ADAM2(RR)                                                                                                \
  return launch_adam2<T, RR>(head, p, g, G1m, G2m, G1v, G2v, r, Qm, Qv, Rm, Rv, Xm, Xv, M, N, mm, nn, beta1, omb1,     \
                             beta2, omb2, eps, step_size, lr_wd, first_step, part, part_bytes, stream)
  if (r <= 8) SOWB_ADAM2(8);
  if (r <= 16) SOWB_ADAM2(16);
  if (r <= 32) SOWB_ADAM2(32);
  SOWB_ADAM2(64);
#undef SOWB_ADAM2
}

// tt_project2 through the register-accumulating kernel (projection only).  part: [splits][r][P] partials when splits > 1
template <typename T, int R, int CT>
static int launch_project2_reg(const T* src, int M, int N, int mm, int nn, const float* Q, float* Rout, int r, float* part,
                               size_t part_bytes, cudaStream_t stream) {
  const int P = mm * nn;
  int per;
  const int splits = reg_kernel_splits(P, &per);
  const int64_t rp = int64_t(r) * P;
  float* dst = Rout;
  if (splits > 1) {
    const size_t need = size_t(splits) * rp * sizeof(float);
    if (part == nullptr || part_bytes < need)
      return set_error(SOWB_EWORKSPACE, "tt_project2: workspace %zu B < required %zu B (tt_project2_workspace_bytes)", part_bytes, need);
    dst = part;
  }
  auto k = tt_adam2_reg_kernel<T, R, CT, true>;
  constexpr size_t smem = reg_proj_smem(R, CT);
  SOWB_CHECK_CUDA(set_max_smem_once(k, smem));
  T* no_p = nullptr;
  const float* nf = nullptr;
  float* nfm = nullptr;
  SOWB_CHECK_CUDA(launch_pdl(k, dim3(ceil_div(P, 64), splits), dim3(256), smem, stream, no_p, src, nf, nf, nf, nf, r, Q, nf, dst,
                             nfm, M, N, mm, nn, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 1, per, splits > 1 ? rp : int64_t(0)));
  if (splits > 1) return launch_sum_splits(part, splits, rp, 0, Rout, 0, rp, 1, stream);
  return SOWB_OK;
}

template <typename T>
static int dispatch_project2_reg(const T* src, int M, int N, int mm, int nn, const float* Q, float* Rout, int r, float* part,
                                 size_t part_bytes, cudaStream_t stream) {
  if (r <= 8) return launch_project2_reg<T, 8, 4>(src, M, N, mm, nn, Q, Rout, r, part, part_bytes, stream);
  if (r <= 16) return launch_project2_reg<T, 16, 4>(src, M, N, mm, nn, Q, Rout, r, part, part_bytes, stream);
  return launch_project2_reg<T, 32, 2>(src, M, N, mm, nn, Q, Rout, r, part, part_bytes, stream);
}

static bool project2_reg_ok(int N, int mm, int nn, int r) {
  static const bool enabled = [] { const char* e = getenv("SOWB_TT_REG"); return e == nullptr || atoi(e) != 0; }();
  // measured at 4096^2 fp32: 21 / 29 / 46 us at r = 8 / 16 / 32 against 83-85 us for the tiled kernel; r = 64 (one column per
  // thread) 133 us against 89 us: the tiled kernel keeps the ranks above 32
  return enabled && r <= 32 && nn >= 4 && (int64_t(mm) * mm + 1) * N < (int64_t(1) << 31);
}

}  // namespace sowb

using namespace sowb;

extern "C" {

static int adam2_common(bool head, void* p, const void* g, const float* G1m, const float* G2m, const float* G1v,
                        const float* G2v, int r, const float* Qm, const float* Qv, float* Rm, float* Rv, float* Xm,
                        float* Xv, int M, int N, int mm, int nn, double beta1_d, double beta2_d, double eps_d,
                        double step_size_d, double lr_wd_d, int first_step, int dtype, void* ws, size_t ws_bytes,
                        void* stream_) {
  float* part = static_cast<float*>(ws);
  const float beta1 = float(beta1_d), beta2 = float(beta2_d), omb1 = float(1.0 - beta1_d), omb2 = float(1.0 - beta2_d);
  SOWB_REQUIRE(g != nullptr, "tt_adam2: null gradient pointer");
  SOWB_REQUIRE_TT_DTYPE("tt_adam2", dtype);
  if (int rc0 = ensure_context_for(g)) return rc0;
  SOWB_REQUIRE(first_step || (G1m && G2m && G1v && G2v), "tt_adam2: null core pointer");
  SOWB_REQUIRE(r > 0 && r <= 64, "tt_adam2: rank %d unsupported (1..64)", r);
  SOWB_REQUIRE(int64_t(mm) * mm >= M && int64_t(nn) * nn >= N, "tt_adam2: mm/nn too small for (M,N)");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (dtype == SOWB_BF16)
    return dispatch_adam2<__nv_bfloat16>(head, p, g, G1m, G2m, G1v, G2v, r, Qm, Qv, Rm, Rv, Xm, Xv, M, N, mm, nn, beta1, omb1,
                                         beta2, omb2, float(eps_d), float(step_size_d), float(lr_wd_d), first_step, part, ws_bytes,
                                         stream);
  if (dtype == SOWB_F32)
    return dispatch_adam2<float>(head, p, g, G1m, G2m, G1v, G2v, r, Qm, Qv, Rm, Rv, Xm, Xv, M, N, mm, nn, beta1, omb1, beta2,
                                 omb2, float(eps_d), float(step_size_d), float(lr_wd_d), first_step, part, ws_bytes, stream);
  return set_error(SOWB_EINVAL, "tt_adam2: unknown dtype %d", dtype);
}

int tt_adam2_head(const void* g, const float* G1m, const float* G2m, const float* G1v, const float* G2v, int r, float* Xm,
                  float* Xv, int M, int N, int mm, int nn, double beta1, double beta2, int first_step, int dtype,
                  void* stream) {
  SOWB_REQUIRE(Xm && Xv, "tt_adam2_head: null output pointer");
  return adam2_common(true, nullptr, g, G1m, G2m, G1v, G2v, r, nullptr, nullptr, nullptr, nullptr, Xm, Xv, M, N, mm, nn,
                      beta1, beta2, 0.0, 0.0, 0.0, first_step, dtype, nullptr, 0, stream);
}

int tt_adam2_fused(void* p, const void* g, const float* G1m, const float* G2m, const float* G1v, const float* G2v, int r,
                   const float* Qm, const float* Qv, float* Rm, float* Rv, int M, int N, int mm, int nn, double beta1,
                   double beta2, double eps, double step_size, double lr_wd, int first_step, int dtype, void* ws,
                   size_t ws_bytes, void* stream) {
  SOWB_REQUIRE(p && Qm && Qv && Rm && Rv, "tt_adam2_fused: null pointer argument");
  return adam2_common(false, p, g, G1m, G2m, G1v, G2v, r, Qm, Qv, Rm, Rv, nullptr, nullptr, M, N, mm, nn, beta1, beta2, eps,
                      step_size, lr_wd, first_step, dtype, ws, ws_bytes, stream);
}

// upper bound of the split-partial scratch of tt_adam2_fused / tt_adam2_step: 2 moments x splits x r x P floats with
// splits * P <= max(P, 2 * ctas_per_sm * sms * 64) and r * ctas_per_sm <= 128 on the CUDA-core kernel (launch_adam2), and
// splits * P <= sms * 128 at r <= 64 on the tensor-core kernel (tt_tc.cu)
size_t tt_adam2_fused_workspace_bytes(int mm, int nn) {
  const size_t P_pad = (size_t(mm) * nn + 127) / 128 * 128;
  const size_t elems = std::max<size_t>(size_t(64) * P_pad, size_t(128) * 2 * size_t(num_sms()) * 64);
  return 2 * elems * sizeof(float);
}

// Cholesky-QR scratch: [2 blocks of batch x (L 64x64 + dinv 64) fp64][batch flags][Gram partials batch x n_part x r x r fp64]
struct CqPlan {
  bool ok;            // Cholesky-QR applies (r <= 64, m >= 64)
  int n_part;         // Gram partials (row-block groups) per matrix
  size_t g_bytes, flag_off, part_off, total;
};

static CqPlan cq_plan(int m, int r, int batch) {
  CqPlan pl{};
  pl.ok = r <= kCqMaxR && m >= 64 && batch <= 65535;
  if (!pl.ok) return pl;
  // enough CTAs for about two waves, never more than the 128-row blocks of one matrix
  pl.n_part = std::max(1, std::min(ceil_div(m, kCqGramRows), ceil_div(2 * num_sms(), batch)));
  pl.g_bytes = size_t(batch) * kCqWsPerBatch;
  pl.flag_off = (2 * pl.g_bytes + 15) & ~size_t(15);
  pl.part_off = (pl.flag_off + size_t(batch) * sizeof(int) + 15) & ~size_t(15);
  pl.total = pl.part_off + size_t(batch) * pl.n_part * r * r * sizeof(double);
  return pl;
}

size_t sow_thin_qr_workspace_bytes(int m, int r, int batch) {
  if (m <= 0 || r <= 0 || batch <= 0) return 0;
  const CqPlan pl = cq_plan(m, r, batch);
  return pl.ok ? pl.total : size_t(batch) * m * r * sizeof(float);
}

int sow_thin_qr(const float* X, int64_t x_batch_stride, int ldx, float* Q, int64_t q_batch_stride, int m, int r,
                int batch, void* ws, size_t ws_bytes, void* stream_) {
  SOWB_REQUIRE(X && Q && ws, "sow_thin_qr: null pointer argument");
  if (int rc0 = ensure_context_for(X)) return rc0;
  SOWB_REQUIRE(m > 0 && r > 0 && batch > 0 && ldx >= r, "sow_thin_qr: bad dimensions (m=%d r=%d ldx=%d batch=%d)", m, r, ldx, batch);
  SOWB_REQUIRE(r <= m, "sow_thin_qr: rank %d exceeds the row count %d (the reference fails here too: tt.py:135)", r, m);
  SOWB_REQUIRE(r <= 4096, "sow_thin_qr: rank %d too large", r);
  SOWB_REQUIRE((reinterpret_cast<uintptr_t>(ws) & 15) == 0, "sow_thin_qr: workspace must be 16-byte aligned");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const size_t need = sow_thin_qr_workspace_bytes(m, r, batch);
  if (ws_bytes < need)
    return set_error(SOWB_EWORKSPACE, "sow_thin_qr: workspace %zu B < required %zu B (sow_thin_qr_workspace_bytes)", ws_bytes, need);
  const CqPlan pl = cq_plan(m, r, batch);
  if (pl.ok) {
    // Cholesky-QR: Gram partials (all SMs) -> fixed-order sum -> Cholesky (one CTA per matrix) -> triangular solve per
    // row (all SMs)
    uint8_t* w8 = static_cast<uint8_t*>(ws);
    double* wsd = reinterpret_cast<double*>(w8);
    double* wsd2 = reinterpret_cast<double*>(w8 + pl.g_bytes);          // second-pass factor block
    int* flags = reinterpret_cast<int*>(w8 + pl.flag_off);
    double* part = reinterpret_cast<double*>(w8 + pl.part_off);
    dim3 ggrid(pl.n_part, batch);
    dim3 grid(ceil_div(m, kCqRows), batch);
    static const bool mma_solve_enabled = [] { const char* e = getenv("SOWB_QR_MMA"); return e == nullptr || atoi(e) != 0; }();
    const bool use_mma_solve = mma_solve_enabled && r > 16;
    constexpr size_t solve_smem = (kCqMaxR * (kCqMaxR + 1) + kCqMaxR) * sizeof(double) + size_t(kCqRows) * (kCqMaxR + 1) * sizeof(float);
    auto solve = [&](const float* src, int64_t bs, int ld, const double* fac, const int* only_if) -> cudaError_t {
      if (use_mma_solve)
        return launch_pdl(cq_solve_mma_kernel, dim3(ceil_div(m, 64), batch), dim3(256), size_t(3) * 64 * kCqLd * sizeof(double),
                          stream, src, bs, ld, Q, q_batch_stride, fac, m, r, only_if);
#define SOWB_CQ_SOLVE(RQ)                                                                                               \
  do {                                                                                                                  \
    cudaError_t e_ = set_max_smem_once(cq_solve_kernel<RQ>, solve_smem);                                                \
    if (e_ != cudaSuccess) return e_;                                                                                   \
    return launch_pdl(cq_solve_kernel<RQ>, grid, dim3(kCqRows), solve_smem, stream, src, bs, ld, Q, q_batch_stride,     \
                      fac, m, r, only_if);                                                                              \
  } while (0)
      if (r <= 8) SOWB_CQ_SOLVE(8);
      if (r <= 16) SOWB_CQ_SOLVE(16);
      if (r <= 32) SOWB_CQ_SOLVE(32);
      SOWB_CQ_SOLVE(64);
#undef SOWB_CQ_SOLVE
    };
    // ranks above 16: Gram and solve on the fp64 tensor path (SOWB_QR_MMA=0 keeps the scalar kernels)
    static const bool mma_enabled = [] { const char* e = getenv("SOWB_QR_MMA"); return e == nullptr || atoi(e) != 0; }();
    const bool use_mma = mma_enabled && r > 16;
    constexpr size_t chol_smem = (size_t(2) * kCqMaxR * (kCqMaxR + 1) + 2 * kCqMaxR) * sizeof(double);
    constexpr size_t gram_mma_smem = size_t(kCqGramRows) * kCqLd * sizeof(double);
    constexpr size_t solve_mma_smem = size_t(3) * 64 * kCqLd * sizeof(double);
    SOWB_CHECK_CUDA(set_max_smem_once(cq_chol_kernel, chol_smem));
    if (use_mma) {
      SOWB_CHECK_CUDA(set_max_smem_once(cq_gram_mma_kernel, gram_mma_smem));
      SOWB_CHECK_CUDA(set_max_smem_once(cq_solve_mma_kernel, solve_mma_smem));
    }
    auto gram = [&](const float* src, int64_t bs, int ld, const int* only_if) -> cudaError_t {
      if (use_mma) return launch_pdl(cq_gram_mma_kernel, ggrid, dim3(256), gram_mma_smem, stream, src, bs, ld, part, m, r, only_if);
      switch (ceil_div(r, 16)) {
        case 1: return launch_pdl(cq_gram_kernel<1>, ggrid, dim3(256), 0, stream, src, bs, ld, part, m, r, only_if);
        case 2: return launch_pdl(cq_gram_kernel<2>, ggrid, dim3(256), 0, stream, src, bs, ld, part, m, r, only_if);
        case 3: return launch_pdl(cq_gram_kernel<3>, ggrid, dim3(256), 0, stream, src, bs, ld, part, m, r, only_if);
        default: return launch_pdl(cq_gram_kernel<4>, ggrid, dim3(256), 0, stream, src, bs, ld, part, m, r, only_if);
      }
    };
    SOWB_CHECK_CUDA(gram(X, x_batch_stride, ldx, nullptr));
    SOWB_CHECK_CUDA(cudaGetLastError());
    dim3 sgrid(ceil_div(r * r, 256), batch);
    // r <= 32: the Cholesky CTA sums the partials itself (same order as cq_sum_kernel); above, the sum needs more CTAs
    const bool fuse_sum = r <= 32;
    const double* no_part = nullptr;
    if (!fuse_sum) SOWB_CHECK_CUDA(launch_pdl(cq_sum_kernel, sgrid, dim3(256), 0, stream, part, pl.n_part, r, wsd, nullptr));
    SOWB_CHECK_CUDA(launch_pdl(cq_chol_kernel, dim3(batch), dim3(1024), chol_smem, stream, wsd, fuse_sum ? part : no_part,
                               pl.n_part, r, flags, nullptr, use_mma ? 1 : 0));
    SOWB_CHECK_CUDA(solve(X, x_batch_stride, ldx, wsd, nullptr));
    // CholeskyQR2 for the flagged matrices only: Q <- Q . chol(Q^T Q)^-T, in place
    SOWB_CHECK_CUDA(gram(Q, q_batch_stride, r, flags));
    SOWB_CHECK_CUDA(cudaGetLastError());
    if (!fuse_sum) SOWB_CHECK_CUDA(launch_pdl(cq_sum_kernel, sgrid, dim3(256), 0, stream, part, pl.n_part, r, wsd2, flags));
    SOWB_CHECK_CUDA(launch_pdl(cq_chol_kernel, dim3(batch), dim3(1024), chol_smem, stream, wsd2, fuse_sum ? part : no_part,
                               pl.n_part, r, nullptr, flags, use_mma ? 1 : 0));
    SOWB_CHECK_CUDA(solve(Q, q_batch_stride, r, wsd2, flags));
    return SOWB_OK;
  }
  const size_t smem = (size_t(r) + kQrWarps * 64 + size_t(kQrWarps) * 32 * 33) * sizeof(float);
  SOWB_CHECK_CUDA(set_max_smem_once(thin_qr_kernel, size_t(smem)));
  thin_qr_kernel<<<batch, kQrThreads, smem, stream>>>(X, x_batch_stride, ldx, Q, q_batch_stride, static_cast<float*>(ws), m, r);
  SOWB_CHECK_CUDA(cudaGetLastError());
  return SOWB_OK;
}

// row-range splits of a projection over m rows: enough CTAs for two waves, at least 4 smem stages per split
static int project_splits(int m, int n_tiles, int batch, int* m_per) {
  int splits = std::max(1, (2 * num_sms()) / std::max(1, n_tiles * batch));
  splits = std::min(splits, ceil_div(m, 4 * kPjTM));
  splits = std::max(1, std::min(splits, 65535));
  *m_per = round_up(ceil_div(m, splits), kPjTM);
  return ceil_div(m, *m_per);
}

// row-range splits of tt_project_reg_kernel: two resident CTAs per SM, about two waves over (strips x batch)
static int project_reg_splits(int m, int n, int batch, int* per) {
  const int n_strips = ceil_div(n, 64), n_rt = ceil_div(m, kRegTileRows);
  int splits = std::max(1, (2 * 2 * num_sms()) / std::max(1, n_strips * batch));
  splits = std::min(std::min(splits, n_rt), 65535);
  *per = ceil_div(n_rt, splits);
  return ceil_div(n_rt, *per);
}

static bool project_reg_ok(int n, int r, int batch) {
  static const bool enabled = [] { const char* e = getenv("SOWB_TT_REG"); return e == nullptr || atoi(e) != 0; }();
  return enabled && r <= 32 && batch <= 65535 && ceil_div(n, 64) <= 2147483647;
}

size_t tt_project_workspace_bytes(int m, int n, int r, int batch) {
  if (m <= 0 || n <= 0 || r <= 0 || batch <= 0) return 0;
  int m_per;
  const int splits = project_splits(m, ceil_div(n, kPjTN), batch, &m_per);
  size_t bytes = splits > 1 ? size_t(batch) * splits * r * n * sizeof(float) : 0;
  if (project_reg_ok(n, r, batch)) {
    int per;
    const int rs = project_reg_splits(m, n, batch, &per);
    if (rs > 1) bytes = std::max(bytes, size_t(batch) * rs * r * n * sizeof(float));
  }
  return bytes;
}

int tt_project(const float* L, int64_t l_batch_stride, const float* Q, int64_t q_batch_stride, float* R,
               int64_t r_batch_stride, int m, int n, int r, int batch, void* ws, size_t ws_bytes, void* stream_) {
  SOWB_REQUIRE(L && Q && R, "tt_project: null pointer argument");
  if (int rc0 = ensure_context_for(L)) return rc0;
  SOWB_REQUIRE(m > 0 && n > 0 && r > 0 && batch > 0, "tt_project: bad dimensions");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (project_reg_ok(n, r, batch)) {
    // ranks <= 32: projection accumulated in registers (the tiled kernel below spends a 64-row rank tile on any rank)
    int per;
    const int splits = project_reg_splits(m, n, batch, &per);
    const int64_t rn = int64_t(r) * n;
    float* dst = R;
    int64_t dst_bs = r_batch_stride, sstride = 0;
    if (splits > 1) {
      const size_t need = size_t(batch) * splits * rn * sizeof(float);
      if (ws == nullptr || ws_bytes < need)
        return set_error(SOWB_EWORKSPACE, "tt_project: workspace %zu B < required %zu B (tt_project_workspace_bytes)", ws_bytes, need);
      dst = static_cast<float*>(ws), dst_bs = splits * rn, sstride = rn;
    }
    const dim3 rgrid(ceil_div(n, 64), splits, batch);
#define SOWB_PJREG(RR, CC)                                                                                             \
  do {                                                                                                                 \
    auto k = tt_project_reg_kernel<RR, CC>;                                                                            \
    constexpr size_t smem = std::max<size_t>(size_t(384) * RR, size_t(1024) * CC * RR);                                \
    SOWB_CHECK_CUDA(set_max_smem_once(k, smem));                                                                       \
    SOWB_CHECK_CUDA(launch_pdl(k, rgrid, dim3(256), smem, stream, L, l_batch_stride, Q, q_batch_stride, dst, dst_bs,   \
                               sstride, m, n, r, per));                                                                \
  } while (0)
    if (r <= 8) SOWB_PJREG(8, 4);
    else if (r <= 16) SOWB_PJREG(16, 4);
    else SOWB_PJREG(32, 2);
#undef SOWB_PJREG
    if (splits > 1) return launch_sum_splits(dst, splits, rn, splits * rn, R, r_batch_stride, rn, batch, stream);
    return SOWB_OK;
  }
  const int n_tiles = ceil_div(n, kPjTN);
  int m_per;
  const int splits = project_splits(m, n_tiles, batch, &m_per);
  const int64_t rn = int64_t(r) * n;
  dim3 grid(n_tiles, splits, batch);
  if (splits == 1) {
    tt_project_kernel<<<grid, kPjThreads, 0, stream>>>(L, l_batch_stride, Q, q_batch_stride, R, r_batch_stride, 0, m, n, r, m_per);
    SOWB_CHECK_CUDA(cudaGetLastError());
    return SOWB_OK;
  }
  const size_t need = size_t(batch) * splits * rn * sizeof(float);
  if (ws == nullptr || ws_bytes < need)
    return set_error(SOWB_EWORKSPACE, "tt_project: workspace %zu B < required %zu B (tt_project_workspace_bytes)", ws_bytes, need);
  float* part = static_cast<float*>(ws);
  tt_project_kernel<<<grid, kPjThreads, 0, stream>>>(L, l_batch_stride, Q, q_batch_stride, part, splits * rn, rn, m, n, r, m_per);
  SOWB_CHECK_CUDA(cudaGetLastError());
  return launch_sum_splits(part, splits, rn, splits * rn, R, r_batch_stride, rn, batch, stream);
}

int tt_gather2(const void* src, int M, int N, int mm, int nn, float* X, int ncols, int dtype, void* stream_) {
  SOWB_REQUIRE(src && X, "tt_gather2: null pointer argument");
  SOWB_REQUIRE_TT_DTYPE("tt_gather2", dtype);
  SOWB_REQUIRE(mm > 0 && nn > 0 && ncols > 0 && int64_t(mm) * mm >= M && int64_t(nn) * nn >= N, "tt_gather2: bad shape");
  if (int rc0 = ensure_context_for(src)) return rc0;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const int64_t total = int64_t(mm) * nn * ncols;
  if (dtype == SOWB_BF16)
    tt_gather2_kernel<__nv_bfloat16><<<grid_for(total, 256), 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(src), M, N, mm, nn, X, ncols);
  else if (dtype == SOWB_F32)
    tt_gather2_kernel<float><<<grid_for(total, 256), 256, 0, stream>>>(static_cast<const float*>(src), M, N, mm, nn, X, ncols);
  else
    return set_error(SOWB_EINVAL, "tt_gather2: unknown dtype %d", dtype);
  SOWB_CHECK_CUDA(cudaGetLastError());
  return SOWB_OK;
}

size_t tt_project2_workspace_bytes(int mm, int nn, int r) {
  if (mm <= 0 || nn <= 0 || r <= 0) return 0;
  int per;
  const int reg_splits = reg_kernel_splits(mm * nn, &per);
  const size_t reg_bytes = reg_splits > 1 ? size_t(reg_splits) * r * mm * nn * sizeof(float) : 0;
  return std::max(reg_bytes, tt_project_workspace_bytes(mm * nn, mm * nn, r, 1));     // either kernel may run
}

int tt_project2(const void* src, int M, int N, int mm, int nn, const float* Q, float* R, int r, int dtype, void* ws,
                size_t ws_bytes, void* stream_) {
  SOWB_REQUIRE(src && Q && R, "tt_project2: null pointer argument");
  SOWB_REQUIRE_TT_DTYPE("tt_project2", dtype);
  SOWB_REQUIRE(mm > 0 && nn > 0 && r > 0 && int64_t(mm) * mm >= M && int64_t(nn) * nn >= N, "tt_project2: bad shape");
  SOWB_REQUIRE(dtype == SOWB_BF16 || dtype == SOWB_F32, "tt_project2: unknown dtype %d", dtype);
  if (int rc0 = ensure_context_for(src)) return rc0;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const int P = mm * nn;
  if (project2_reg_ok(N, mm, nn, r)) {
    // ranks <= 32: the projection accumulates in registers (the tiled kernel below spends a 64-row rank tile on any rank)
    if (dtype == SOWB_BF16)
      return dispatch_project2_reg(static_cast<const __nv_bfloat16*>(src), M, N, mm, nn, Q, R, r, static_cast<float*>(ws), ws_bytes, stream);
    return dispatch_project2_reg(static_cast<const float*>(src), M, N, mm, nn, Q, R, r, static_cast<float*>(ws), ws_bytes, stream);
  }
  const int n_tiles = ceil_div(P, kPjTN);
  int m_per;
  const int splits = project_splits(P, n_tiles, 1, &m_per);
  const int64_t rp = int64_t(r) * P;
  float* dst = R;
  if (splits > 1) {
    const size_t need = size_t(splits) * rp * sizeof(float);
    if (ws == nullptr || ws_bytes < need)
      return set_error(SOWB_EWORKSPACE, "tt_project2: workspace %zu B < required %zu B (tt_project2_workspace_bytes)", ws_bytes, need);
    dst = static_cast<float*>(ws);
  }
  const int64_t stride = splits > 1 ? rp : 0;
  dim3 grid(n_tiles, splits);
  if (dtype == SOWB_BF16)
    tt_project2_kernel<__nv_bfloat16><<<grid, kPjThreads, 0, stream>>>(static_cast<const __nv_bfloat16*>(src), M, N, mm, nn, Q, dst, stride, r, m_per);
  else
    tt_project2_kernel<float><<<grid, kPjThreads, 0, stream>>>(static_cast<const float*>(src), M, N, mm, nn, Q, dst, stride, r, m_per);
  SOWB_CHECK_CUDA(cudaGetLastError());
  if (splits > 1) return launch_sum_splits(dst, splits, rp, 0, R, 0, rp, 1, stream);
  return SOWB_OK;
}

int tt_reconstruct2(const float* G1, const float* G2, int r, void* dst, int M, int N, int mm, int nn, int dtype, void* stream_) {
  SOWB_REQUIRE(G1 && G2 && dst, "tt_reconstruct2: null pointer argument");
  SOWB_REQUIRE_TT_DTYPE("tt_reconstruct2", dtype);
  SOWB_REQUIRE(mm > 0 && nn > 0 && r > 0 && int64_t(mm) * mm >= M && int64_t(nn) * nn >= N, "tt_reconstruct2: bad shape");
  if (int rc0 = ensure_context_for(G1)) return rc0;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const int P = mm * nn;
  SOWB_REQUIRE(dtype == SOWB_BF16 || dtype == SOWB_F32, "tt_reconstruct2: unknown dtype %d", dtype);
  static const bool use_reg = [] { const char* e = getenv("SOWB_TT_REG"); return e == nullptr || atoi(e) != 0; }();
  if (use_reg && r <= 64 && nn >= 4 && (int64_t(mm) * mm + 1) * N < (int64_t(1) << 31)) {
    // strips x row ranges: three resident CTAs per SM, about two waves
    const int n_strips = ceil_div(P, 64), n_rt = ceil_div(P, 64);
    int splits = std::min(n_rt, std::max(1, (2 * 3 * num_sms()) / n_strips));
    const int per = ceil_div(n_rt, splits);
    splits = ceil_div(n_rt, per);
    const dim3 rgrid(n_strips, splits);
#define SOWB_RECON(TT, RR)                                                                                              \
  do {                                                                                                                  \
    auto k = tt_reconstruct2_reg_kernel<TT, RR>;                                                                        \
    constexpr size_t smem = size_t(1024) * RR;                                                                          \
    SOWB_CHECK_CUDA(set_max_smem_once(k, smem));                                                                        \
    SOWB_CHECK_CUDA(launch_pdl(k, rgrid, dim3(256), smem, stream, G1, G2, r, static_cast<TT*>(dst), M, N, mm, nn, per)); \
    return SOWB_OK;                                                                                                     \
  } while (0)
#define SOWB_RECON_R(TT)        \
  do {                          \
    if (r <= 8) SOWB_RECON(TT, 8);   \
    if (r <= 16) SOWB_RECON(TT, 16); \
    if (r <= 32) SOWB_RECON(TT, 32); \
    SOWB_RECON(TT, 64);              \
  } while (0)
    if (dtype == SOWB_BF16) SOWB_RECON_R(__nv_bfloat16);
    SOWB_RECON_R(float);
#undef SOWB_RECON_R
#undef SOWB_RECON
  }
  dim3 grid(ceil_div(P, kRkTile), ceil_div(P, kRkTile));
  SOWB_REQUIRE(grid.y <= 65535, "tt_reconstruct2: unfolding too large");
  if (dtype == SOWB_BF16)
    tt_reconstruct2_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>(G1, G2, r, static_cast<__nv_bfloat16*>(dst), M, N, mm, nn);
  else if (dtype == SOWB_F32)
    tt_reconstruct2_kernel<float><<<grid, 256, 0, stream>>>(G1, G2, r, static_cast<float*>(dst), M, N, mm, nn);
  else
    return set_error(SOWB_EINVAL, "tt_reconstruct2: unknown dtype %d", dtype);
  SOWB_CHECK_CUDA(cudaGetLastError());
  return SOWB_OK;
}

int tt_interleave(const void* src, int M, int N, int mm, int nn, int order, float* out, int dtype, void* stream_) {
  SOWB_REQUIRE(src && out, "tt_interleave: null pointer argument");
  SOWB_REQUIRE_TT_DTYPE("tt_interleave", dtype);
  if (int rc0 = ensure_context_for(src)) return rc0;
  SOWB_REQUIRE(order >= 1 && order <= 8 && mm > 0 && nn > 0, "tt_interleave: bad order/shape");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  int64_t total = 1;
  for (int k = 0; k < order; ++k) total *= int64_t(mm) * nn;
  if (interleaved_vec4_ok(nn, total, out, nullptr) && (dtype == SOWB_BF16 || dtype == SOWB_F32)) {
    const uint32_t total4 = static_cast<uint32_t>(total / 4);
    float* nf = nullptr;
    if (dtype == SOWB_BF16)
      tt_interleaved_vec4_kernel<__nv_bfloat16, 0><<<grid_for(total4, 256), 256, 0, stream>>>(
          nullptr, static_cast<const __nv_bfloat16*>(src), out, nf, M, N, make_fastdiv(mm), make_fastdiv(nn), order, total4, 0.f, 0.f,
          0.f, 0.f, 0.f, 0.f, 0.f);
    else
      tt_interleaved_vec4_kernel<float, 0><<<grid_for(total4, 256), 256, 0, stream>>>(
          nullptr, static_cast<const float*>(src), out, nf, M, N, make_fastdiv(mm), make_fastdiv(nn), order, total4, 0.f, 0.f, 0.f,
          0.f, 0.f, 0.f, 0.f);
    SOWB_CHECK_CUDA(cudaGetLastError());
    return SOWB_OK;
  }
  if (dtype == SOWB_BF16)
    tt_interleave_kernel<__nv_bfloat16><<<grid_for(total, 256), 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(src), M, N, make_fastdiv(mm), make_fastdiv(nn), order, out, total);
  else if (dtype == SOWB_F32)
    tt_interleave_kernel<float><<<grid_for(total, 256), 256, 0, stream>>>(static_cast<const float*>(src), M, N, make_fastdiv(mm), make_fastdiv(nn), order, out, total);
  else
    return set_error(SOWB_EINVAL, "tt_interleave: unknown dtype %d", dtype);
  SOWB_CHECK_CUDA(cudaGetLastError());
  return SOWB_OK;
}

int tt_deinterleave(const float* src, int M, int N, int mm, int nn, int order, void* out, int dtype, void* stream_) {
  SOWB_REQUIRE(src && out, "tt_deinterleave: null pointer argument");
  SOWB_REQUIRE_TT_DTYPE("tt_deinterleave", dtype);
  if (int rc0 = ensure_context_for(src)) return rc0;
  SOWB_REQUIRE(order >= 1 && order <= 8 && mm > 0 && nn > 0, "tt_deinterleave: bad order/shape");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  int64_t total = 1;
  for (int k = 0; k < order; ++k) total *= int64_t(mm) * nn;
  if (interleaved_vec4_ok(nn, total, src, nullptr) && (dtype == SOWB_BF16 || dtype == SOWB_F32)) {
    const uint32_t total4 = static_cast<uint32_t>(total / 4);
    float* in = const_cast<float*>(src);       // MODE 1 only reads it
    float* nf = nullptr;
    if (dtype == SOWB_BF16)
      tt_interleaved_vec4_kernel<__nv_bfloat16, 1><<<grid_for(total4, 256), 256, 0, stream>>>(
          static_cast<__nv_bfloat16*>(out), nullptr, in, nf, M, N, make_fastdiv(mm), make_fastdiv(nn), order, total4, 0.f, 0.f, 0.f,
          0.f, 0.f, 0.f, 0.f);
    else
      tt_interleaved_vec4_kernel<float, 1><<<grid_for(total4, 256), 256, 0, stream>>>(
          static_cast<float*>(out), nullptr, in, nf, M, N, make_fastdiv(mm), make_fastdiv(nn), order, total4, 0.f, 0.f, 0.f, 0.f, 0.f,
          0.f, 0.f);
    SOWB_CHECK_CUDA(cudaGetLastError());
    return SOWB_OK;
  }
  if (dtype == SOWB_BF16)
    tt_deinterleave_kernel<__nv_bfloat16><<<grid_for(total, 256), 256, 0, stream>>>(src, M, N, make_fastdiv(mm), make_fastdiv(nn), order, static_cast<__nv_bfloat16*>(out), total);
  else if (dtype == SOWB_F32)
    tt_deinterleave_kernel<float><<<grid_for(total, 256), 256, 0, stream>>>(src, M, N, make_fastdiv(mm), make_fastdiv(nn), order, static_cast<float*>(out), total);
  else
    return set_error(SOWB_EINVAL, "tt_deinterleave: unknown dtype %d", dtype);
  SOWB_CHECK_CUDA(cudaGetLastError());
  return SOWB_OK;
}

int tt_matmul_rk(const float* A, const float* B, float* C, int m, int n, int r, void* stream_) {
  SOWB_REQUIRE(A && B && C, "tt_matmul_rk: null pointer argument");
  if (int rc0 = ensure_context_for(A)) return rc0;
  SOWB_REQUIRE(m > 0 && n > 0 && r > 0, "tt_matmul_rk: bad dimensions");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  static const bool use_reg = [] { const char* e = getenv("SOWB_TT_REG"); return e == nullptr || atoi(e) != 0; }();
  if (use_reg && r <= 64) {
    const int n_strips = ceil_div(n, 64), n_rt = ceil_div(m, 64);
    int splits = std::min(n_rt, std::max(1, (2 * 3 * num_sms()) / n_strips));
    splits = std::min(splits, 65535);
    const int per = ceil_div(n_rt, splits);
    splits = ceil_div(n_rt, per);
    const dim3 rgrid(n_strips, splits);
#define SOWB_MMRK(RR)                                                                                     \
  do {                                                                                                    \
    auto k = tt_matmul_rk_reg_kernel<RR>;                                                                 \
    constexpr size_t smem = size_t(1024) * RR;                                                            \
    SOWB_CHECK_CUDA(set_max_smem_once(k, smem));                                                          \
    SOWB_CHECK_CUDA(launch_pdl(k, rgrid, dim3(256), smem, stream, A, B, r, C, m, n, per));                \
    return SOWB_OK;                                                                                       \
  } while (0)
    if (r <= 8) SOWB_MMRK(8);
    if (r <= 16) SOWB_MMRK(16);
    if (r <= 32) SOWB_MMRK(32);
    SOWB_MMRK(64);
#undef SOWB_MMRK
  }
  dim3 grid(ceil_div(n, kRkTile), ceil_div(m, kRkTile));
  SOWB_REQUIRE(grid.y <= 65535, "tt_matmul_rk: m too large");
  tt_matmul_rk_kernel<<<grid, 256, 0, stream>>>(A, B, C, m, n, r);
  SOWB_CHECK_CUDA(cudaGetLastError());
  return SOWB_OK;
}

int tt_adam_fused2(void* p, const void* g, const float* G1m, const float* G2m, const float* G1v,
                   const float* G2v, int r, float* m_out, float* v_out, int M, int N, int mm, int nn,
                   double beta1_d, double beta2_d, double eps_d, double step_size_d, double lr_wd_d, int first_step,
                   int dtype, void* stream_) {
  const float beta1 = float(beta1_d), beta2 = float(beta2_d), omb1 = float(1.0 - beta1_d), omb2 = float(1.0 - beta2_d);
  const float eps = float(eps_d), step_size = float(step_size_d), lr_wd = float(lr_wd_d);
  SOWB_REQUIRE(p && g && m_out && v_out, "tt_adam_fused2: null pointer argument");
  SOWB_REQUIRE_TT_DTYPE("tt_adam_fused2", dtype);
  if (int rc0 = ensure_context_for(g)) return rc0;
  SOWB_REQUIRE(first_step || (G1m && G2m && G1v && G2v), "tt_adam_fused2: null core pointer");
  SOWB_REQUIRE(r > 0 && r <= 128, "tt_adam_fused2: rank %d unsupported (1..128)", r);
  SOWB_REQUIRE(int64_t(mm) * mm >= M && int64_t(nn) * nn >= N, "tt_adam_fused2: mm/nn too small for (M,N)");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const int P = mm * nn;
  dim3 grid(ceil_div(P, 64), ceil_div(P, 64));
  const size_t smem = size_t(4) * r * 64 * sizeof(float);
  if (dtype == SOWB_BF16) {
    auto k = tt_adam_fused2_kernel<__nv_bfloat16>;
    SOWB_CHECK_CUDA(set_max_smem_once(k, size_t(smem)));
    k<<<grid, 256, smem, stream>>>(static_cast<__nv_bfloat16*>(p), static_cast<const __nv_bfloat16*>(g), G1m, G2m, G1v,
                                   G2v, r, m_out, v_out, M, N, mm, nn, beta1, omb1, beta2, omb2, eps, step_size, lr_wd, first_step);
  } else if (dtype == SOWB_F32) {
    auto k = tt_adam_fused2_kernel<float>;
    SOWB_CHECK_CUDA(set_max_smem_once(k, size_t(smem)));
    k<<<grid, 256, smem, stream>>>(static_cast<float*>(p), static_cast<const float*>(g), G1m, G2m, G1v, G2v, r, m_out,
                                   v_out, M, N, mm, nn, beta1, omb1, beta2, omb2, eps, step_size, lr_wd, first_step);
  } else {
    return set_error(SOWB_EINVAL, "tt_adam_fused2: unknown dtype %d", dtype);
  }
  SOWB_CHECK_CUDA(cudaGetLastError());
  return SOWB_OK;
}

int tt_adam_interleaved(void* p, const void* g, float* m, float* v, int M, int N, int mm, int nn, int order, double beta1_d,
                        double beta2_d, double eps_d, double step_size_d, double lr_wd_d, int dtype, void* stream_) {
  const float beta1 = float(beta1_d), beta2 = float(beta2_d), omb1 = float(1.0 - beta1_d), omb2 = float(1.0 - beta2_d);
  const float eps = float(eps_d), step_size = float(step_size_d), lr_wd = float(lr_wd_d);
  SOWB_REQUIRE(p && g && m && v, "tt_adam_interleaved: null pointer argument");
  SOWB_REQUIRE_TT_DTYPE("tt_adam_interleaved", dtype);
  SOWB_REQUIRE(order >= 1 && order <= 8 && mm > 0 && nn > 0, "tt_adam_interleaved: bad order/shape");
  if (int rc0 = ensure_context_for(g)) return rc0;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  int64_t total = 1;
  for (int k = 0; k < order; ++k) total *= int64_t(mm) * nn;
  if (interleaved_vec4_ok(nn, total, m, v) && (dtype == SOWB_BF16 || dtype == SOWB_F32)) {
    const uint32_t total4 = static_cast<uint32_t>(total / 4);
    if (dtype == SOWB_BF16)
      tt_interleaved_vec4_kernel<__nv_bfloat16, 2><<<grid_for(total4, 256), 256, 0, stream>>>(
          static_cast<__nv_bfloat16*>(p), static_cast<const __nv_bfloat16*>(g), m, v, M, N, make_fastdiv(mm), make_fastdiv(nn), order,
          total4, beta1, omb1, beta2, omb2, eps, step_size, lr_wd);
    else
      tt_interleaved_vec4_kernel<float, 2><<<grid_for(total4, 256), 256, 0, stream>>>(
          static_cast<float*>(p), static_cast<const float*>(g), m, v, M, N, make_fastdiv(mm), make_fastdiv(nn), order, total4, beta1,
          omb1, beta2, omb2, eps, step_size, lr_wd);
    SOWB_CHECK_CUDA(cudaGetLastError());
    return SOWB_OK;
  }
  if (dtype == SOWB_BF16)
    tt_adam_interleaved_kernel<__nv_bfloat16><<<grid_for(total, 256), 256, 0, stream>>>(
        static_cast<__nv_bfloat16*>(p), static_cast<const __nv_bfloat16*>(g), m, v, M, N, make_fastdiv(mm), make_fastdiv(nn),
        order, total, beta1, omb1, beta2, omb2, eps, step_size, lr_wd);
  else if (dtype == SOWB_F32)
    tt_adam_interleaved_kernel<float><<<grid_for(total, 256), 256, 0, stream>>>(
        static_cast<float*>(p), static_cast<const float*>(g), m, v, M, N, make_fastdiv(mm), make_fastdiv(nn), order, total,
        beta1, omb1, beta2, omb2, eps, step_size, lr_wd);
  else
    return set_error(SOWB_EINVAL, "tt_adam_interleaved: unknown dtype %d", dtype);
  SOWB_CHECK_CUDA(cudaGetLastError());
  return SOWB_OK;
}

// ---- the whole TT-Adam step of an order >= 3 tensor train in one call ---------------------------------------------------
// Host-side composition of the kernels above (no new device code): per moment the reconstruction chain into the interleaved
// dense layout, one interleaved Adam pass over p / g / m / v, then ONE left-to-right sweep that decomposes both moments as a
// batch of two (thin QR + projection per core).  Replaces ~25 separate C-ABI calls issued from Python, which is what bounded
// the step (0.47 ms of host time per 4096 x 4096 order-3 parameter).
struct AdamNPlan {
  int64_t P, T;                 // P = mm * nn, T = P^order
  size_t dense_off, buf_off[2], buf_bytes, qr_off, qr_bytes, pj_off, pj_bytes, total;
  bool ok;
};

static AdamNPlan adamN_plan(int mm, int nn, int order, const int* ranks, int batch = 2) {
  AdamNPlan pl{};
  pl.ok = false;
  if (order < 3 || order > 8 || mm <= 0 || nn <= 0 || ranks == nullptr || ranks[0] != 1 || ranks[order] != 1) return pl;
  pl.P = int64_t(mm) * nn;
  pl.T = 1;
  for (int k = 0; k < order; ++k) {
    pl.T *= pl.P;
    if (pl.T > (int64_t(1) << 34)) return pl;
  }
  int64_t cols = pl.T, buf_elems = 0;
  for (int k = 0; k + 1 < order; ++k) {
    const int64_t rows = int64_t(ranks[k]) * pl.P;
    cols /= pl.P;                                           // columns of the unfolding at core k: P^(order-1-k)
    const int r = ranks[k + 1];
    if (r <= 0 || r > kCqMaxR || r > rows || r > cols || rows > 2147483647 || cols > 2147483647) return pl;
    buf_elems = std::max(buf_elems, int64_t(r) * cols);     // R of the sweep == intermediate of the reconstruction chain
    pl.qr_bytes = std::max(pl.qr_bytes, sow_thin_qr_workspace_bytes(int(rows), r, batch));
    pl.pj_bytes = std::max(pl.pj_bytes, tt_project_workspace_bytes(int(rows), int(cols), r, batch));
  }
  auto up = [](size_t x) { return (x + 255) & ~size_t(255); };
  pl.buf_bytes = up(size_t(batch) * buf_elems * sizeof(float));
  pl.dense_off = 0;
  pl.buf_off[0] = up(size_t(batch) * pl.T * sizeof(float));
  pl.buf_off[1] = pl.buf_off[0] + pl.buf_bytes;
  pl.qr_off = pl.buf_off[1] + pl.buf_bytes;
  pl.qr_bytes = up(pl.qr_bytes);
  pl.pj_off = pl.qr_off + pl.qr_bytes;
  pl.total = pl.pj_off + up(pl.pj_bytes);
  pl.ok = true;
  return pl;
}

size_t tt_adam_nd_workspace_bytes(int mm, int nn, int order, const int* ranks) {
  const AdamNPlan pl = adamN_plan(mm, nn, order, ranks);
  return pl.ok ? pl.total : 0;
}

int tt_adam_nd_step(void* p, const void* g, const float* const* cores_in, float* const* cores_out, const int* ranks, int M, int N,
                  int mm, int nn, int order, double beta1, double beta2, double eps, double step_size, double lr_wd,
                  int first_step, int dtype, void* ws, size_t ws_bytes, void* stream_) {
  SOWB_REQUIRE(p && g && cores_out && ranks && ws, "tt_adam_nd_step: null pointer argument");
  SOWB_REQUIRE_TT_DTYPE("tt_adam_nd_step", dtype);
  SOWB_REQUIRE(first_step || cores_in, "tt_adam_nd_step: null core table");
  const AdamNPlan pl = adamN_plan(mm, nn, order, ranks);
  SOWB_REQUIRE(pl.ok, "tt_adam_nd_step: unsupported order / ranks (order 3..8, boundary ranks 1, inner ranks <= 64 and <= the unfolding sizes)");
  SOWB_REQUIRE((reinterpret_cast<uintptr_t>(ws) & 255) == 0, "tt_adam_nd_step: workspace must be 256-byte aligned");
  if (ws_bytes < pl.total)
    return set_error(SOWB_EWORKSPACE, "tt_adam_nd_step: workspace %zu B < required %zu B (tt_adam_nd_workspace_bytes)", ws_bytes, pl.total);
  if (int rc0 = ensure_context_for(g)) return rc0;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  uint8_t* w = static_cast<uint8_t*>(ws);
  float* dense = reinterpret_cast<float*>(w + pl.dense_off);           // [2][T]: m, v in the interleaved layout
  float* buf[2] = {reinterpret_cast<float*>(w + pl.buf_off[0]), reinterpret_cast<float*>(w + pl.buf_off[1])};
  const int64_t P = pl.P, T = pl.T;
  int rc;
  // 1. old moments: reconstruction chain per moment (tt.py:213-237), or zeros on the first step (ttadam.py:68-70,76-78)
  if (first_step) {
    SOWB_CHECK_CUDA(cudaMemsetAsync(dense, 0, size_t(2) * T * sizeof(float), stream));
  } else {
    for (int b = 0; b < 2; ++b) {
      const float* res = cores_in[0] + int64_t(b) * ranks[0] * P * ranks[1];     // [P, r_1]
      int64_t rows = P;
      for (int k = 1; k < order; ++k) {
        const float* core = cores_in[k] + int64_t(b) * ranks[k] * P * ranks[k + 1];   // [r_k, P * r_{k+1}]
        float* out = (k == order - 1) ? dense + int64_t(b) * T : buf[k & 1];
        const int64_t n = P * ranks[k + 1];
        SOWB_REQUIRE(rows <= 2147483647 && n <= 2147483647, "tt_adam_nd_step: unfolding too large");
        rc = tt_matmul_rk(res, core, out, int(rows), int(n), ranks[k], stream_);
        if (rc) return rc;
        res = out;
        rows *= P;                                                               // [rows, P * r] viewed as [rows * P, r]
      }
    }
  }
  // 2. Adam on p, new moments in place (interleaved layout, zero at padded positions)
  rc = tt_adam_interleaved(p, g, dense, dense + T, M, N, mm, nn, order, beta1, beta2, eps, step_size, lr_wd, dtype, stream_);
  if (rc) return rc;
  // 3. decomposition sweep, both moments as a batch of two (tt.py:111-140)
  const float* cur = dense;
  int64_t cur_bs = T, cols = T;
  for (int k = 0; k + 1 < order; ++k) {
    const int64_t rows = int64_t(ranks[k]) * P;
    cols /= P;
    const int r = ranks[k + 1];
    float* Qk = cores_out[k];                                                    // [2][rows, r]
    rc = sow_thin_qr(cur, cur_bs, int(cols), Qk, rows * r, int(rows), r, 2, w + pl.qr_off, pl.qr_bytes, stream_);
    if (rc) return rc;
    const bool last = (k + 2 == order);
    float* Rk = last ? cores_out[order - 1] : buf[k & 1];                        // [2][r, cols]
    rc = tt_project(cur, cur_bs, Qk, rows * r, Rk, int64_t(r) * cols, int(rows), int(cols), r, 2, w + pl.pj_off, pl.pj_bytes, stream_);
    if (rc) return rc;
    cur = Rk;
    cur_bs = int64_t(r) * cols;
  }
  return SOWB_OK;
}

// from_matrix / to_matrix of an order >= 3 tensor train as one call each (same composition, one matrix instead of two moments)
size_t tt_nd_workspace_bytes(int mm, int nn, int order, const int* ranks) {
  const AdamNPlan pl = adamN_plan(mm, nn, order, ranks, 1);
  return pl.ok ? pl.total : 0;
}

int tt_decompose_nd(const void* src, float* const* cores_out, const int* ranks, int M, int N, int mm, int nn, int order, int dtype,
                    void* ws, size_t ws_bytes, void* stream_) {
  SOWB_REQUIRE(src && cores_out && ranks && ws, "tt_decompose_nd: null pointer argument");
  SOWB_REQUIRE_TT_DTYPE("tt_decompose_nd", dtype);
  const AdamNPlan pl = adamN_plan(mm, nn, order, ranks, 1);
  SOWB_REQUIRE(pl.ok, "tt_decompose_nd: unsupported order / ranks");
  SOWB_REQUIRE((reinterpret_cast<uintptr_t>(ws) & 255) == 0, "tt_decompose_nd: workspace must be 256-byte aligned");
  if (ws_bytes < pl.total)
    return set_error(SOWB_EWORKSPACE, "tt_decompose_nd: workspace %zu B < required %zu B (tt_nd_workspace_bytes)", ws_bytes, pl.total);
  uint8_t* w = static_cast<uint8_t*>(ws);
  float* dense = reinterpret_cast<float*>(w + pl.dense_off);
  float* buf[2] = {reinterpret_cast<float*>(w + pl.buf_off[0]), reinterpret_cast<float*>(w + pl.buf_off[1])};
  int rc = tt_interleave(src, M, N, mm, nn, order, dense, dtype, stream_);
  if (rc) return rc;
  const float* cur = dense;
  int64_t cols = pl.T;
  for (int k = 0; k + 1 < order; ++k) {
    const int64_t rows = int64_t(ranks[k]) * pl.P;
    cols /= pl.P;
    const int r = ranks[k + 1];
    rc = sow_thin_qr(cur, 0, int(cols), cores_out[k], 0, int(rows), r, 1, w + pl.qr_off, pl.qr_bytes, stream_);
    if (rc) return rc;
    float* Rk = (k + 2 == order) ? cores_out[order - 1] : buf[k & 1];
    rc = tt_project(cur, 0, cores_out[k], 0, Rk, 0, int(rows), int(cols), r, 1, w + pl.pj_off, pl.pj_bytes, stream_);
    if (rc) return rc;
    cur = Rk;
  }
  return SOWB_OK;
}

int tt_reconstruct_nd(const float* const* cores, const int* ranks, void* dst, int M, int N, int mm, int nn, int order, int dtype,
                      void* ws, size_t ws_bytes, void* stream_) {
  SOWB_REQUIRE(cores && ranks && dst && ws, "tt_reconstruct_nd: null pointer argument");
  SOWB_REQUIRE_TT_DTYPE("tt_reconstruct_nd", dtype);
  const AdamNPlan pl = adamN_plan(mm, nn, order, ranks, 1);
  SOWB_REQUIRE(pl.ok, "tt_reconstruct_nd: unsupported order / ranks");
  SOWB_REQUIRE((reinterpret_cast<uintptr_t>(ws) & 255) == 0, "tt_reconstruct_nd: workspace must be 256-byte aligned");
  if (ws_bytes < pl.total)
    return set_error(SOWB_EWORKSPACE, "tt_reconstruct_nd: workspace %zu B < required %zu B (tt_nd_workspace_bytes)", ws_bytes, pl.total);
  uint8_t* w = static_cast<uint8_t*>(ws);
  float* dense = reinterpret_cast<float*>(w + pl.dense_off);
  float* buf[2] = {reinterpret_cast<float*>(w + pl.buf_off[0]), reinterpret_cast<float*>(w + pl.buf_off[1])};
  const float* res = cores[0];
  int64_t rows = pl.P;
  for (int k = 1; k < order; ++k) {
    float* out = (k == order - 1) ? dense : buf[k & 1];
    const int64_t n = pl.P * ranks[k + 1];
    SOWB_REQUIRE(rows <= 2147483647 && n <= 2147483647, "tt_reconstruct_nd: unfolding too large");
    const int rc = tt_matmul_rk(res, cores[k], out, int(rows), int(n), ranks[k], stream_);
    if (rc) return rc;
    res = out;
    rows *= pl.P;
  }
  return tt_deinterleave(dense, M, N, mm, nn, order, dst, dtype, stream_);
}

int tt_adam_dense(void* p, const void* g, float* m, float* v, int64_t numel, double beta1_d, double beta2_d,
                  double eps_d, double step_size_d, double lr_wd_d, int dtype, void* stream_) {
  const float beta1 = float(beta1_d), beta2 = float(beta2_d), omb1 = float(1.0 - beta1_d), omb2 = float(1.0 - beta2_d);
  const float eps = float(eps_d), step_size = float(step_size_d), lr_wd = float(lr_wd_d);
  SOWB_REQUIRE(p && g && m && v && numel > 0, "tt_adam_dense: bad argument");
  SOWB_REQUIRE_TT_DTYPE("tt_adam_dense", dtype);
  if (int rc0 = ensure_context_for(g)) return rc0;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (dtype == SOWB_BF16)
    tt_adam_dense_kernel<__nv_bfloat16><<<grid_for(numel, 256), 256, 0, stream>>>(
        static_cast<__nv_bfloat16*>(p), static_cast<const __nv_bfloat16*>(g), m, v, numel, beta1, omb1, beta2, omb2, eps, step_size, lr_wd);
  else if (dtype == SOWB_F32)
    tt_adam_dense_kernel<float><<<grid_for(numel, 256), 256, 0, stream>>>(static_cast<float*>(p), static_cast<const float*>(g),
                                                                         m, v, numel, beta1, omb1, beta2, omb2, eps, step_size, lr_wd);
  else
    return set_error(SOWB_EINVAL, "tt_adam_dense: unknown dtype %d", dtype);
  SOWB_CHECK_CUDA(cudaGetLastError());
  return SOWB_OK;
}

}  // extern "C"
