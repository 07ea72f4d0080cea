// Element-wise glue of the Llama block: rotary position embedding (q and k) and the SwiGLU gate, forward and backward.
//
// Replaces the eager HF chains of transformers/models/llama/modeling_llama.py:
//     q_embed = (q * cos) + (rotate_half(q) * sin)          (apply_rotary_pos_emb, and the same for k)
//     h = act_fn(gate_proj(x)) * up_proj(x)                 (LlamaMLP.forward, act_fn = silu)
// which run as ~12 separate kernels per layer on strided views (mul, neg, cat, add, the zero-filled slice-backward
// buffers and their copies).  Here each element is read once and written once per pass.
//
// The results are bit-identical to the eager chains.  Every rounding eager performs is reproduced in the same place:
// products and sums are formed in fp32 and rounded to the 16-bit type (round to nearest even) exactly where eager writes
// a 16-bit tensor.  r() below means that rounding.
//   rope forward   out[d] = r(r(q[d] cos[d]) + r(-q[d+h] sin[d]))   d <  h = D/2
//                  out[d] = r(r(q[d] cos[d]) + r( q[d-h] sin[d]))   d >= h
//   rope backward  a = r(g cos), b = r(g sin)
//                  dq[d] = r(a[d] + b[d+h]) + 0   d <  h
//                  dq[d] = r(a[d] - b[d-h]) + 0   d >= h
//                  (autograd sums the two slice-backward buffers, which are zero outside their half, into the gradient:
//                  the "+ 0" is that sum, and it turns a -0 into +0)
//   swiglu forward h = r(r(silu(g)) u),  silu(x) = x / (1 + expf(-x))                 (torch's silu_kernel)
//   swiglu bwd     du = r(dh r(silu(g))),  dg = r(silu_backward(r(dh u), g))
//                  silu_backward(dy, x) = dy s (1 + x (1 - s)), s = 1 / (1 + expf(-x))  (torch's silu_backward_kernel)
// The build does not use --use_fast_math: expf, the divisions and the fp32 products are the IEEE / libdevice ones torch
// uses.  The one place where FMA contraction decides the bits, 1 + x (1 - s), is pinned to the fused form nvcc emits
// for torch's expression.
#include "common.cuh"

#include <cuda_fp16.h>

#include <cfloat>

namespace sowb {

namespace {

template <typename H>
struct Cvt;
template <>
struct Cvt<__nv_bfloat16> {
  using H2 = __nv_bfloat162;
  static __device__ __forceinline__ float2 to_f2(H2 v) { return __bfloat1622float2(v); }
  static __device__ __forceinline__ H2 from_f2(float a, float b) { return __floats2bfloat162_rn(a, b); }
  static __device__ __forceinline__ float to_f(__nv_bfloat16 v) { return __bfloat162float(v); }
  static __device__ __forceinline__ __nv_bfloat16 from_f(float v) { return __float2bfloat16_rn(v); }
};
template <>
struct Cvt<__half> {
  using H2 = __half2;
  static __device__ __forceinline__ float2 to_f2(H2 v) { return __half22float2(v); }
  static __device__ __forceinline__ H2 from_f2(float a, float b) { return __floats2half2_rn(a, b); }
  static __device__ __forceinline__ float to_f(__half v) { return __half2float(v); }
  static __device__ __forceinline__ __half from_f(float v) { return __float2half_rn(v); }
};

// r(v): round an fp32 value to the 16-bit type and back
template <typename H>
__device__ __forceinline__ float rnd(float v) {
  return Cvt<H>::to_f(Cvt<H>::from_f(v));
}

// 8 consecutive 16-bit elements <-> 8 floats (one 16-byte access)
template <typename H>
__device__ __forceinline__ void load8(const H* p, float (&f)[8]) {
  const uint4 v = *reinterpret_cast<const uint4*>(p);
  const typename Cvt<H>::H2* h2 = reinterpret_cast<const typename Cvt<H>::H2*>(&v);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float2 t = Cvt<H>::to_f2(h2[j]);
    f[2 * j] = t.x;
    f[2 * j + 1] = t.y;
  }
}
template <typename H>
__device__ __forceinline__ void store8(H* p, const float (&f)[8]) {
  uint4 v;
  typename Cvt<H>::H2* h2 = reinterpret_cast<typename Cvt<H>::H2*>(&v);
#pragma unroll
  for (int j = 0; j < 4; ++j) h2[j] = Cvt<H>::from_f2(f[2 * j], f[2 * j + 1]);
  *reinterpret_cast<uint4*>(p) = v;
}

// One rotary call covers q and k of a layer.  Source (B, H, S, D) with element strides sb / sh / ss and a contiguous last
// dimension; destination (B, S, H, D) contiguous.  cos / sin: (B or 1, S, D) contiguous, batch stride cs_sb (0 when
// broadcast).  One thread owns the 8-element chunk c of the first half of a row and the matching chunk of the second half.
struct RopeSide {
  const void* src;
  void* dst;
  int64_t sb, sh, ss;
  int heads;
  int64_t n;   // B * S * heads * (D / 16) threads
};
struct RopeArgs {
  RopeSide t[2];
  const void* cos;
  const void* sin;
  int64_t cs_sb;
  int S, D;
};

template <typename H, bool kBackward>
__global__ void __launch_bounds__(256) rope_kernel(const RopeArgs a) {
  int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  int side = 0;
  if (i >= a.t[0].n) {
    i -= a.t[0].n;
    side = 1;
    if (i >= a.t[1].n) return;
  }
  const RopeSide& t = a.t[side];
  const int half = a.D >> 1;
  const int chunks = half >> 3;
  const int c = int(i % chunks);
  int64_t r = i / chunks;
  const int hh = int(r % t.heads);
  r /= t.heads;
  const int s = int(r % a.S);
  const int64_t b = r / a.S;

  const H* src = static_cast<const H*>(t.src) + b * t.sb + hh * t.sh + s * t.ss + c * 8;
  H* dst = static_cast<H*>(t.dst) + ((b * a.S + s) * t.heads + hh) * a.D + c * 8;
  const int64_t co = b * a.cs_sb + int64_t(s) * a.D + c * 8;
  const H* cs = static_cast<const H*>(a.cos) + co;
  const H* sn = static_cast<const H*>(a.sin) + co;

  float x1[8], x2[8], c1[8], c2[8], s1[8], s2[8], o1[8], o2[8];
  load8<H>(src, x1);
  load8<H>(src + half, x2);
  load8<H>(cs, c1);
  load8<H>(cs + half, c2);
  load8<H>(sn, s1);
  load8<H>(sn + half, s2);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    if (!kBackward) {
      o1[j] = rnd<H>(x1[j] * c1[j]) + rnd<H>(-x2[j] * s1[j]);
      o2[j] = rnd<H>(x2[j] * c2[j]) + rnd<H>(x1[j] * s2[j]);
    } else {
      // x = upstream gradient g
      const float a1 = rnd<H>(x1[j] * c1[j]), a2 = rnd<H>(x2[j] * c2[j]);
      const float b1 = rnd<H>(x1[j] * s1[j]), b2 = rnd<H>(x2[j] * s2[j]);
      o1[j] = (a1 + b2) + 0.0f;
      o2[j] = (a2 - b1) + 0.0f;
    }
  }
  store8<H>(dst, o1);
  store8<H>(dst + half, o2);
}

// torch's silu / silu_backward in fp32 (ActivationSiluKernel.cu)
__device__ __forceinline__ float silu_f(float x) { return x / (1.0f + expf(-x)); }
__device__ __forceinline__ float silu_bwd_f(float dy, float x) {
  const float s = 1.0f / (1.0f + expf(-x));
  return __fmul_rn(__fmul_rn(dy, s), __fmaf_rn(x, 1.0f - s, 1.0f));
}

template <typename H>
__device__ __forceinline__ void swiglu_fwd_elem(float g, float u, float& h) {
  h = rnd<H>(silu_f(g)) * u;
}
template <typename H>
__device__ __forceinline__ void swiglu_bwd_elem(float dh, float g, float u, float& dg, float& du) {
  du = dh * rnd<H>(silu_f(g));
  dg = silu_bwd_f(rnd<H>(dh * u), g);
}

// n elements, contiguous; 8 per thread with 16-byte accesses, the last n % 8 by the first threads one by one
template <typename H>
__global__ void __launch_bounds__(256) swiglu_fwd_kernel(const H* __restrict__ gate, const H* __restrict__ up,
                                                         H* __restrict__ h, int64_t n) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t nvec = n >> 3;
  if (i < nvec) {
    float g[8], u[8], o[8];
    load8<H>(gate + i * 8, g);
    load8<H>(up + i * 8, u);
#pragma unroll
    for (int j = 0; j < 8; ++j) swiglu_fwd_elem<H>(g[j], u[j], o[j]);
    store8<H>(h + i * 8, o);
  } else if (i - nvec < (n & 7)) {
    const int64_t e = nvec * 8 + (i - nvec);
    float o;
    swiglu_fwd_elem<H>(Cvt<H>::to_f(gate[e]), Cvt<H>::to_f(up[e]), o);
    h[e] = Cvt<H>::from_f(o);
  }
}

template <typename H>
__global__ void __launch_bounds__(256) swiglu_bwd_kernel(const H* __restrict__ dh, const H* __restrict__ gate,
                                                         const H* __restrict__ up, H* __restrict__ dgate,
                                                         H* __restrict__ dup, int64_t n) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t nvec = n >> 3;
  if (i < nvec) {
    float d[8], g[8], u[8], og[8], ou[8];
    load8<H>(dh + i * 8, d);
    load8<H>(gate + i * 8, g);
    load8<H>(up + i * 8, u);
#pragma unroll
    for (int j = 0; j < 8; ++j) swiglu_bwd_elem<H>(d[j], g[j], u[j], og[j], ou[j]);
    store8<H>(dgate + i * 8, og);
    store8<H>(dup + i * 8, ou);
  } else if (i - nvec < (n & 7)) {
    const int64_t e = nvec * 8 + (i - nvec);
    float og, ou;
    swiglu_bwd_elem<H>(Cvt<H>::to_f(dh[e]), Cvt<H>::to_f(gate[e]), Cvt<H>::to_f(up[e]), og, ou);
    dgate[e] = Cvt<H>::from_f(og);
    dup[e] = Cvt<H>::from_f(ou);
  }
}

// ---- RMSNorm (LlamaRMSNorm.forward and its autograd backward) ------------------------------------------------------
//
// Eager runs, per row of H elements (xf = f32(x), r16() = rounding to the 16-bit type, every other op an fp32 op):
//   forward   ms = sum(xf * xf) * factor          (mean: torch's MeanOps multiplies by float(rows) / float(rows * H))
//             rs = rsqrtf(ms + eps),  hb = r16(xf * rs),  y = r16(w * hb)
//   backward  dh = f32(r16(dy * w)),  s = sum(dh * xf)
//             gv = (s * -0.5) * ((rs * rs) * rs)              (rsqrt backward; pow(rs, 3) is rs * rs * rs)
//             d2 = gv * (1 / H)                               (mean backward: torch divides by a scalar as a product
//                                                             with its reciprocal)
//             dx = r16(dh * rs + d2 * (xf * 2))               (the two gradients of xf, each product rounded to fp32)
//             p  = r16(dy * hb), reduced over the rows to dw by torch itself (sum_to_size), as eager's engine does
// The two row sums are torch's inner-dimension fp32 reductions, and at the shapes dispatched here (H a multiple of 128
// up to 4096 and rows >= 16, or H == 128) their order is fixed (ATen/native/cuda/Reduce.cuh, setReduceConfig with
// vectorised input): one warp per row, lane t keeps four accumulators j = 0..3 over the elements 128 k + 4 t + j in
// ascending k, combines them as ((a0 + a1) + a2) + a3, then a shfl_down tree with offsets 16, 8, 4, 2, 1.  The kernels
// below use exactly that mapping, with the row held in registers.  Every product is written with __fmul_rn / __fadd_rn
// so that nvcc cannot contract a product and a sum into one FMA where eager rounds the product first.

template <typename H>
__device__ __forceinline__ void unpack4(uint2 v, float (&f)[4]) {
  const typename Cvt<H>::H2* h2 = reinterpret_cast<const typename Cvt<H>::H2*>(&v);
  const float2 a = Cvt<H>::to_f2(h2[0]), b = Cvt<H>::to_f2(h2[1]);
  f[0] = a.x;
  f[1] = a.y;
  f[2] = b.x;
  f[3] = b.y;
}
template <typename H>
__device__ __forceinline__ uint2 pack4(const float (&f)[4]) {
  uint2 v;
  typename Cvt<H>::H2* h2 = reinterpret_cast<typename Cvt<H>::H2*>(&v);
  h2[0] = Cvt<H>::from_f2(f[0], f[1]);
  h2[1] = Cvt<H>::from_f2(f[2], f[3]);
  return v;
}

// torch's row sum from the four per-lane accumulators; the result in every lane
__device__ __forceinline__ float warp_row_sum(const float (&a)[4]) {
  float v = __fadd_rn(__fadd_rn(__fadd_rn(a[0], a[1]), a[2]), a[3]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = __fadd_rn(v, __shfl_down_sync(0xffffffffu, v, o));
  return __shfl_sync(0xffffffffu, v, 0);
}

constexpr int kNormRowsPerBlock = 8;   // one warp per row

// NK = H / 128: lane t holds the 4 NK elements 128 k + 4 t + j of its row
template <typename H, int NK>
__global__ void __launch_bounds__(32 * kNormRowsPerBlock) rmsnorm_fwd_kernel(const H* __restrict__ x,
                                                                             const H* __restrict__ w, H* __restrict__ y,
                                                                             float* __restrict__ rs_out, int64_t rows,
                                                                             float factor, float eps) {
  const int64_t row = int64_t(blockIdx.x) * kNormRowsPerBlock + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const int64_t base = row * (NK * 128) + lane * 4;
  uint2 xv[NK];
#pragma unroll
  for (int k = 0; k < NK; ++k) xv[k] = *reinterpret_cast<const uint2*>(x + base + k * 128);
  float a[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
  for (int k = 0; k < NK; ++k) {
    float f[4];
    unpack4<H>(xv[k], f);
#pragma unroll
    for (int j = 0; j < 4; ++j) a[j] = __fadd_rn(a[j], __fmul_rn(f[j], f[j]));
  }
  const float rs = rsqrtf(__fadd_rn(__fmul_rn(warp_row_sum(a), factor), eps));
#pragma unroll
  for (int k = 0; k < NK; ++k) {
    float f[4], wf[4], o[4];
    unpack4<H>(xv[k], f);
    unpack4<H>(*reinterpret_cast<const uint2*>(w + lane * 4 + k * 128), wf);
#pragma unroll
    for (int j = 0; j < 4; ++j) o[j] = __fmul_rn(wf[j], rnd<H>(__fmul_rn(f[j], rs)));
    *reinterpret_cast<uint2*>(y + base + k * 128) = pack4<H>(o);
  }
  if (lane == 0) rs_out[row] = rs;
}

// p (the per-element weight-gradient product) is written only when it is not null
template <typename H, int NK>
__global__ void __launch_bounds__(32 * kNormRowsPerBlock) rmsnorm_bwd_kernel(const H* __restrict__ dy,
                                                                             const H* __restrict__ x,
                                                                             const H* __restrict__ w,
                                                                             const float* __restrict__ rs_in,
                                                                             H* __restrict__ dx, H* __restrict__ p,
                                                                             int64_t rows, float inv_h) {
  const int64_t row = int64_t(blockIdx.x) * kNormRowsPerBlock + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const int64_t base = row * (NK * 128) + lane * 4;
  uint2 xv[NK], dv[NK];
#pragma unroll
  for (int k = 0; k < NK; ++k) {
    xv[k] = *reinterpret_cast<const uint2*>(x + base + k * 128);
    dv[k] = *reinterpret_cast<const uint2*>(dy + base + k * 128);
  }
  const float rs = rs_in[row];
  float a[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
  for (int k = 0; k < NK; ++k) {
    float f[4], d[4], wf[4], dh[4];
    unpack4<H>(xv[k], f);
    unpack4<H>(dv[k], d);
    unpack4<H>(*reinterpret_cast<const uint2*>(w + lane * 4 + k * 128), wf);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      dh[j] = rnd<H>(__fmul_rn(d[j], wf[j]));
      a[j] = __fadd_rn(a[j], __fmul_rn(dh[j], f[j]));
    }
    if (p != nullptr) {
      float pf[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) pf[j] = __fmul_rn(d[j], rnd<H>(__fmul_rn(f[j], rs)));
      *reinterpret_cast<uint2*>(p + base + k * 128) = pack4<H>(pf);
    }
    dv[k] = pack4<H>(dh);   // dh is a 16-bit value: from here on dv holds it instead of dy
  }
  const float gv = __fmul_rn(__fmul_rn(warp_row_sum(a), -0.5f), __fmul_rn(__fmul_rn(rs, rs), rs));
  const float d2 = __fmul_rn(gv, inv_h);
#pragma unroll
  for (int k = 0; k < NK; ++k) {
    float f[4], dh[4], o[4];
    unpack4<H>(xv[k], f);
    unpack4<H>(dv[k], dh);
#pragma unroll
    for (int j = 0; j < 4; ++j) o[j] = __fadd_rn(__fmul_rn(dh[j], rs), __fmul_rn(d2, __fmul_rn(f[j], 2.0f)));
    *reinterpret_cast<uint2*>(dx + base + k * 128) = pack4<H>(o);
  }
}

// ---- causal-LM cross-entropy (HF ForCausalLMLoss: F.cross_entropy(logits.float(), labels)) --------------------------
//
// Eager upcasts the (N, V) logits to fp32 and runs torch's log_softmax, nll_loss and their backwards over fp32 copies.
// The kernels below read the 16-bit logits directly (the upcast is exact) and reproduce torch's fp32 results bit for bit.
// Per row (x = f32(logits[i]), t = target, v = the NLL gradient of the row: -grad_loss / total_weight, or +0 if ignored):
//   forward   m = max_j x_j,  s = sum_j expf(x_j - m),  ls = logf(s),  logp_t = (x_t - m) - ls
//   backward  g_j = r16(fma(expf((x_j - m) - ls), -(0 + v), j == t ? v : +0))
// torch's cunn_SoftMaxForward<ILP = 4> with its LogSoftMaxForwardEpilogue (ATen/native/cuda/SoftMax.cu) does the forward
// sums; for fp32 rows of 16384 <= V <= 32768 it runs with one 1024-thread block per row (smaller rows take its warp,
// register or shared-memory variants, which sum in other orders).  Its order, which ce_fwd_kernel copies:
//   * thread t folds the float4 groups t + 1024 k (k < V / 4096) lane by lane, then the scalars V - V % 4096 + t + 1024 m;
//   * m: fmaxf per thread from -FLT_MAX, then the block tree below; the order does not change a max;
//   * s: from 0, s = s + expf(x - m), where nvcc fuses the last product of expf (2^i * ex2(f)) and the add into one FFMA,
//     as in torch's build;
//   * block tree: shfl_down 16, 8, 4, 2, 1 in each warp, warp totals through shared memory, the same tree in warp 0.
// The NLL reduction over the rows is torch's own (nll_loss of the gathered (N, 1) logp_t, see llama_glue.py): its order
// depends on N only.  In the backward torch's row sum of the NLL gradient is 0 + v (one non-zero entry; -0 becomes +0),
// and its LogSoftMaxBackwardEpilogue, grad - expf(logp) * sum, compiles to a rounded expf and one FFMA: the __fmaf_rn
// below.  The fp32 gradient is rounded to the 16-bit type as the backward of `.float()` does.  No --use_fast_math: expf
// and logf are the libdevice ones torch calls.

constexpr int kCeThreads = 1024;
constexpr int kCeMaxVocab = 32768;
constexpr int kCeMaxVec = kCeMaxVocab / (4 * kCeThreads);   // float4 groups per thread
constexpr int kCeMaxTail = 4;                                // scalars per thread from the V % 4096 tail

// torch's cuda_utils::BlockReduce followed by blockReduceWarp's broadcast of thread 0's value
template <typename Op>
__device__ __forceinline__ float ce_block_reduce(float v, float* smem, Op op, float identity) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = op(v, __shfl_down_sync(0xffffffffu, v, o));
  __syncthreads();   // smem is reused by the next reduction
  if (lane == 0) smem[warp] = v;
  __syncthreads();
  if (warp == 0) {
    v = threadIdx.x < kCeThreads / 32 ? smem[lane] : identity;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = op(v, __shfl_down_sync(0xffffffffu, v, o));
  }
  if (threadIdx.x == 0) smem[0] = v;
  __syncthreads();
  return smem[0];
}

// one block per row, the row held in registers (at most 32 values per thread); writes the row's max, logf(sum) and
// logp at the target (0 when the target is outside [0, V): ignored rows, which read nothing more)
template <typename H>
__global__ void __launch_bounds__(kCeThreads) ce_fwd_kernel(const H* __restrict__ logits, const int64_t* __restrict__ target,
                                                           float* __restrict__ row_max, float* __restrict__ row_logsum,
                                                           float* __restrict__ logp_t, int V) {
  __shared__ float smem[kCeThreads / 32];
  const int t = threadIdx.x;
  const H* x = logits + int64_t(blockIdx.x) * V;
  const int nvec = V / (4 * kCeThreads);
  const int tail = nvec * 4 * kCeThreads;
  uint2 xv[kCeMaxVec];
  float xs[kCeMaxTail] = {};
#pragma unroll
  for (int k = 0; k < kCeMaxVec; ++k)
    if (k < nvec) xv[k] = *reinterpret_cast<const uint2*>(x + 4 * (t + k * kCeThreads));
#pragma unroll
  for (int m = 0; m < kCeMaxTail; ++m)
    if (tail + t + m * kCeThreads < V) xs[m] = Cvt<H>::to_f(x[tail + t + m * kCeThreads]);

  float mx = -FLT_MAX;
#pragma unroll
  for (int k = 0; k < kCeMaxVec; ++k)
    if (k < nvec) {
      float f[4];
      unpack4<H>(xv[k], f);
#pragma unroll
      for (int j = 0; j < 4; ++j) mx = fmaxf(mx, f[j]);
    }
#pragma unroll
  for (int m = 0; m < kCeMaxTail; ++m)
    if (tail + t + m * kCeThreads < V) mx = fmaxf(mx, xs[m]);
  mx = ce_block_reduce(mx, smem, [](float a, float b) { return a < b ? b : a; }, -FLT_MAX);

  float s = 0.0f;
#pragma unroll
  for (int k = 0; k < kCeMaxVec; ++k)
    if (k < nvec) {
      float f[4];
      unpack4<H>(xv[k], f);
#pragma unroll
      for (int j = 0; j < 4; ++j) s = s + expf(f[j] - mx);
    }
#pragma unroll
  for (int m = 0; m < kCeMaxTail; ++m)
    if (tail + t + m * kCeThreads < V) s = s + expf(xs[m] - mx);
  s = ce_block_reduce(s, smem, [](float a, float b) { return a + b; }, 0.0f);

  if (t == 0) {
    const float ls = logf(s);
    const int64_t tg = target[blockIdx.x];
    row_max[blockIdx.x] = mx;
    row_logsum[blockIdx.x] = ls;
    logp_t[blockIdx.x] = (tg >= 0 && tg < V) ? (Cvt<H>::to_f(x[tg]) - mx) - ls : 0.0f;
  }
}

constexpr int kCeBwdThreads = 256;   // 8 elements (16 bytes) per thread; a row takes ceil(V / 2048) blocks

template <typename H>
__global__ void __launch_bounds__(kCeBwdThreads) ce_bwd_kernel(const H* __restrict__ logits,
                                                              const float* __restrict__ row_max,
                                                              const float* __restrict__ row_logsum,
                                                              const int64_t* __restrict__ target,
                                                              const float* __restrict__ dlogp_t, H* __restrict__ grad, int V,
                                                              int blocks_per_row) {
  const int row = blockIdx.x / blocks_per_row;
  const int c = (blockIdx.x - row * blocks_per_row) * kCeBwdThreads + threadIdx.x;
  if (c * 8 >= V) return;
  const float mx = row_max[row], ls = row_logsum[row], v = dlogp_t[row];
  const float sum = 0.0f + v;
  const int64_t tg = target[row];
  const int64_t off = int64_t(row) * V + c * 8;
  float f[8];
  load8<H>(logits + off, f);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float go = (c * 8 + j == tg) ? v : 0.0f;
    f[j] = __fmaf_rn(expf((f[j] - mx) - ls), -sum, go);
  }
  store8<H>(grad + off, f);
}

int ce_check(const char* fn, int64_t rows, int vocab, int dtype) {
  SOWB_REQUIRE(dtype == SOWB_BF16 || dtype == SOWB_F16, "%s: dtype %d unsupported (bf16 / fp16)", fn, dtype);
  SOWB_REQUIRE(rows >= 0, "%s: negative row count", fn);
  // below 16384 torch's log_softmax reduces in another order; above 32768 a row does not fit the registers
  SOWB_REQUIRE(vocab >= 16384 && vocab <= kCeMaxVocab && vocab % 8 == 0,
               "%s: vocabulary %d unsupported (a multiple of 8 in [16384, %d])", fn, vocab, kCeMaxVocab);
  SOWB_REQUIRE(rows < (int64_t(1) << 31) / ((vocab + 8 * kCeBwdThreads - 1) / (8 * kCeBwdThreads)), "%s: too many rows",
               fn);
  return SOWB_OK;
}

// calls f(std::integral_constant<int, H / 128>{}) for the widths that have kernels; false for any other width
template <typename F>
bool with_norm_width(int width, F&& f) {
  switch (width) {
    case 128: f(std::integral_constant<int, 1>{}); return true;
    case 256: f(std::integral_constant<int, 2>{}); return true;
    case 512: f(std::integral_constant<int, 4>{}); return true;
    case 768: f(std::integral_constant<int, 6>{}); return true;
    case 1024: f(std::integral_constant<int, 8>{}); return true;
    case 2048: f(std::integral_constant<int, 16>{}); return true;
    case 3072: f(std::integral_constant<int, 24>{}); return true;
    case 4096: f(std::integral_constant<int, 32>{}); return true;
    default: return false;
  }
}

int rmsnorm_check(const char* fn, int64_t rows, int width, int dtype) {
  SOWB_REQUIRE(dtype == SOWB_BF16 || dtype == SOWB_F16, "%s: dtype %d unsupported (bf16 / fp16)", fn, dtype);
  SOWB_REQUIRE(rows >= 0, "%s: negative row count", fn);
  SOWB_REQUIRE(with_norm_width(width, [](auto) {}),
               "%s: width %d has no kernel (128, 256, 512, 768, 1024, 2048, 3072, 4096)", fn, width);
  // below 16 rows torch's reduction uses wider blocks and another summation order (one row is the same for H == 128)
  SOWB_REQUIRE(rows == 0 || rows >= 16 || width == 128, "%s: %lld rows: at least 16 are needed for width %d", fn,
               static_cast<long long>(rows), width);
  SOWB_REQUIRE(rows / kNormRowsPerBlock < (int64_t(1) << 31) - 1, "%s: too many rows", fn);
  return SOWB_OK;
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

int rope_launch(const char* fn, bool backward, const void* q, const void* k, const void* cos, const void* sin, void* q_out,
                void* k_out, int B, int S, int Hq, int Hk, int D, int64_t q_sb, int64_t q_sh, int64_t q_ss, int64_t k_sb,
                int64_t k_sh, int64_t k_ss, int64_t cs_sb, int dtype, void* stream_) {
  SOWB_REQUIRE(dtype == SOWB_BF16 || dtype == SOWB_F16, "%s: dtype %d unsupported (bf16 / fp16)", fn, dtype);
  SOWB_REQUIRE(q && k && cos && sin && q_out && k_out, "%s: null pointer", fn);
  SOWB_REQUIRE(aligned16(q) && aligned16(k) && aligned16(cos) && aligned16(sin) && aligned16(q_out) && aligned16(k_out),
               "%s: pointers must be 16-byte aligned", fn);
  SOWB_REQUIRE(B >= 0 && S >= 0 && Hq >= 0 && Hk >= 0, "%s: negative size", fn);
  SOWB_REQUIRE(D > 0 && D % 16 == 0, "%s: head dim %d must be a positive multiple of 16", fn, D);
  SOWB_REQUIRE(q_sb % 8 == 0 && q_sh % 8 == 0 && q_ss % 8 == 0 && k_sb % 8 == 0 && k_sh % 8 == 0 && k_ss % 8 == 0 &&
                   cs_sb % 8 == 0 && q_sb >= 0 && q_sh >= 0 && q_ss >= 0 && k_sb >= 0 && k_sh >= 0 && k_ss >= 0 && cs_sb >= 0,
               "%s: strides must be non-negative multiples of 8 elements", fn);
  RopeArgs a;
  a.t[0] = {q, q_out, q_sb, q_sh, q_ss, Hq, int64_t(B) * S * Hq * (D / 16)};
  a.t[1] = {k, k_out, k_sb, k_sh, k_ss, Hk, int64_t(B) * S * Hk * (D / 16)};
  a.cos = cos;
  a.sin = sin;
  a.cs_sb = cs_sb;
  a.S = S;
  a.D = D;
  const int64_t total = a.t[0].n + a.t[1].n;
  if (total == 0) return SOWB_OK;
  const int64_t blocks = (total + 255) / 256;
  SOWB_REQUIRE(blocks < (int64_t(1) << 31), "%s: tensors too large", fn);
  if (int rc = ensure_context_for(q)) return rc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (dtype == SOWB_BF16) {
    if (backward) rope_kernel<__nv_bfloat16, true><<<unsigned(blocks), 256, 0, stream>>>(a);
    else rope_kernel<__nv_bfloat16, false><<<unsigned(blocks), 256, 0, stream>>>(a);
  } else {
    if (backward) rope_kernel<__half, true><<<unsigned(blocks), 256, 0, stream>>>(a);
    else rope_kernel<__half, false><<<unsigned(blocks), 256, 0, stream>>>(a);
  }
  SOWB_CHECK_CUDA(cudaGetLastError());
  return SOWB_OK;
}

int swiglu_check(const char* fn, int64_t n, int dtype) {
  SOWB_REQUIRE(dtype == SOWB_BF16 || dtype == SOWB_F16, "%s: dtype %d unsupported (bf16 / fp16)", fn, dtype);
  SOWB_REQUIRE(n >= 0, "%s: negative element count", fn);
  SOWB_REQUIRE((n / 8 + 256) / 256 < (int64_t(1) << 31), "%s: tensors too large", fn);
  return SOWB_OK;
}

}  // namespace

}  // namespace sowb

using namespace sowb;

extern "C" {

int sow_rope_fwd(const void* q, const void* k, const void* cos, const void* sin, void* q_out, void* k_out, int B, int S, int Hq,
                 int Hk, int D, int64_t q_sb, int64_t q_sh, int64_t q_ss, int64_t k_sb, int64_t k_sh, int64_t k_ss,
                 int64_t cs_sb, int dtype, void* stream) {
  return rope_launch("sow_rope_fwd", false, q, k, cos, sin, q_out, k_out, B, S, Hq, Hk, D, q_sb, q_sh, q_ss, k_sb, k_sh, k_ss,
                     cs_sb, dtype, stream);
}

int sow_rope_bwd(const void* gq, const void* gk, const void* cos, const void* sin, void* dq, void* dk, int B, int S, int Hq,
                 int Hk, int D, int64_t gq_sb, int64_t gq_sh, int64_t gq_ss, int64_t gk_sb, int64_t gk_sh, int64_t gk_ss,
                 int64_t cs_sb, int dtype, void* stream) {
  return rope_launch("sow_rope_bwd", true, gq, gk, cos, sin, dq, dk, B, S, Hq, Hk, D, gq_sb, gq_sh, gq_ss, gk_sb, gk_sh, gk_ss,
                     cs_sb, dtype, stream);
}

int sow_swiglu_fwd(const void* gate, const void* up, void* h, int64_t n, int dtype, void* stream_) {
  if (int rc = swiglu_check("sow_swiglu_fwd", n, dtype)) return rc;
  SOWB_REQUIRE(gate && up && h, "sow_swiglu_fwd: null pointer");
  SOWB_REQUIRE(aligned16(gate) && aligned16(up) && aligned16(h), "sow_swiglu_fwd: pointers must be 16-byte aligned");
  if (n == 0) return SOWB_OK;
  if (int rc = ensure_context_for(gate)) return rc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const unsigned blocks = unsigned((n / 8 + (n % 8) + 255) / 256);
  if (dtype == SOWB_BF16)
    swiglu_fwd_kernel<__nv_bfloat16><<<blocks, 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(gate),
                                                                  static_cast<const __nv_bfloat16*>(up),
                                                                  static_cast<__nv_bfloat16*>(h), n);
  else
    swiglu_fwd_kernel<__half><<<blocks, 256, 0, stream>>>(static_cast<const __half*>(gate), static_cast<const __half*>(up),
                                                          static_cast<__half*>(h), n);
  SOWB_CHECK_CUDA(cudaGetLastError());
  return SOWB_OK;
}

int sow_swiglu_bwd(const void* dh, const void* gate, const void* up, void* dgate, void* dup, int64_t n, int dtype,
                   void* stream_) {
  if (int rc = swiglu_check("sow_swiglu_bwd", n, dtype)) return rc;
  SOWB_REQUIRE(dh && gate && up && dgate && dup, "sow_swiglu_bwd: null pointer");
  SOWB_REQUIRE(aligned16(dh) && aligned16(gate) && aligned16(up) && aligned16(dgate) && aligned16(dup),
               "sow_swiglu_bwd: pointers must be 16-byte aligned");
  if (n == 0) return SOWB_OK;
  if (int rc = ensure_context_for(gate)) return rc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const unsigned blocks = unsigned((n / 8 + (n % 8) + 255) / 256);
  if (dtype == SOWB_BF16)
    swiglu_bwd_kernel<__nv_bfloat16><<<blocks, 256, 0, stream>>>(
        static_cast<const __nv_bfloat16*>(dh), static_cast<const __nv_bfloat16*>(gate), static_cast<const __nv_bfloat16*>(up),
        static_cast<__nv_bfloat16*>(dgate), static_cast<__nv_bfloat16*>(dup), n);
  else
    swiglu_bwd_kernel<__half><<<blocks, 256, 0, stream>>>(static_cast<const __half*>(dh), static_cast<const __half*>(gate),
                                                          static_cast<const __half*>(up), static_cast<__half*>(dgate),
                                                          static_cast<__half*>(dup), n);
  SOWB_CHECK_CUDA(cudaGetLastError());
  return SOWB_OK;
}

int sow_rmsnorm_fwd(const void* x, const void* w, void* y, float* rs, int64_t rows, int width, float eps, int dtype,
                    void* stream_) {
  if (int rc = rmsnorm_check("sow_rmsnorm_fwd", rows, width, dtype)) return rc;
  SOWB_REQUIRE(x && w && y && rs, "sow_rmsnorm_fwd: null pointer");
  SOWB_REQUIRE(aligned16(x) && aligned16(w) && aligned16(y), "sow_rmsnorm_fwd: pointers must be 16-byte aligned");
  if (rows == 0) return SOWB_OK;
  if (int rc = ensure_context_for(x)) return rc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const unsigned blocks = unsigned((rows + kNormRowsPerBlock - 1) / kNormRowsPerBlock);
  const float factor = float(rows) / float(rows * width);   // torch's mean: float(outputs) / numel
  with_norm_width(width, [&](auto nk) {
    constexpr int NK = decltype(nk)::value;
    if (dtype == SOWB_BF16)
      rmsnorm_fwd_kernel<__nv_bfloat16, NK><<<blocks, 32 * kNormRowsPerBlock, 0, stream>>>(
          static_cast<const __nv_bfloat16*>(x), static_cast<const __nv_bfloat16*>(w), static_cast<__nv_bfloat16*>(y), rs,
          rows, factor, eps);
    else
      rmsnorm_fwd_kernel<__half, NK><<<blocks, 32 * kNormRowsPerBlock, 0, stream>>>(
          static_cast<const __half*>(x), static_cast<const __half*>(w), static_cast<__half*>(y), rs, rows, factor, eps);
  });
  SOWB_CHECK_CUDA(cudaGetLastError());
  return SOWB_OK;
}

int sow_rmsnorm_bwd(const void* dy, const void* x, const void* w, const float* rs, void* dx, void* p, int64_t rows,
                    int width, int dtype, void* stream_) {
  if (int rc = rmsnorm_check("sow_rmsnorm_bwd", rows, width, dtype)) return rc;
  SOWB_REQUIRE(dy && x && w && rs && dx, "sow_rmsnorm_bwd: null pointer");
  SOWB_REQUIRE(aligned16(dy) && aligned16(x) && aligned16(w) && aligned16(dx) && aligned16(p),
               "sow_rmsnorm_bwd: pointers must be 16-byte aligned");
  if (rows == 0) return SOWB_OK;
  if (int rc = ensure_context_for(x)) return rc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const unsigned blocks = unsigned((rows + kNormRowsPerBlock - 1) / kNormRowsPerBlock);
  const float inv_h = 1.0f / float(width);   // torch's division by a scalar: a product with its reciprocal
  with_norm_width(width, [&](auto nk) {
    constexpr int NK = decltype(nk)::value;
    if (dtype == SOWB_BF16)
      rmsnorm_bwd_kernel<__nv_bfloat16, NK><<<blocks, 32 * kNormRowsPerBlock, 0, stream>>>(
          static_cast<const __nv_bfloat16*>(dy), static_cast<const __nv_bfloat16*>(x),
          static_cast<const __nv_bfloat16*>(w), rs, static_cast<__nv_bfloat16*>(dx), static_cast<__nv_bfloat16*>(p), rows,
          inv_h);
    else
      rmsnorm_bwd_kernel<__half, NK><<<blocks, 32 * kNormRowsPerBlock, 0, stream>>>(
          static_cast<const __half*>(dy), static_cast<const __half*>(x), static_cast<const __half*>(w), rs,
          static_cast<__half*>(dx), static_cast<__half*>(p), rows, inv_h);
  });
  SOWB_CHECK_CUDA(cudaGetLastError());
  return SOWB_OK;
}

int sow_ce_fwd(const void* logits, const int64_t* target, float* row_max, float* row_logsum, float* logp_t, int64_t rows,
               int vocab, int dtype, void* stream_) {
  if (int rc = ce_check("sow_ce_fwd", rows, vocab, dtype)) return rc;
  SOWB_REQUIRE(logits && target && row_max && row_logsum && logp_t, "sow_ce_fwd: null pointer");
  SOWB_REQUIRE(aligned16(logits), "sow_ce_fwd: logits must be 16-byte aligned");
  if (rows == 0) return SOWB_OK;
  if (int rc = ensure_context_for(logits)) return rc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (dtype == SOWB_BF16)
    ce_fwd_kernel<__nv_bfloat16><<<unsigned(rows), kCeThreads, 0, stream>>>(
        static_cast<const __nv_bfloat16*>(logits), target, row_max, row_logsum, logp_t, vocab);
  else
    ce_fwd_kernel<__half><<<unsigned(rows), kCeThreads, 0, stream>>>(static_cast<const __half*>(logits), target, row_max,
                                                                     row_logsum, logp_t, vocab);
  SOWB_CHECK_CUDA(cudaGetLastError());
  return SOWB_OK;
}

int sow_ce_bwd(const void* logits, const float* row_max, const float* row_logsum, const int64_t* target,
               const float* dlogp_t, void* grad, int64_t rows, int vocab, int dtype, void* stream_) {
  if (int rc = ce_check("sow_ce_bwd", rows, vocab, dtype)) return rc;
  SOWB_REQUIRE(logits && row_max && row_logsum && target && dlogp_t && grad, "sow_ce_bwd: null pointer");
  SOWB_REQUIRE(aligned16(logits) && aligned16(grad), "sow_ce_bwd: logits and grad must be 16-byte aligned");
  if (rows == 0) return SOWB_OK;
  if (int rc = ensure_context_for(logits)) return rc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const int bpr = (vocab + 8 * kCeBwdThreads - 1) / (8 * kCeBwdThreads);
  const unsigned blocks = unsigned(rows * bpr);
  if (dtype == SOWB_BF16)
    ce_bwd_kernel<__nv_bfloat16><<<blocks, kCeBwdThreads, 0, stream>>>(
        static_cast<const __nv_bfloat16*>(logits), row_max, row_logsum, target, dlogp_t,
        static_cast<__nv_bfloat16*>(grad), vocab, bpr);
  else
    ce_bwd_kernel<__half><<<blocks, kCeBwdThreads, 0, stream>>>(static_cast<const __half*>(logits), row_max, row_logsum,
                                                                target, dlogp_t, static_cast<__half*>(grad), vocab, bpr);
  SOWB_CHECK_CUDA(cudaGetLastError());
  return SOWB_OK;
}

}  // extern "C"
