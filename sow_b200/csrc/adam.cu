// Multi-tensor fused Adam / AdamW: every tensor of a param group updated by ONE launch.
//
// Replaces torch.optim.AdamW over the factor + dense groups (scripts/simple_train.py:502-511), which in eager
// mode issues ~8 elementwise kernels per group chunk and, for bf16 parameters, rounds to bf16 after every one
// of them.  Here each element is read once (p, g, m, v), updated in fp32 registers and written once:
// 4 reads + 3 writes of the parameter dtype per element -> 14 B/element in bf16, the HBM floor for Adam.
// State stays per-parameter and by default in the parameter dtype, exactly where torch keeps it (sow_adam_multi_amp can keep
// fp32 moments for 16-bit parameters: 22 B/element), so
// scripts/utils/training_utils.py:257-277 (reset_optimizer, which REBINDS exp_avg / exp_avg_sq) keeps working:
// the host side re-resolves the pointers whenever they change.
#include "common.cuh"

#include <cuda_fp16.h>

#include <cmath>

namespace sowb {

struct AdamChunk {   // 40 bytes; the host passes an int64[n_chunks][5] table with exactly this layout
  void* p;
  const void* g;
  void* m;
  void* v;
  int64_t n;
};

struct AdamHyper {
  float lr, beta1, omb1, beta2, omb2, eps, decay_mul, weight_decay, step_size, inv_sqrt_bc2;
  int decoupled;
};

__device__ __forceinline__ void adam_update(float& p, float g, float& m, float& v, const AdamHyper& h) {
  if (h.decoupled) p *= h.decay_mul;
  else g = fmaf(h.weight_decay, p, g);
  m = fmaf(h.beta1, m, h.omb1 * g);
  v = fmaf(h.beta2, v, h.omb2 * g * g);
  const float denom = sqrtf(v) * h.inv_sqrt_bc2 + h.eps;
  p -= h.step_size * (m / denom);
}

// CUDA-graph friendly step counter: the bias corrections are derived ON THE DEVICE from a counter that the launch
// sequence itself advances, so a captured optimizer step replays with the right corrections (host-computed ones would
// be frozen into the graph).  A step skipped for found_inf does not advance it (torch's fused AdamW subtracts found_inf
// from the step it incremented).
__global__ void adam_step_inc_kernel(float* step, const float* found_inf) {
  if (found_inf == nullptr || *found_inf == 0.0f) *step += 1.0f;
}

__device__ __forceinline__ AdamHyper with_device_step(AdamHyper h, const float* __restrict__ step_dev) {
  if (step_dev != nullptr) {
    const double t = static_cast<double>(*step_dev);
    const double bc1 = 1.0 - pow(static_cast<double>(h.beta1), t);
    const double bc2 = 1.0 - pow(static_cast<double>(h.beta2), t);
    h.step_size = static_cast<float>(static_cast<double>(h.lr) / bc1);
    h.inv_sqrt_bc2 = static_cast<float>(1.0 / sqrt(bc2));
  }
  return h;
}

// 16-bit parameter types (bf16, fp16): conversions of one element and of a packed pair, round to nearest even
template <typename H>
struct Half16;
template <>
struct Half16<__nv_bfloat16> {
  using H2 = __nv_bfloat162;
  static __device__ __forceinline__ float2 to_f2(H2 v) { return __bfloat1622float2(v); }
  static __device__ __forceinline__ H2 from_f2(float a, float b) { return __floats2bfloat162_rn(a, b); }
  static __device__ __forceinline__ float to_f(__nv_bfloat16 v) { return __bfloat162float(v); }
  static __device__ __forceinline__ __nv_bfloat16 from_f(float v) { return __float2bfloat16(v); }
};
template <>
struct Half16<__half> {
  using H2 = __half2;
  static __device__ __forceinline__ float2 to_f2(H2 v) { return __half22float2(v); }
  static __device__ __forceinline__ H2 from_f2(float a, float b) { return __floats2half2_rn(a, b); }
  static __device__ __forceinline__ float to_f(__half v) { return __half2float(v); }
  static __device__ __forceinline__ __half from_f(float v) { return __float2half_rn(v); }
};

// Moments are either of the parameter type H or fp32 (state_dtype): element conversions for both (Moment<float, float>
// also serves the fp32 kernel's gradients)
template <typename H, typename S>
struct Moment {
  static __device__ __forceinline__ float to_f(S v) { return Half16<H>::to_f(v); }
  static __device__ __forceinline__ S from_f(float v) { return Half16<H>::from_f(v); }
};
template <typename H>
struct Moment<H, float> {
  static __device__ __forceinline__ float to_f(float v) { return v; }
  static __device__ __forceinline__ float from_f(float v) { return v; }
};

// Gradient element i as the update reads it.  kAmp with a loss scale: g / scale (IEEE division, as torch's fused Adam
// divides), and the unscaled value is written back to the gradient, rounded to its type, as torch._fused_adamw_ does.
template <bool kAmp, typename G, typename C>
__device__ __forceinline__ float grad_in(G* g, int64_t i, const float* scale) {
  float x = C::to_f(g[i]);
  if constexpr (kAmp) {
    if (scale != nullptr) {
      x = x / *scale;
      g[i] = C::from_f(x);
    }
  }
  return x;
}
// A packed pair of 16-bit gradients, unscaled in place as grad_in does for one element
template <bool kAmp, typename C>
__device__ __forceinline__ void unscale2(float2& gf, typename C::H2& g2, const float* scale) {
  if constexpr (kAmp) {
    if (scale != nullptr) {
      gf.x = gf.x / *scale;
      gf.y = gf.y / *scale;
      g2 = C::from_f2(gf.x, gf.y);
    }
  }
}

// kClip (always with kAmp): the gradient is unscaled (when a scale is given) and rounded to its type, as unscale_ leaves
// it, then multiplied by the fp32 clip coefficient in fp32 and rounded once more to its type.  That value
// is the update's gradient and is written back.  __fmul_rn: the product is rounded on its own, never contracted into an FMA.
template <typename G, typename C>
__device__ __forceinline__ float grad_clip_in(G* g, int64_t i, const float* scale, float coef) {
  float x = C::to_f(g[i]);
  if (scale != nullptr) x = C::to_f(C::from_f(x / *scale));
  const G y = C::from_f(__fmul_rn(x, coef));
  g[i] = y;
  return C::to_f(y);
}
template <typename C>
__device__ __forceinline__ void clip2(float2& gf, typename C::H2& g2, const float* scale, float coef) {
  if (scale != nullptr) gf = C::to_f2(C::from_f2(gf.x / *scale, gf.y / *scale));
  g2 = C::from_f2(__fmul_rn(gf.x, coef), __fmul_rn(gf.y, coef));
  gf = C::to_f2(g2);
}
// The 16-bit kernels' packed-pair gradient: clipped (kClip), unscaled (kAmp) or as read
template <bool kAmp, bool kClip, typename C>
__device__ __forceinline__ void grad_in2(float2& gf, typename C::H2& g2, const float* scale, float coef) {
  if constexpr (kClip) clip2<C>(gf, g2, scale, coef);
  else unscale2<kAmp, C>(gf, g2, scale);
}

// kAmp: the launch carries GradScaler's two device scalars.  found_inf != 0 -> the block returns before touching anything
// (no decay, p / m / v / g keep every bit); grad_scale != NULL -> gradients are unscaled in the kernel.  Without kAmp the
// pointers are never read, so these instantiations are the plain Adam kernels.
template <bool kAmp>
__device__ __forceinline__ bool amp_skip(const float* __restrict__ found_inf) {
  if constexpr (kAmp) return found_inf != nullptr && *found_inf != 0.0f;
  return false;
}

// Clip coefficient of a kClip launch (a device scalar written by grad_norm_finalize_kernel); never read otherwise
template <bool kClip>
__device__ __forceinline__ float clip_coef_of(const float* __restrict__ clip_coef) {
  if constexpr (kClip) return *clip_coef;
  return 1.0f;
}

// p, g of type H (bf16 or fp16), m, v of type S (H or fp32): 16-byte vector accesses (8 elements of p and g, one or two
// 16-byte accesses of m and v) when all four are 16-byte aligned
template <typename H, typename S, bool kAmp, bool kClip = false>
__global__ void __launch_bounds__(256)
adam_multi_16bit_kernel(const AdamChunk* __restrict__ chunks, const AdamHyper h0, const float* __restrict__ step_dev,
                        const float* __restrict__ grad_scale, const float* __restrict__ found_inf,
                        const float* __restrict__ clip_coef = nullptr) {
  static_assert(kAmp || !kClip, "clipping is launched through the AMP entry point");
  using C = Half16<H>;
  using M = Moment<H, S>;
  using H2 = typename C::H2;
  if (amp_skip<kAmp>(found_inf)) return;
  const float coef = clip_coef_of<kClip>(clip_coef);
  const AdamHyper h = with_device_step(h0, step_dev);
  const AdamChunk c = chunks[blockIdx.x];
  H* p = static_cast<H*>(c.p);
  H* g = static_cast<H*>(const_cast<void*>(c.g));
  S* m = static_cast<S*>(c.m);
  S* v = static_cast<S*>(c.v);
  const bool aligned = ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) |
                         reinterpret_cast<uintptr_t>(m) | reinterpret_cast<uintptr_t>(v)) & 15) == 0;
  int64_t done = 0;
  if (aligned) {
    const int64_t nvec = c.n / 8;
    for (int64_t i = threadIdx.x; i < nvec; i += blockDim.x) {
      uint4 pp = reinterpret_cast<uint4*>(p)[i];
      uint4 gg = reinterpret_cast<const uint4*>(g)[i];
      H2* p2 = reinterpret_cast<H2*>(&pp);
      H2* g2 = reinterpret_cast<H2*>(&gg);
      if constexpr (std::is_same<S, H>::value) {
        uint4 mm = reinterpret_cast<uint4*>(m)[i];
        uint4 vv = reinterpret_cast<uint4*>(v)[i];
        H2* m2 = reinterpret_cast<H2*>(&mm);
        H2* v2 = reinterpret_cast<H2*>(&vv);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float2 pf = C::to_f2(p2[j]), gf = C::to_f2(g2[j]);
          float2 mf = C::to_f2(m2[j]), vf = C::to_f2(v2[j]);
          grad_in2<kAmp, kClip, C>(gf, g2[j], grad_scale, coef);
          adam_update(pf.x, gf.x, mf.x, vf.x, h);
          adam_update(pf.y, gf.y, mf.y, vf.y, h);
          p2[j] = C::from_f2(pf.x, pf.y);
          m2[j] = C::from_f2(mf.x, mf.y);
          v2[j] = C::from_f2(vf.x, vf.y);
        }
        reinterpret_cast<uint4*>(p)[i] = pp;
        reinterpret_cast<uint4*>(m)[i] = mm;
        reinterpret_cast<uint4*>(v)[i] = vv;
      } else {
        float4 mm[2] = {reinterpret_cast<float4*>(m)[2 * i], reinterpret_cast<float4*>(m)[2 * i + 1]};
        float4 vv[2] = {reinterpret_cast<float4*>(v)[2 * i], reinterpret_cast<float4*>(v)[2 * i + 1]};
        float* mf = reinterpret_cast<float*>(mm);
        float* vf = reinterpret_cast<float*>(vv);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float2 pf = C::to_f2(p2[j]), gf = C::to_f2(g2[j]);
          grad_in2<kAmp, kClip, C>(gf, g2[j], grad_scale, coef);
          adam_update(pf.x, gf.x, mf[2 * j], vf[2 * j], h);
          adam_update(pf.y, gf.y, mf[2 * j + 1], vf[2 * j + 1], h);
          p2[j] = C::from_f2(pf.x, pf.y);
        }
        reinterpret_cast<uint4*>(p)[i] = pp;
        reinterpret_cast<float4*>(m)[2 * i] = mm[0];
        reinterpret_cast<float4*>(m)[2 * i + 1] = mm[1];
        reinterpret_cast<float4*>(v)[2 * i] = vv[0];
        reinterpret_cast<float4*>(v)[2 * i + 1] = vv[1];
      }
      if constexpr (kClip) {
        reinterpret_cast<uint4*>(g)[i] = gg;
      } else if constexpr (kAmp) {
        if (grad_scale != nullptr) reinterpret_cast<uint4*>(g)[i] = gg;
      }
    }
    done = nvec * 8;
  }
  for (int64_t i = done + threadIdx.x; i < c.n; i += blockDim.x) {
    float pf = C::to_f(p[i]), mf = M::to_f(m[i]), vf = M::to_f(v[i]);
    float gi;
    if constexpr (kClip) gi = grad_clip_in<H, C>(g, i, grad_scale, coef);
    else gi = grad_in<kAmp, H, C>(g, i, grad_scale);
    adam_update(pf, gi, mf, vf, h);
    p[i] = C::from_f(pf);
    m[i] = M::from_f(mf);
    v[i] = M::from_f(vf);
  }
}

template <bool kAmp, bool kClip = false>
__global__ void __launch_bounds__(256)
adam_multi_f32_kernel(const AdamChunk* __restrict__ chunks, const AdamHyper h0, const float* __restrict__ step_dev,
                      const float* __restrict__ grad_scale, const float* __restrict__ found_inf,
                      const float* __restrict__ clip_coef = nullptr) {
  static_assert(kAmp || !kClip, "clipping is launched through the AMP entry point");
  if (amp_skip<kAmp>(found_inf)) return;
  const float coef = clip_coef_of<kClip>(clip_coef);
  const AdamHyper h = with_device_step(h0, step_dev);
  const AdamChunk c = chunks[blockIdx.x];
  float* p = static_cast<float*>(c.p);
  float* g = static_cast<float*>(const_cast<void*>(c.g));
  float* m = static_cast<float*>(c.m);
  float* v = static_cast<float*>(c.v);
  const bool aligned = ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) |
                         reinterpret_cast<uintptr_t>(m) | reinterpret_cast<uintptr_t>(v)) & 15) == 0;
  int64_t done = 0;
  if (aligned) {
    const int64_t nvec = c.n / 4;
    for (int64_t i = threadIdx.x; i < nvec; i += blockDim.x) {
      float4 pp = reinterpret_cast<float4*>(p)[i];
      float4 gg = reinterpret_cast<const float4*>(g)[i];
      if constexpr (kClip) {
        if (grad_scale != nullptr) {
          const float s = *grad_scale;
          gg.x = gg.x / s;
          gg.y = gg.y / s;
          gg.z = gg.z / s;
          gg.w = gg.w / s;
        }
        gg.x = __fmul_rn(gg.x, coef);
        gg.y = __fmul_rn(gg.y, coef);
        gg.z = __fmul_rn(gg.z, coef);
        gg.w = __fmul_rn(gg.w, coef);
        reinterpret_cast<float4*>(g)[i] = gg;
      } else if constexpr (kAmp) {
        if (grad_scale != nullptr) {
          const float s = *grad_scale;
          gg.x = gg.x / s;
          gg.y = gg.y / s;
          gg.z = gg.z / s;
          gg.w = gg.w / s;
          reinterpret_cast<float4*>(g)[i] = gg;
        }
      }
      float4 mm = reinterpret_cast<float4*>(m)[i];
      float4 vv = reinterpret_cast<float4*>(v)[i];
      adam_update(pp.x, gg.x, mm.x, vv.x, h);
      adam_update(pp.y, gg.y, mm.y, vv.y, h);
      adam_update(pp.z, gg.z, mm.z, vv.z, h);
      adam_update(pp.w, gg.w, mm.w, vv.w, h);
      reinterpret_cast<float4*>(p)[i] = pp;
      reinterpret_cast<float4*>(m)[i] = mm;
      reinterpret_cast<float4*>(v)[i] = vv;
    }
    done = nvec * 4;
  }
  for (int64_t i = done + threadIdx.x; i < c.n; i += blockDim.x) {
    if constexpr (kClip)
      adam_update(p[i], grad_clip_in<float, Moment<float, float>>(g, i, grad_scale, coef), m[i], v[i], h);
    else
      adam_update(p[i], grad_in<kAmp, float, Moment<float, float>>(g, i, grad_scale), m[i], v[i], h);
  }
}

// ---- global gradient norm for clipping (torch.nn.utils.clip_grad_norm_, norm type 2) ----------------------------------
// Pass 1 runs over an Adam chunk table and reads only g and n of each row: one 256-thread block per row squares each
// element and accumulates in fp32 (n / 256 <= sow_adam_chunk_elems() / 256 sequential FMAs per thread), reduces in a fixed
// shuffle order and writes one fp32 partial.  kAmp with a scale: the element is round_G(g / scale), exactly the value the
// Adam kernel's unscale writes back, so the norm is that of the gradients GradScaler.unscale_ would have produced.
// Pass 2 (one block) sums the partials in a fixed order in fp64.  No atomics: the same inputs give the same bits, eagerly
// and under graph replay.
template <typename T>
__device__ __forceinline__ T block_sum_256(T x) {
  __shared__ T warp_sums[8];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_down_sync(0xffffffffu, x, o);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) warp_sums[warp] = x;
  __syncthreads();
  x = lane < 8 ? warp_sums[lane] : T(0);
  if (warp == 0) {
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) x += __shfl_down_sync(0xffffffffu, x, o);
  }
  return x;   // the sum in thread 0
}

template <typename G, bool kAmp>
__device__ __forceinline__ float norm_elem(G v, float scale) {
  using C = Moment<G, G>;
  float x = C::to_f(v);
  if constexpr (kAmp) x = C::to_f(C::from_f(x / scale));
  return x;
}

template <typename G, bool kAmp>
__global__ void __launch_bounds__(256)
grad_norm_partial_kernel(const AdamChunk* __restrict__ chunks, const float* __restrict__ grad_scale,
                         float* __restrict__ partials) {
  constexpr int kVec = 16 / sizeof(G);
  const AdamChunk c = chunks[blockIdx.x];
  const G* g = static_cast<const G*>(c.g);
  const float scale = kAmp ? *grad_scale : 1.0f;
  float acc = 0.0f;
  int64_t done = 0;
  if ((reinterpret_cast<uintptr_t>(g) & 15) == 0) {
    const int64_t nvec = c.n / kVec;
#pragma unroll 4
    for (int64_t i = threadIdx.x; i < nvec; i += blockDim.x) {
      const uint4 raw = reinterpret_cast<const uint4*>(g)[i];
      const G* e = reinterpret_cast<const G*>(&raw);
#pragma unroll
      for (int j = 0; j < kVec; ++j) {
        const float x = norm_elem<G, kAmp>(e[j], scale);
        acc = fmaf(x, x, acc);
      }
    }
    done = nvec * kVec;
  }
  for (int64_t i = done + threadIdx.x; i < c.n; i += blockDim.x) {
    const float x = norm_elem<G, kAmp>(g[i], scale);
    acc = fmaf(x, x, acc);
  }
  acc = block_sum_256(acc);
  if (threadIdx.x == 0) partials[blockIdx.x] = acc;
}

// total_norm = float(sqrt(sum of partials)), then the clip coefficient as torch's _clip_grads_with_norm_ computes it on an
// fp32 CUDA tensor: `max_norm / (total_norm + 1e-6)` is Tensor.__rtruediv__, i.e. reciprocal() * max_norm, two roundings,
// then clamp(max=1), which propagates NaN.  An inf norm gives 0, a NaN norm NaN (error_if_nonfinite=False).
__global__ void __launch_bounds__(256)
grad_norm_finalize_kernel(const float* __restrict__ partials, int n_partials, float max_norm, float* __restrict__ total_norm,
                          float* __restrict__ clip_coef) {
  double acc = 0.0;
  for (int i = threadIdx.x; i < n_partials; i += blockDim.x) acc += static_cast<double>(partials[i]);
  acc = block_sum_256(acc);
  if (threadIdx.x == 0) {
    const float norm = static_cast<float>(sqrt(acc));
    const float r = __fdiv_rn(1.0f, __fadd_rn(norm, 1e-6f));
    const float coef = __fmul_rn(r, max_norm);
    *total_norm = norm;
    *clip_coef = isnan(coef) ? coef : fminf(coef, 1.0f);
  }
}

}  // namespace sowb

using namespace sowb;

static int elem_bytes(int dtype) { return dtype == SOWB_F32 ? 4 : 2; }

template <bool kAmp, typename H>
static void launch_16bit(int n_chunks, const AdamChunk* ch, const AdamHyper& h, const float* step_dev,
                         const float* grad_scale, const float* found_inf, int state_dtype, cudaStream_t stream) {
  if (state_dtype == SOWB_F32)
    adam_multi_16bit_kernel<H, float, true><<<n_chunks, 256, 0, stream>>>(ch, h, step_dev, grad_scale, found_inf);
  else
    adam_multi_16bit_kernel<H, H, kAmp><<<n_chunks, 256, 0, stream>>>(ch, h, step_dev, grad_scale, found_inf);
}

template <typename H>
static void launch_16bit_clip(int n_chunks, const AdamChunk* ch, const AdamHyper& h, const float* step_dev,
                              const float* grad_scale, const float* found_inf, const float* clip_coef, int state_dtype,
                              cudaStream_t stream) {
  if (state_dtype == SOWB_F32)
    adam_multi_16bit_kernel<H, float, true, true>
        <<<n_chunks, 256, 0, stream>>>(ch, h, step_dev, grad_scale, found_inf, clip_coef);
  else
    adam_multi_16bit_kernel<H, H, true, true>
        <<<n_chunks, 256, 0, stream>>>(ch, h, step_dev, grad_scale, found_inf, clip_coef);
}

template <typename G>
static void launch_norm_partials(int n_chunks, const AdamChunk* ch, const float* grad_scale, float* partials,
                                 cudaStream_t stream) {
  if (grad_scale != nullptr)
    grad_norm_partial_kernel<G, true><<<n_chunks, 256, 0, stream>>>(ch, grad_scale, partials);
  else
    grad_norm_partial_kernel<G, false><<<n_chunks, 256, 0, stream>>>(ch, nullptr, partials);
}

extern "C" {

int sow_adam_chunk_elems(void) { return 32768; }

int sow_adam_multi_ex(const void* chunks_dev, int n_chunks, int64_t total_elems, double lr, double beta1, double beta2,
                      double eps, double weight_decay, double bias_correction1, double bias_correction2, int decoupled,
                      int dtype, void* stream_);

int sow_adam_multi(const void* chunks_dev, int n_chunks, double lr, double beta1, double beta2, double eps,
                   double weight_decay, double bias_correction1, double bias_correction2, int decoupled, int dtype,
                   void* stream_) {
  return sow_adam_multi_ex(chunks_dev, n_chunks, 0, lr, beta1, beta2, eps, weight_decay, bias_correction1,
                           bias_correction2, decoupled, dtype, stream_);
}

static int adam_launch(const void* chunks_dev, int n_chunks, int64_t total_elems, double lr, double beta1, double beta2,
                       double eps, double weight_decay, double bias_correction1, double bias_correction2, float* step_dev,
                       const float* grad_scale, const float* found_inf, const float* clip_coef, bool amp, int decoupled,
                       int dtype, int state_dtype, void* stream_);

int sow_adam_multi_ex(const void* chunks_dev, int n_chunks, int64_t total_elems, double lr, double beta1, double beta2, double eps,
                      double weight_decay, double bias_correction1, double bias_correction2, int decoupled,
                      int dtype, void* stream_) {
  SOWB_REQUIRE(bias_correction1 > 0.0 && bias_correction2 > 0.0, "sow_adam_multi: bias corrections must be positive");
  return adam_launch(chunks_dev, n_chunks, total_elems, lr, beta1, beta2, eps, weight_decay, bias_correction1,
                     bias_correction2, nullptr, nullptr, nullptr, nullptr, false, decoupled, dtype, dtype, stream_);
}

int sow_adam_multi_dev(const void* chunks_dev, int n_chunks, int64_t total_elems, double lr, double beta1, double beta2,
                       double eps, double weight_decay, float* step_dev, int decoupled, int dtype, void* stream_) {
  SOWB_REQUIRE(step_dev != nullptr, "sow_adam_multi_dev: null step counter");
  return adam_launch(chunks_dev, n_chunks, total_elems, lr, beta1, beta2, eps, weight_decay, 1.0, 1.0, step_dev, nullptr,
                     nullptr, nullptr, false, decoupled, dtype, dtype, stream_);
}

// The argument checks shared by sow_adam_multi_amp and sow_adam_multi_clip; `fn` starts every message
static int check_amp_args(const char* fn, double bias_correction1, double bias_correction2, const float* step_dev,
                          const float* found_inf, int dtype, int state_dtype) {
  SOWB_REQUIRE(dtype == SOWB_BF16 || dtype == SOWB_F16 || dtype == SOWB_F32, "%s: unknown dtype %d", fn, dtype);
  SOWB_REQUIRE(state_dtype == dtype || state_dtype == SOWB_F32,
               "%s: state dtype %d unsupported for parameter dtype %d (the parameter's, or fp32)", fn, state_dtype, dtype);
  SOWB_REQUIRE(found_inf == nullptr || step_dev != nullptr,
               "%s: found_inf needs the device step counter (a host counter skips on the host)", fn);
  SOWB_REQUIRE(step_dev != nullptr || (bias_correction1 > 0.0 && bias_correction2 > 0.0),
               "%s: bias corrections must be positive", fn);
  return SOWB_OK;
}

int sow_adam_multi_amp(const void* chunks_dev, int n_chunks, int64_t total_elems, double lr, double beta1, double beta2,
                       double eps, double weight_decay, double bias_correction1, double bias_correction2, float* step_dev,
                       const float* grad_scale, const float* found_inf, int decoupled, int dtype, int state_dtype,
                       void* stream_) {
  if (int rc = check_amp_args("sow_adam_multi_amp", bias_correction1, bias_correction2, step_dev, found_inf, dtype,
                              state_dtype))
    return rc;
  return adam_launch(chunks_dev, n_chunks, total_elems, lr, beta1, beta2, eps, weight_decay,
                     step_dev != nullptr ? 1.0 : bias_correction1, step_dev != nullptr ? 1.0 : bias_correction2, step_dev,
                     grad_scale, found_inf, nullptr, true, decoupled, dtype, state_dtype, stream_);
}

int sow_adam_multi_clip(const void* chunks_dev, int n_chunks, int64_t total_elems, double lr, double beta1, double beta2,
                        double eps, double weight_decay, double bias_correction1, double bias_correction2, float* step_dev,
                        const float* grad_scale, const float* found_inf, const float* clip_coef, int decoupled, int dtype,
                        int state_dtype, void* stream_) {
  if (int rc = check_amp_args("sow_adam_multi_clip", bias_correction1, bias_correction2, step_dev, found_inf, dtype,
                              state_dtype))
    return rc;
  SOWB_REQUIRE(clip_coef != nullptr, "sow_adam_multi_clip: null clip coefficient");
  SOWB_REQUIRE(n_chunks >= 0, "sow_adam_multi_clip: n_chunks %d < 0", n_chunks);
  return adam_launch(chunks_dev, n_chunks, total_elems, lr, beta1, beta2, eps, weight_decay,
                     step_dev != nullptr ? 1.0 : bias_correction1, step_dev != nullptr ? 1.0 : bias_correction2, step_dev,
                     grad_scale, found_inf, clip_coef, true, decoupled, dtype, state_dtype, stream_);
}

int sow_grad_norm_partials(const void* chunks_dev, int n_chunks, int dtype, const float* grad_scale, float* partials,
                           void* stream_) {
  SOWB_REQUIRE(dtype == SOWB_BF16 || dtype == SOWB_F16 || dtype == SOWB_F32, "sow_grad_norm_partials: unknown dtype %d",
               dtype);
  SOWB_REQUIRE(n_chunks >= 0, "sow_grad_norm_partials: n_chunks %d < 0", n_chunks);
  SOWB_REQUIRE(partials != nullptr, "sow_grad_norm_partials: null partials");
  SOWB_REQUIRE(n_chunks == 0 || chunks_dev != nullptr, "sow_grad_norm_partials: null chunk table");
  if (n_chunks == 0) return SOWB_OK;
  if (int rc0 = ensure_context_for(chunks_dev)) return rc0;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const AdamChunk* ch = static_cast<const AdamChunk*>(chunks_dev);
  if (dtype == SOWB_F32) launch_norm_partials<float>(n_chunks, ch, grad_scale, partials, stream);
  else if (dtype == SOWB_BF16) launch_norm_partials<__nv_bfloat16>(n_chunks, ch, grad_scale, partials, stream);
  else launch_norm_partials<__half>(n_chunks, ch, grad_scale, partials, stream);
  SOWB_CHECK_CUDA(cudaGetLastError());
  return SOWB_OK;
}

int sow_grad_norm_finalize(const float* partials, int n_partials, double max_norm, float* total_norm, float* clip_coef,
                           void* stream_) {
  SOWB_REQUIRE(n_partials >= 1, "sow_grad_norm_finalize: n_partials %d < 1", n_partials);
  SOWB_REQUIRE(partials != nullptr && total_norm != nullptr && clip_coef != nullptr,
               "sow_grad_norm_finalize: null pointer argument");
  SOWB_REQUIRE(std::isfinite(max_norm) && max_norm > 0.0, "sow_grad_norm_finalize: max_norm %g must be finite and > 0",
               max_norm);
  if (int rc0 = ensure_context_for(partials)) return rc0;
  grad_norm_finalize_kernel<<<1, 256, 0, static_cast<cudaStream_t>(stream_)>>>(partials, n_partials, float(max_norm),
                                                                               total_norm, clip_coef);
  SOWB_CHECK_CUDA(cudaGetLastError());
  return SOWB_OK;
}

static int adam_launch(const void* chunks_dev, int n_chunks, int64_t total_elems, double lr, double beta1, double beta2,
                       double eps, double weight_decay, double bias_correction1, double bias_correction2, float* step_dev,
                       const float* grad_scale, const float* found_inf, const float* clip_coef, bool amp, int decoupled,
                       int dtype, int state_dtype, void* stream_) {
  if (n_chunks <= 0) return SOWB_OK;
  SOWB_REQUIRE(chunks_dev != nullptr, "sow_adam_multi: null chunk table");
  SOWB_REQUIRE(dtype == SOWB_BF16 || dtype == SOWB_F16 || dtype == SOWB_F32, "sow_adam_multi: unknown dtype %d", dtype);
  if (int rc0 = ensure_context_for(chunks_dev)) return rc0;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (step_dev != nullptr) {
    adam_step_inc_kernel<<<1, 1, 0, stream>>>(step_dev, found_inf);
    SOWB_CHECK_CUDA(cudaGetLastError());
  }
  AdamHyper h;
  h.lr = float(lr);
  h.beta1 = float(beta1);
  h.omb1 = float(1.0 - beta1);
  h.beta2 = float(beta2);
  h.omb2 = float(1.0 - beta2);
  h.eps = float(eps);
  h.decay_mul = float(1.0 - lr * weight_decay);
  h.weight_decay = float(weight_decay);
  h.step_size = float(lr / bias_correction1);
  h.inv_sqrt_bc2 = float(1.0 / sqrt(bias_correction2));
  h.decoupled = decoupled;
  // algorithmic bytes: p and the moments read + written, g read (and written back when it is unscaled or clipped)
  const int ep = elem_bytes(dtype), es = elem_bytes(state_dtype);
  const bool g_written = grad_scale != nullptr || clip_coef != nullptr;
  ProfileScope prof(stream, PROF_ADAM, double(2 * ep + ep + 4 * es + (g_written ? ep : 0)) * double(total_elems));
  const AdamChunk* ch = static_cast<const AdamChunk*>(chunks_dev);
  if (clip_coef != nullptr) {
    if (dtype == SOWB_F32)
      adam_multi_f32_kernel<true, true><<<n_chunks, 256, 0, stream>>>(ch, h, step_dev, grad_scale, found_inf, clip_coef);
    else if (dtype == SOWB_BF16)
      launch_16bit_clip<__nv_bfloat16>(n_chunks, ch, h, step_dev, grad_scale, found_inf, clip_coef, state_dtype, stream);
    else
      launch_16bit_clip<__half>(n_chunks, ch, h, step_dev, grad_scale, found_inf, clip_coef, state_dtype, stream);
  } else if (dtype == SOWB_F32) {
    if (amp)
      adam_multi_f32_kernel<true><<<n_chunks, 256, 0, stream>>>(ch, h, step_dev, grad_scale, found_inf);
    else
      adam_multi_f32_kernel<false><<<n_chunks, 256, 0, stream>>>(ch, h, step_dev, nullptr, nullptr);
  } else if (dtype == SOWB_BF16) {
    if (amp) launch_16bit<true, __nv_bfloat16>(n_chunks, ch, h, step_dev, grad_scale, found_inf, state_dtype, stream);
    else launch_16bit<false, __nv_bfloat16>(n_chunks, ch, h, step_dev, nullptr, nullptr, state_dtype, stream);
  } else {
    if (amp) launch_16bit<true, __half>(n_chunks, ch, h, step_dev, grad_scale, found_inf, state_dtype, stream);
    else launch_16bit<false, __half>(n_chunks, ch, h, step_dev, nullptr, nullptr, state_dtype, stream);
  }
  SOWB_CHECK_CUDA(cudaGetLastError());
  return SOWB_OK;
}

}  // extern "C"
