// Host-side plumbing shared by the C-ABI translation units: error reporting, device checks, and the
// TMA tensor-map encoder (driver entry point fetched at run time so that the library loads on GPU-less hosts).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/sow_b200.h"

namespace sowb {

int set_error(int code, const char* fmt, ...);

#define SOWB_CHECK_CUDA(expr)                                                                          \
  do {                                                                                                 \
    cudaError_t _e = (expr);                                                                           \
    if (_e != cudaSuccess)                                                                             \
      return ::sowb::set_error(SOWB_ECUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),    \
                               __FILE__, __LINE__);                                                    \
  } while (0)

#define SOWB_REQUIRE(cond, ...)                                   \
  do {                                                            \
    if (!(cond)) return ::sowb::set_error(SOWB_EINVAL, __VA_ARGS__); \
  } while (0)

// Programmatic dependent launch: the chains of small dependent kernels on the TT path (head -> Gram -> sum -> Cholesky ->
// solve -> ... ) spend as long in launch gaps as in the kernels.  Launched through launch_pdl, a kernel may be scheduled
// while its predecessor in the stream drains; pdl_wait() -- the first statement that touches global memory must come
// after it -- blocks until the predecessor has completed and its writes are visible, so the stream order is unchanged.
// Both instructions are no-ops for a kernel launched the ordinary way.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                              Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) once per (device, kernel): ~1 us of host time on every launch otherwise.
cudaError_t set_max_smem_once(const void* kernel, size_t bytes);
template <typename K>
inline cudaError_t set_max_smem_once(K* kernel, size_t bytes) {
  return set_max_smem_once(reinterpret_cast<const void*>(kernel), bytes);
}

// Number of SMs of the current device (cached per device).
int num_sms();
// 0 if the current device is sm_100, else an error code (message set).
int require_sm100();
// dst[b][i] = sum over s (ascending) of part[b][s][i]: the fixed-order reduction of split partials (tt.cu)
int launch_sum_splits(const float* part, int splits, int64_t split_stride, int64_t part_bs, float* dst, int64_t dst_bs,
                      int64_t n, int batch, cudaStream_t stream);

// Bind the primary context of the device owning `ptr` to the calling thread if the thread has none (see common.cu).
int ensure_context_for(const void* ptr);

// 2-D row-major tensor map with 128B swizzle.  `inner` is the contiguous dimension (elements), `outer` the row
// count, `pitch_bytes` the row pitch; box = (box_inner x box_outer) elements.  dt: BFLOAT16, FLOAT16 or FLOAT32.
int make_tensor_map_2d(CUtensorMap* out, const void* base, uint64_t inner, uint64_t outer, uint64_t pitch_bytes,
                       uint32_t box_inner, uint32_t box_outer, CUtensorMapDataType dt);
// TMA element type of the 2-byte operands of a SOWB_BF16 / SOWB_F16 call
inline CUtensorMapDataType map_type16(bool f16) {
  return f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
}

// The tensor-train entry points take bf16 and fp32 only: reject SOWB_F16 (and unknown codes) before any work is queued.
#define SOWB_REQUIRE_TT_DTYPE(fn, dtype) \
  SOWB_REQUIRE((dtype) == SOWB_BF16 || (dtype) == SOWB_F32, "%s: dtype %d unsupported (tensor-train path: bf16 / fp32)", fn, dtype)

// ------------------------------------------------------------------------------------------------
// Live per-kernel timing (bench.py roofline): when enabled, launches are bracketed by CUDA events recorded on the
// launching stream; sow_profile_read() sums elapsed time / algorithmic work per kernel class.
// ------------------------------------------------------------------------------------------------
enum ProfClass : int {
  PROF_GEMM_FWD = 0,     // y  = x.W + t.B          (flops)
  PROF_GEMM_DX = 1,      // dX = dY.W^T + dt.A^T    (flops)
  PROF_GEMM_SKINNY = 2,  // t_cat = x.[A_q|A_k|..]  (flops)
  PROF_GEMM_SPLITK = 3,  // dA_cat = x^T.dt_cat     (flops)
  PROF_MERGE = 4,        // grouped merge           (bytes)
  PROF_ADAM = 5,         // multi-tensor Adam       (bytes)
  PROF_GEMM_K2 = 6,      // fused dt + dB pass over dY (flops)
  PROF_NUM = 7,
};
bool profile_enabled();
struct ProfileScope {
  cudaStream_t stream;
  cudaEvent_t start = nullptr;
  int klass;
  double work;
  ProfileScope(cudaStream_t s, int klass, double work);
  ~ProfileScope();
};

__host__ __device__ static inline int round_up(int x, int m) { return (x + m - 1) / m * m; }
static inline int64_t round_up64(int64_t x, int64_t m) { return (x + m - 1) / m * m; }
__host__ __device__ static inline int ceil_div(int x, int m) { return (x + m - 1) / m; }

}  // namespace sowb
