#include "common.cuh"

#include <map>
#include <mutex>
#include <stdlib.h>
#include <string.h>
#include <unordered_map>
#include <vector>

namespace sowb {

static thread_local char g_err[512] = "";

int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

cudaError_t set_max_smem_once(const void* kernel, size_t bytes) {
  static std::mutex mu;
  static std::map<std::pair<int, const void*>, size_t> done;     // (device, kernel) -> largest size already set
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) dev = -1;
  {
    std::lock_guard<std::mutex> lk(mu);
    auto it = done.find({dev, kernel});
    if (dev >= 0 && it != done.end() && it->second >= bytes) return cudaSuccess;
  }
  const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bytes));
  if (e == cudaSuccess && dev >= 0) {
    std::lock_guard<std::mutex> lk(mu);
    size_t& slot = done[{dev, kernel}];
    slot = std::max(slot, bytes);
  }
  return e;
}

int num_sms() {
  static std::mutex mu;
  static int cache[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  std::lock_guard<std::mutex> lk(mu);
  if (cache[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cache[dev] = n;
  }
  return cache[dev];
}

int require_sm100() {
  static std::mutex mu;
  static int cache[64] = {0};  // 0 unknown, 1 ok, -1 bad
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return set_error(SOWB_ECUDA, "cudaGetDevice failed: %s", cudaGetErrorString(e));
  if (dev < 0 || dev >= 64) return SOWB_OK;
  std::lock_guard<std::mutex> lk(mu);
  if (cache[dev] == 0) {
    int major = 0;
    e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    if (e != cudaSuccess) return set_error(SOWB_ECUDA, "cudaDeviceGetAttribute failed: %s", cudaGetErrorString(e));
    cache[dev] = (major == 10) ? 1 : -1;
  }
  if (cache[dev] < 0) return set_error(SOWB_ENOTSUP, "sow_b200 kernels require an sm_100 (B200) device");
  return SOWB_OK;
}

// ------------------------------------------------------------------------------------------------
// Tensor maps.  cuTensorMapEncodeTiled is resolved through the runtime so that the library has no link-time
// dependency on libcuda (it must dlopen on the GPU-less build host).  Encoded maps are cached: weights and
// workspaces keep their addresses across steps, so the steady state does no driver calls.
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, []() {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

struct MapKey {
  const void* base;
  uint64_t inner, outer, pitch;
  uint32_t b0, b1;
  int dt;   // CUtensorMapDataType: a bf16 and an fp16 map of the same memory are different maps
  bool operator==(const MapKey& o) const {
    return base == o.base && inner == o.inner && outer == o.outer && pitch == o.pitch && b0 == o.b0 && b1 == o.b1 &&
           dt == o.dt;
  }
};
struct MapKeyHash {
  size_t operator()(const MapKey& k) const {
    uint64_t h = reinterpret_cast<uint64_t>(k.base) * 0x9E3779B97F4A7C15ull;
    h ^= (k.inner * 0xC2B2AE3D27D4EB4Full) ^ (k.outer << 17) ^ (k.pitch << 29) ^ (uint64_t(k.b0) << 7) ^
         (uint64_t(k.b1) << 43) ^ uint64_t(k.dt);
    return static_cast<size_t>(h ^ (h >> 31));
  }
};

// A thread that has issued no CUDA call yet (autograd's per-device worker when the first backward node is ours) has no
// current driver context, and cuTensorMapEncodeTiled then fails with CUDA_ERROR_INVALID_CONTEXT.  Bind the primary
// context of the device that owns `ptr` -- derived from the pointer, not from the runtime's per-thread default (device 0),
// so that rank k of a multi-GPU job never touches another device.
typedef CUresult (*CtxGetCurrentFn)(CUcontext*);
typedef CUresult (*CtxSetCurrentFn)(CUcontext);
typedef CUresult (*PtrGetAttrFn)(void*, CUpointer_attribute, CUdeviceptr);
typedef CUresult (*PrimaryRetainFn)(CUcontext*, CUdevice);
typedef CUresult (*DeviceGetFn)(CUdevice*, int);

int ensure_context_for(const void* ptr) {
  static CtxGetCurrentFn get_cur = nullptr;
  static CtxSetCurrentFn set_cur = nullptr;
  static PtrGetAttrFn ptr_attr = nullptr;
  static PrimaryRetainFn retain = nullptr;
  static DeviceGetFn dev_get = nullptr;
  static std::once_flag once;
  std::call_once(once, []() {
    auto fetch = [](const char* name) -> void* {
      void* p = nullptr;
      cudaDriverEntryPointQueryResult q;
      if (cudaGetDriverEntryPoint(name, &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) return nullptr;
      return p;
    };
    get_cur = reinterpret_cast<CtxGetCurrentFn>(fetch("cuCtxGetCurrent"));
    set_cur = reinterpret_cast<CtxSetCurrentFn>(fetch("cuCtxSetCurrent"));
    ptr_attr = reinterpret_cast<PtrGetAttrFn>(fetch("cuPointerGetAttribute"));
    retain = reinterpret_cast<PrimaryRetainFn>(fetch("cuDevicePrimaryCtxRetain"));
    dev_get = reinterpret_cast<DeviceGetFn>(fetch("cuDeviceGet"));
  });
  if (!get_cur || !set_cur || !ptr_attr || !retain || !dev_get || ptr == nullptr) return SOWB_OK;   // best effort
  CUcontext cur = nullptr;
  if (get_cur(&cur) == CUDA_SUCCESS && cur != nullptr) return SOWB_OK;
  int ordinal = -1;
  if (ptr_attr(&ordinal, CU_POINTER_ATTRIBUTE_DEVICE_ORDINAL, reinterpret_cast<CUdeviceptr>(ptr)) != CUDA_SUCCESS || ordinal < 0)
    return SOWB_OK;
  CUdevice dev;
  CUcontext primary = nullptr;
  if (dev_get(&dev, ordinal) != CUDA_SUCCESS || retain(&primary, dev) != CUDA_SUCCESS || primary == nullptr)
    return set_error(SOWB_ECUDA, "could not retain the primary context of device %d", ordinal);
  if (set_cur(primary) != CUDA_SUCCESS) return set_error(SOWB_ECUDA, "could not bind the primary context of device %d", ordinal);
  return SOWB_OK;
}

int make_tensor_map_2d(CUtensorMap* out, const void* base, uint64_t inner, uint64_t outer, uint64_t pitch_bytes,
                       uint32_t box_inner, uint32_t box_outer, CUtensorMapDataType dt) {
  if (base == nullptr) return set_error(SOWB_EINVAL, "tensor map: null base pointer");
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0)
    return set_error(SOWB_EINVAL, "tensor map: base pointer %p is not 16-byte aligned", base);
  if (pitch_bytes % 16 != 0)
    return set_error(SOWB_EINVAL, "tensor map: row pitch %llu B is not a multiple of 16 (features must be multiples of 8)",
                     (unsigned long long)pitch_bytes);
  if (dt != CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 && dt != CU_TENSOR_MAP_DATA_TYPE_FLOAT16 && dt != CU_TENSOR_MAP_DATA_TYPE_FLOAT32)
    return set_error(SOWB_EINVAL, "tensor map: unsupported data type %d", (int)dt);
  const uint32_t elem_bytes = (dt == CU_TENSOR_MAP_DATA_TYPE_FLOAT32) ? 4 : 2;
  if (box_inner * elem_bytes != 128 || box_outer == 0 || box_outer > 256)
    return set_error(SOWB_EINVAL, "tensor map: unsupported box %u x %u", box_inner, box_outer);

  static std::mutex mu;
  static std::unordered_map<MapKey, CUtensorMap, MapKeyHash> cache;
  MapKey key{base, inner, outer, pitch_bytes, box_inner, box_outer, static_cast<int>(dt)};
  {
    std::lock_guard<std::mutex> lk(mu);
    auto it = cache.find(key);
    if (it != cache.end()) {
      memcpy(out, &it->second, sizeof(CUtensorMap));
      return SOWB_OK;
    }
  }
  EncodeTiledFn fn = get_encode_fn();
  if (fn == nullptr) return set_error(SOWB_ECUDA, "cuTensorMapEncodeTiled is unavailable (no CUDA driver?)");
  {
    const int rc = ensure_context_for(base);
    if (rc) return rc;
  }
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {pitch_bytes};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  static const CUtensorMapL2promotion promo = []() {
    const char* e = getenv("SOWB_TMA_PROMO");   // tuning knob: 0 none, 1 64 B, 2 128 B, 3 256 B (default)
    const int v = e ? atoi(e) : 3;
    return v == 0 ? CU_TENSOR_MAP_L2_PROMOTION_NONE
                  : (v == 1 ? CU_TENSOR_MAP_L2_PROMOTION_L2_64B
                            : (v == 2 ? CU_TENSOR_MAP_L2_PROMOTION_L2_128B : CU_TENSOR_MAP_L2_PROMOTION_L2_256B));
  }();
  CUresult r = fn(out, dt, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return set_error(SOWB_ECUDA,
                     "cuTensorMapEncodeTiled failed with CUresult %d (base %p inner %llu outer %llu pitch %llu box %ux%u)",
                     (int)r, base, (unsigned long long)inner, (unsigned long long)outer,
                     (unsigned long long)pitch_bytes, box_inner, box_outer);
  {
    std::lock_guard<std::mutex> lk(mu);
    if (cache.size() > 8192) cache.clear();  // activations churn addresses; weights re-enter immediately
    cache.emplace(key, *out);
  }
  return SOWB_OK;
}

// ---- live profiling --------------------------------------------------------------------------------
struct ProfRecord {
  cudaEvent_t a, b;
  int klass;
  double work;
};
static std::mutex g_prof_mu;
static bool g_prof_on = false;
static std::vector<ProfRecord> g_prof;

bool profile_enabled() { return g_prof_on; }

ProfileScope::ProfileScope(cudaStream_t s, int k, double w) : stream(s), klass(k), work(w) {
  if (!g_prof_on) return;
  if (cudaEventCreate(&start) != cudaSuccess) {
    start = nullptr;
    return;
  }
  cudaEventRecord(start, stream);
}
ProfileScope::~ProfileScope() {
  if (start == nullptr) return;
  cudaEvent_t end;
  if (cudaEventCreate(&end) != cudaSuccess) {
    cudaEventDestroy(start);
    return;
  }
  cudaEventRecord(end, stream);
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_prof.push_back({start, end, klass, work});
}

}  // namespace sowb

extern "C" {
int sow_profile_enable(int on) {
  std::lock_guard<std::mutex> lk(sowb::g_prof_mu);
  for (auto& r : sowb::g_prof) {
    cudaEventDestroy(r.a);
    cudaEventDestroy(r.b);
  }
  sowb::g_prof.clear();
  sowb::g_prof_on = on != 0;
  return SOWB_OK;
}
int sow_profile_read(int klass, double* total_ms, double* total_work, int64_t* launches) {
  std::lock_guard<std::mutex> lk(sowb::g_prof_mu);
  double ms = 0, work = 0;
  int64_t n = 0;
  for (auto& r : sowb::g_prof) {
    if (r.klass != klass) continue;
    cudaError_t e = cudaEventSynchronize(r.b);
    if (e != cudaSuccess) return sowb::set_error(SOWB_ECUDA, "sow_profile_read: %s", cudaGetErrorString(e));
    float t = 0;
    e = cudaEventElapsedTime(&t, r.a, r.b);
    if (e != cudaSuccess) return sowb::set_error(SOWB_ECUDA, "sow_profile_read: %s", cudaGetErrorString(e));
    ms += t;
    work += r.work;
    ++n;
  }
  if (total_ms) *total_ms = ms;
  if (total_work) *total_work = work;
  if (launches) *launches = n;
  return SOWB_OK;
}
int sow_abi_version(void) { return 3; }
const char* sow_last_error(void) { return sowb::g_err; }
}
