// Thin inline-PTX wrappers for sm_100a: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (MMA / TMEM).
// Everything here is device-only and header-only.  No CUTLASS/CuTe dependency.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda.h>
#include <stdint.h>

namespace sowb {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ uint32_t lane_id() {
  uint32_t l;
  asm volatile("mov.u32 %0, %%laneid;" : "=r"(l));
  return l;
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n"
      ".reg .b32 %%rx;\n"
      ".reg .pred %%px;\n"
      "elect.sync %%rx|%%px, %1;\n"
      "@%%px mov.s32 %0, 1;\n"
      "}\n"
      : "+r"(pred)
      : "r"(0xffffffffu));
  return pred != 0;
}

// ----------------------------------------------------------------------------------------------
// mbarrier
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}

// ----------------------------------------------------------------------------------------------
// TMA
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// Make a tensor map that lives in GLOBAL memory (written by a host copy before the launch) safe to use from
// the async proxy even if the same address held a different descriptor in an earlier launch.
__device__ __forceinline__ void tma_acquire_desc(const CUtensorMap* m) {
  asm volatile("fence.proxy.tensormap::generic.acquire.gpu [%0], 128;" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 2-D tiled load: coordinates are (c0 = innermost/contiguous dim, c1 = outer dim), in elements.
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int32_t c0,
                                            int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* smem_src, int32_t c0, int32_t c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
// Pull a tile from HBM into L2 ahead of the TMA load that will consume it (no shared-memory slot needed).
__device__ __forceinline__ void tma_prefetch_l2_2d(const CUtensorMap* m, int32_t c0, int32_t c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];" ::"l"(reinterpret_cast<uint64_t>(m)),
               "r"(c0), "r"(c1)
               : "memory");
}
// L2 eviction-priority policies for streaming (evict_first) and re-used (evict_last) data
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void tma_load_2d_hint(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int32_t c0,
                                                 int32_t c1, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint "
      "[%0], [%1, {%3, %4}], [%2], %5;" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "l"(policy)
      : "memory");
}
__device__ __forceinline__ void tma_store_2d_hint(const CUtensorMap* m, const void* smem_src, int32_t c0, int32_t c1,
                                                  uint64_t policy) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group.L2::cache_hint [%0, {%2, %3}], [%1], %4;" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "l"(policy)
               : "memory");
}
// 1-D bulk copy global -> shared, completion counted in bytes on an mbarrier.
__device__ __forceinline__ void bulk_load_1d_hint(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar,
                                                  uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
          smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
      : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait_all() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// ----------------------------------------------------------------------------------------------
// tcgen05 / TMEM
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc]; issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// tf32 x tf32 -> f32 (operands are fp32 words in smem; the tensor core reads the top 19 bits)
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// ---- CTA pairs (cta_group::2): two CTAs of a cluster (ranks 2j, 2j+1) share one MMA -------------------------------------
// Allocation and deallocation are collective over one warp of EACH CTA of the pair; both get the same TMEM address.
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish_pair() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// Issued by one thread of the even CTA: A (M = 256) is rows 0..127 from the even CTA's smem and 128..255 from the odd CTA's,
// B's N columns are split in halves the same way (the descriptors are offsets valid in both CTAs); D is each CTA's own
// 128 TMEM lanes x N columns at tmem_d.
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive once on the mbarrier at the same smem offset in every CTA of cta_mask, when all earlier pair MMAs have completed.
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"(cta_mask)
      : "memory");
}
// 2-D tiled load into THIS CTA's smem whose completed bytes are counted on `cluster_bar`, a shared::cluster address that
// may be the peer CTA's barrier (the even CTA of the pair counts both CTAs' bytes).
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* m, uint32_t cluster_bar, int32_t c0,
                                                 int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(cluster_bar), "r"(c0), "r"(c1)
      : "memory");
}

// TMEM -> registers: this warp's 32 lanes x 32 consecutive fp32 columns.
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ----------------------------------------------------------------------------------------------
// Descriptors (bit layouts: SM100 UMMA shared-memory matrix descriptor and instruction descriptor)
// ----------------------------------------------------------------------------------------------
// Shared-memory matrix descriptor, SWIZZLE_128B, descriptor version 1 (Blackwell).
//   K-major operand  : rows of 128 B (64 x 16-bit or 32 x 32-bit along K), 8-row atoms of 1024 B;
//                      SBO = byte distance between 8-row atoms; LBO unused (encoded 1).
//   MN-major operand : atoms of (64 x 16-bit along MN) x (8 along K) = 1024 B; LBO = byte distance between
//                      consecutive 64-element MN blocks, SBO = byte distance between consecutive 8-deep K groups.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= static_cast<uint64_t>(1) << 46;  // version = 1
  d |= static_cast<uint64_t>(2) << 61;  // layout_type = SWIZZLE_128B
  return d;
}

// Instruction descriptor for kind::f16 / kind::tf32, fp32 accumulate.
//   ab_format: 0 = f16, 1 = bf16, 2 = tf32.  a_mn / b_mn: 1 = operand is MN-major in smem.
__host__ __device__ constexpr uint32_t make_idesc(uint32_t ab_format, uint32_t M, uint32_t N, uint32_t a_mn,
                                                   uint32_t b_mn) {
  return (1u << 4)                 // c_format = f32
         | (ab_format << 7)        // a_format
         | (ab_format << 10)       // b_format
         | (a_mn << 15)            // a_major
         | (b_mn << 16)            // b_major
         | ((N >> 3) << 17)        // n_dim
         | ((M >> 4) << 24);       // m_dim
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

// The 16-bit operand type of the tcgen05 paths as a template flag: F16 = false -> bf16, true -> IEEE fp16.
//   kind::f16 instruction-descriptor format: 1 = bf16, 0 = fp16 (same rate).
//   pack: round to nearest even (cvt.rn.f16x2.f32 / cvt.rn.bf16x2.f32, no .satfinite: fp16 overflow gives +-inf).
template <bool F16>
__host__ __device__ constexpr uint32_t ab_format16() { return F16 ? 0u : 1u; }
template <bool F16>
__device__ __forceinline__ uint32_t pack16x2(float lo, float hi) {
  if (F16) {
    __half2 v = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
  }
  return pack_bf16x2(lo, hi);
}
// the low / high 16-bit element of a packed pair, widened exactly to fp32
template <bool F16>
__device__ __forceinline__ float lo16_to_f32(uint32_t w) {
  return F16 ? __half2float(__ushort_as_half(static_cast<unsigned short>(w & 0xffffu))) : __uint_as_float(w << 16);
}
template <bool F16>
__device__ __forceinline__ float hi16_to_f32(uint32_t w) {
  return F16 ? __half2float(__ushort_as_half(static_cast<unsigned short>(w >> 16))) : __uint_as_float(w & 0xffff0000u);
}

// ----------------------------------------------------------------------------------------------
// thread-block clusters / distributed shared memory
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t cluster_id_x() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r));
  return r;
}
// shared::cta address of this CTA -> shared::cluster address of the same offset in CTA `rank`
__device__ __forceinline__ uint32_t map_to_cta(uint32_t local_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void st_cluster_f32x4(uint32_t remote_addr, float a, float b, float c, float d) {
  asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(remote_addr), "f"(a), "f"(b), "f"(c), "f"(d)
               : "memory");
}
// arrive on an mbarrier that lives in another CTA of the cluster; release orders this thread's earlier DSMEM stores
__device__ __forceinline__ void mbar_arrive_remote(uint32_t remote_bar_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote_bar_addr) : "memory");
}
// wait with cluster-scope acquire: data written by peer CTAs before their arrive is visible afterwards
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  uint32_t ok = 0;
  while (!ok) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  }
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// 1-D bulk copy shared -> global (bulk async-group completion)
__device__ __forceinline__ void bulk_store_1d(void* gdst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(reinterpret_cast<uint64_t>(gdst)),
               "r"(smem_u32(smem_src)), "r"(bytes)
               : "memory");
}

__device__ __forceinline__ void named_barrier_sync(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

}  // namespace sowb
