// Grouped SoW merge:  W <- W_prev + scale * A . B   for every SoW linear of a model in ONE launch.
//
// Replaces the dense branch of SoWLinear.accumulate (tn_gradient/layer/sow.py:131-134,140,151-153), which in the
// reference materialises >= 4 in x out temporaries per layer (stack, sum, scale, add) through separate kernels.
//
// The op is HBM-bound (2 bytes read + 2 bytes written per element) but at r = 50 it needs 25 flop/byte, above what
// the CUDA cores sustain at full bandwidth, so the rank-r product runs on tcgen05 (one 128x128x64 UMMA block per
// tile) and everything else is a streaming read-modify-write pipeline.  Each matrix is cut into STRIPS of 4 column
// tiles; the 128x128 tiles of all layers are flattened (layer, strip, m, n-in-strip) and every CTA owns one
// CONTIGUOUS range of that index space.  The B tiles of a strip stay resident in shared memory while the CTA walks
// down the strip, and the [128 x r] block of A is staged once per row of the strip, so per tile only W moves
// (measured: re-fetching the B tile from L2 for every W tile cost 11-16 % of the achieved bandwidth):
//
//   warp  8    : TMA producer.  Per tile: W_prev tile (2 boxes of [128 rows x 64 cols], swizzle 128B) into one of
//                the W slots.  Per strip: up to 4 B tiles ([64 k-rows x 128 cols], rows >= r zero-filled by the
//                tensor-map bounds), each issued together with the first W tile that needs it.
//   warps 10-13: A operand.  Per strip row: ONE bulk copy of the contiguous A[m0:m0+128, 0:r] block (pitch r*2
//                bytes is not TMA-tensor legal, but the block is contiguous) into a staging buffer, issued one
//                strip row AHEAD, then repacked (thread per row, conflict-free 4-byte reads when r/2 is odd) into
//                the zero-padded K-major swizzled operand tile the tensor core reads.
//   warp  9    : TMEM allocation; lane 0 issues the UMMAs (4 accumulator stages in TMEM = one per W slot, so
//                the tensor core never waits for the epilogue).
//   warps 0-7  : epilogue.  tcgen05.ld of the accumulator, add in place onto the W tile in smem (16-byte swizzled
//                accesses, conflict-free), hand the slot to the store warp.
//   warps 14-17: store group.  Coalesced 16-byte global stores of the finished tile (2 rows x 256 B per warp
//                instruction), clipped at the matrix edge; frees the slot.
//
// 3 W slots of 32 KB keep a tile load in flight per SM while one tile is in the epilogue and one is being stored
// (4 slots measured no faster: the memory system, not the slot count, binds).  The scalar fields of every table
// entry are staged in shared memory at kernel start and the next matrix's tensor maps are prefetched one matrix
// ahead, because under HBM saturation a dependent global load costs microseconds.
// F16 (template flag): W, A and B are IEEE fp16 instead of bf16 -- the instruction-descriptor format, the widening of
// W_prev and the one rounding of the new W in the epilogue (TMA element types on the host side).  The A repack and the
// store group move 16-bit words without interpreting them.
// Debug aid: sow_merge_debug_timeline() makes CTA 0 record clock64 stamps per tile (tools/merge_timeline.py).
#include "common.cuh"
#include "ptx.cuh"

#include <algorithm>
#include <mutex>
#include <stdlib.h>
#include <string.h>
#include <vector>

namespace sowb {

// W slots / resident B tiles per strip.  Re-measured in round 2 (Llama-350M r=50, kernel only): 3 slots + strip 4 ->
// 0.250-0.256 ms; 4 slots + strip 3 (what fits 227 KB) -> 0.265 ms, with the load latency growing from 5.4 k to 6.5 k
// cycles: the memory system, not the slot count, binds.  The CTAs do not finish together (globaltimer per CTA: first
// 216 us, median 232 us, last 246 us): the remaining gap to the copy bandwidth is that tail plus start-up.  Giving every CTA
// 2 / 4 / 8 interleaved sub-ranges instead of one contiguous range does not help (0.262 / 0.264 / 0.268 ms): the slow CTAs
// are slow because of where their SM sits, not because of which addresses they touch.  A work-stealing scheduler was
// built and measured as well (static first range + 8-tile chunks claimed with an atomic counter, published by the producer
// to the other roles through an smem ring): it balances the tail (0.272 -> 0.260 ms in that build) but the extra live state
// pushes the 18-warp kernel past its 96-register budget (5 warps share a 16 K-register sub-partition, so 96 is the cap;
// 64 B of spills in the epilogue loop) and the steady state loses more (0.253 -> 0.272 ms) than the tail gains.
#ifndef SOWB_MG_SLOTS
#define SOWB_MG_SLOTS 3
#endif
#ifndef SOWB_MG_STRIP
#define SOWB_MG_STRIP 4
#endif
constexpr int kMgBM = 128, kMgBN = 128, kMgSlots = SOWB_MG_SLOTS;
constexpr int kMgWBytes = kMgBM * kMgBN * 2;        // 32 KB
constexpr int kMgBBytes = 64 * kMgBN * 2;           // 16 KB
constexpr int kMgABytes = kMgBM * 64 * 2;           // 16 KB (operand tile and staging buffer)
constexpr int kMgSlotBytes = kMgWBytes;
constexpr int kMgStrip = SOWB_MG_STRIP;             // column tiles per strip (B tiles resident in smem)
constexpr int kMgAcc = 4;                           // TMEM accumulator stages
// W tiles pulled into L2 (cp.async.bulk.prefetch.tensor) ahead of the slot that will load them.  OFF: measured on B200
// (Llama-350M r=50, 20 merges each) distance 0 / 4 / 6 / 10 / 16 -> 0.250 / 0.351 / 0.366 / 0.377 / 0.379 ms: the
// prefetches compete with the demand loads for the same TMA unit and L2 slots.  SOWB_MERGE_PREFETCH=<n> re-enables it.
constexpr int kMgPrefetchDefault = 0;
constexpr int kMgMaxEntries = 384;                  // per launch (longer tables are split by the host)
constexpr int kMgNumBars = 3 * kMgSlots + 2 * kMgAcc + 3 + 2 * kMgStrip;   // + one 8-byte cell for the TMEM address
constexpr int kMgBarBytes = 320;
static_assert((kMgNumBars + 1) * 8 <= kMgBarBytes, "barrier block overflows into the entry table");
constexpr int kMgSmemTotal =
    1024 + kMgSlots * kMgSlotBytes + kMgStrip * kMgBBytes + 2 * kMgABytes + kMgBarBytes + kMgMaxEntries * 56;
constexpr int kMgThreads = 576;
constexpr int kMgStoreThreads = 128;
constexpr int kMgEpiThreads = 256;
constexpr int kMgRepackThreads = 128;
constexpr uint32_t kMgTmemCols = kMgAcc * kMgBN;   // 512: the whole TMEM (1 CTA per SM)
static_assert(kMgSmemTotal <= 232448, "merge kernel exceeds the 227 KB shared-memory opt-in limit");

struct alignas(128) MergeDevEntry {
  CUtensorMap tmWin;   // W_prev loads  (box 64 cols x 128 rows)
  CUtensorMap tmWout;  // W stores
  CUtensorMap tmB;     // B[r, out] as MN-major operand (box 64 cols x 64 rows)
  const __nv_bfloat16* A;
  __nv_bfloat16* W;    // destination matrix
  int lda;             // row pitch of A in elements (= full rank)
  int in, out, r;      // r = rank chunk handled by this entry (<= 64)
  float scale;
  int m_tiles, n_tiles, tile_begin;
  int has_prev;
  int a_bulk;          // the [rows x r] blocks of A are contiguous, 16-byte aligned and a multiple of 16 bytes long
};

// Scalar part of an entry, staged in shared memory at kernel start: under HBM saturation a global load costs
// microseconds, and every role needs these fields whenever its range crosses into the next matrix.
struct MergeInfo {
  const __nv_bfloat16* A;
  __nv_bfloat16* W;
  int lda, in, out, r;
  float scale;
  int m_tiles, n_tiles, tile_end;
  int has_prev, a_bulk;
};
static_assert(sizeof(MergeInfo) == 56, "MergeInfo layout");

// Position of one CTA inside the flattened (entry, strip, m-tile, n-in-strip) space.  Every role walks the same
// sequence of tiles.
struct MergeCursor {
  const MergeDevEntry* tab;   // global: tensor maps
  const MergeInfo* info;      // smem: scalar fields of every entry
  int ei, ebeg, nt, mtiles;
  int prev_mt, prev_strip;
  bool entry_changed, new_strip, new_item, last_of_item, b_first_use, b_last_use;
  int m0, n0, mt, strip, j, width;
  const MergeInfo* e;
  const MergeDevEntry* g;
  int n_entries;

  __device__ __forceinline__ void init(const MergeDevEntry* t, const MergeInfo* inf, int n, int first_tile) {
    tab = t;
    info = inf;
    n_entries = n;
    int lo = 0, hi = n_entries - 1;   // smallest ei with tile_end > first_tile
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (info[mid].tile_end > first_tile) hi = mid; else lo = mid + 1;
    }
    ei = lo;
    ebeg = ei ? info[ei - 1].tile_end : 0;
    e = &info[ei];
    g = &tab[ei];
    nt = e->n_tiles;
    mtiles = e->m_tiles;
    prev_mt = -1;
    prev_strip = -1;
    entry_changed = true;
  }
  // [first, last] = this CTA's range of tiles.  Every role calls seek() with consecutive tile numbers, so after the first
  // call (which locates the tile with divisions) the position is advanced incrementally: j -> mt -> strip -> entry.  The
  // kernel is partly issue-bound (17 warps walk this cursor for every 32 KB tile), and the divisions were a quarter of
  // its instructions.
  __device__ __forceinline__ void seek(int tile, int first, int last) {
    bool changed = false;
    if (prev_mt < 0) {
      // first tile of this CTA
      changed = entry_changed;
      while (tile >= info[ei].tile_end) {
        ebeg = info[ei].tile_end;
        ++ei;
      }
      e = &info[ei];
      g = &tab[ei];
      nt = e->n_tiles;
      mtiles = e->m_tiles;
      const int local = tile - ebeg;
      const int per_full = mtiles * kMgStrip;          // tiles in a full strip
      strip = local / per_full;
      const int rem = local - strip * per_full;
      width = min(kMgStrip, nt - strip * kMgStrip);     // only the last strip of a matrix can be narrower
      mt = rem / width;
      j = rem - mt * width;
      new_strip = true;
      new_item = true;
    } else {
      new_strip = false;
      new_item = false;
      if (++j == width) {
        j = 0;
        new_item = true;
        if (++mt == mtiles) {
          mt = 0;
          new_strip = true;
          ++strip;
          if (tile >= info[ei].tile_end) {
            do {
              ebeg = info[ei].tile_end;
              ++ei;
            } while (tile >= info[ei].tile_end);
            changed = true;
            e = &info[ei];
            g = &tab[ei];
            nt = e->n_tiles;
            mtiles = e->m_tiles;
            strip = 0;
          }
          width = min(kMgStrip, nt - strip * kMgStrip);
        }
      }
    }
    entry_changed = changed;
    prev_mt = mt;
    prev_strip = strip;
    last_of_item = (j == width - 1) || tile == last;
    // B tile j of a strip is used by tiles (tile0 + j + k*width): first / last use inside this CTA's range
    b_first_use = mt == 0 || tile - width < first;
    b_last_use = mt == mtiles - 1 || tile + width > last;
    m0 = mt * kMgBM;
    n0 = (strip * kMgStrip + j) * kMgBN;
  }
};

template <bool F16>
__global__ void __launch_bounds__(kMgThreads, 1)
sow_merge_kernel(const MergeDevEntry* __restrict__ tab, int n_entries, int total_tiles, int prefetch,
                 long long* __restrict__ dbg_ts) {
  // debug timeline (SOWB_MERGE_TS): CTA 0 records clock64 stamps per tile: [tile][8]
  auto stamp = [&](int tile_local, int k) {
    if (dbg_ts != nullptr && blockIdx.x == 0 && tile_local < 256) dbg_ts[tile_local * 8 + k] = clock64();
  };
  if (dbg_ts != nullptr && threadIdx.x == 0) {   // per-CTA start / end wall time (debug): dbg_ts[2048 + 2 * cta]
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    dbg_ts[2048 + 2 * blockIdx.x] = static_cast<long long>(t);
  }
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sBt = smem + kMgSlots * kMgSlotBytes;      // the strip's B tiles (MN-major swizzled operands)
  uint8_t* sA = sBt + kMgStrip * kMgBBytes;           // K-major swizzled A operand tile
  uint8_t* stage = sA + kMgABytes;                    // raw [rows x r] block of A
  uint64_t* bars = reinterpret_cast<uint64_t*>(stage + kMgABytes);
  uint64_t* full_bar = bars;                          // [slots] 1 + tx      : W_prev landed
  uint64_t* empty_bar = bars + kMgSlots;              // [slots] 1           : store has read the slot
  uint64_t* wready_bar = bars + 2 * kMgSlots;         // [slots] 256         : epilogue finished the tile
  uint64_t* tfull_bar = bars + 3 * kMgSlots;          // [kMgAcc] 1 (umma commit)
  uint64_t* tempty_bar = tfull_bar + kMgAcc;          // [kMgAcc] 256
  uint64_t* astage_full = tempty_bar + kMgAcc;        // 1 + tx
  uint64_t* a_full = astage_full + 1;                 // 128
  uint64_t* a_empty = astage_full + 2;                // 1 (umma commit)
  uint64_t* b_full = astage_full + 3;                 // [kMgStrip] 1 + tx
  uint64_t* b_empty = b_full + kMgStrip;              // [kMgStrip] 1 (umma commit)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(b_empty + kMgStrip);
  MergeInfo* info = reinterpret_cast<MergeInfo*>(reinterpret_cast<uint8_t*>(bars) + kMgBarBytes);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < n_entries; i += kMgThreads) {
    const MergeDevEntry* t = &tab[i];
    MergeInfo mi;
    mi.A = t->A;
    mi.W = t->W;
    mi.lda = t->lda;
    mi.in = t->in;
    mi.out = t->out;
    mi.r = t->r;
    mi.scale = t->scale;
    mi.m_tiles = t->m_tiles;
    mi.n_tiles = t->n_tiles;
    mi.tile_end = t->tile_begin + t->m_tiles * t->n_tiles;
    mi.has_prev = t->has_prev;
    mi.a_bulk = t->a_bulk;
    info[i] = mi;
  }
  if (threadIdx.x == 0) {
    for (int i = 0; i < kMgSlots; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], kMgStoreThreads);
      mbar_init(&wready_bar[i], kMgEpiThreads);
    }
    for (int i = 0; i < kMgAcc; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], kMgEpiThreads);
    }
    for (int i = 0; i < kMgStrip; ++i) {
      mbar_init(&b_full[i], 1);
      mbar_init(&b_empty[i], 1);
    }
    mbar_init(astage_full, 1);
    mbar_init(a_full, kMgRepackThreads);
    mbar_init(a_empty, 1);
    fence_mbar_init();
  }
  if (warp == 9) {
    tmem_alloc(tmem_slot, kMgTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int lo = static_cast<int>(static_cast<int64_t>(blockIdx.x) * total_tiles / gridDim.x);
  const int hi = static_cast<int>(static_cast<int64_t>(blockIdx.x + 1) * total_tiles / gridDim.x);

  if (warp == 8) {
    if (lane == 0 && lo < hi) {
      // ===================== TMA producer =====================
      MergeCursor c, pf;                  // pf runs kMgPrefetch tiles ahead and pulls W tiles from HBM into L2
      c.init(tab, info, n_entries, lo);
      pf.init(tab, info, n_entries, lo);
      int pf_tile = lo;
      int slot = 0;
      uint32_t phase = 0, b_phases = 0;   // b_phases: one parity bit per resident B tile
      const uint64_t pol_keep = l2_policy_evict_last();
      for (int tile = lo; tile < hi; ++tile) {
        // optional (off by default, see kMgPrefetchDefault): deepen the HBM pipeline beyond the 3 shared-memory slots
        while (prefetch > 0 && pf_tile < hi && pf_tile <= tile + prefetch) {
          pf.seek(pf_tile, lo, hi - 1);
          if (pf_tile > tile + kMgSlots - 1 && pf.e->has_prev) {
            if (pf.entry_changed) tma_acquire_desc(&pf.g->tmWin);
            tma_prefetch_l2_2d(&pf.g->tmWin, pf.n0, pf.m0);
            tma_prefetch_l2_2d(&pf.g->tmWin, pf.n0 + 64, pf.m0);
          }
          ++pf_tile;
        }
        c.seek(tile, lo, hi - 1);
        const MergeInfo* e = c.e;
        if (c.entry_changed) {
          // descriptors live in global memory: fetch the NEXT matrix's into the descriptor cache now, so that the
          // first loads of that matrix do not wait a (loaded) HBM round trip
          if (tile == lo) {
            tma_acquire_desc(&c.g->tmWin);
            tma_acquire_desc(&c.g->tmB);
          }
          if (c.ei + 1 < n_entries) {
            tma_acquire_desc(&c.g[1].tmWin);
            tma_acquire_desc(&c.g[1].tmB);
            tma_prefetch_desc(&c.g[1].tmWin);
            tma_prefetch_desc(&c.g[1].tmB);
          }
        }
        // W first: it depends on nothing but a free slot
        uint8_t* sW = smem + slot * kMgSlotBytes;
        stamp(tile - lo, 0);
        mbar_wait(&empty_bar[slot], phase ^ 1);
        stamp(tile - lo, 1);
        if (e->has_prev) {
          mbar_expect_tx(&full_bar[slot], kMgWBytes);
          // default L2 policy on purpose: the line must still be in L2 when the store group writes it back a few
          // microseconds later (measured: evict_first loads / streaming stores cost 8 % of the achieved bandwidth)
          tma_load_2d(sW, &c.g->tmWin, &full_bar[slot], c.n0, c.m0);
          tma_load_2d(sW + 16384, &c.g->tmWin, &full_bar[slot], c.n0 + 64, c.m0);
        } else {
          mbar_arrive(&full_bar[slot]);
        }
        if (++slot == kMgSlots) {
          slot = 0;
          phase ^= 1;
        }
        if (c.b_first_use) {
          // B tile j of this strip travels with the first W tile that needs it; its buffer is free once the last
          // UMMA of the previous strip that read it has completed (issued >= 4 tiles ago)
          uint8_t* sB = sBt + c.j * kMgBBytes;
          mbar_wait(&b_empty[c.j], ((b_phases >> c.j) & 1u) ^ 1u);
          mbar_expect_tx(&b_full[c.j], kMgBBytes);
          tma_load_2d_hint(sB, &c.g->tmB, &b_full[c.j], c.n0, 0, pol_keep);
          tma_load_2d_hint(sB + 8192, &c.g->tmB, &b_full[c.j], c.n0 + 64, 0, pol_keep);
          b_phases ^= 1u << c.j;
        }
      }
    }
  } else if (warp >= 10 && warp < 14) {
    // ===================== A repack group =====================
    if (lo < hi) {
      const int row = threadIdx.x - 320;  // 0..127: one row of the operand tile per thread
      MergeCursor c, nx;                  // nx runs one strip row ahead: its A block is fetched while c's is used
      c.init(tab, info, n_entries, lo);
      nx.init(tab, info, n_entries, lo);
      int nx_tile = lo;
      const uint64_t pol_keep = l2_policy_evict_last();
      auto prefetch_next_item = [&]() {
        while (nx_tile < hi) {
          nx.seek(nx_tile, lo, hi - 1);
          ++nx_tile;
          if (nx.new_item) {
            if (nx.e->a_bulk && row == 0) {
              const int rows = min(kMgBM, nx.e->in - nx.m0);
              const uint32_t bytes = static_cast<uint32_t>(rows) * nx.e->r * 2u;
              mbar_expect_tx(astage_full, bytes);
              bulk_load_1d_hint(stage, nx.e->A + static_cast<int64_t>(nx.m0) * nx.e->r, bytes, astage_full, pol_keep);
            }
            return;
          }
        }
      };
      prefetch_next_item();
      uint32_t st_phase = 0, ae_phase = 0;
      for (int tile = lo; tile < hi; ++tile) {
        c.seek(tile, lo, hi - 1);
        if (!c.new_item) continue;
        const MergeInfo* e = c.e;
        const int r = e->r, lda = e->lda;
        const bool live = row < min(kMgBM, e->in - c.m0);
        uint32_t w[32];  // the row as 32 packed 16-bit pairs, zero beyond r
        if (e->a_bulk) {
          mbar_wait(astage_full, st_phase);
          st_phase ^= 1;
          if ((r & 1) == 0) {
            const uint32_t* src = reinterpret_cast<const uint32_t*>(stage + row * r * 2);
            const int words = r >> 1;
#pragma unroll
            for (int j = 0; j < 32; ++j) w[j] = (live && j < words) ? src[j] : 0u;
          } else {
            const uint16_t* src = reinterpret_cast<const uint16_t*>(stage) + row * r;
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const uint32_t lo16 = (live && 2 * j < r) ? src[2 * j] : 0u;
              const uint32_t hi16 = (live && 2 * j + 1 < r) ? src[2 * j + 1] : 0u;
              w[j] = lo16 | (hi16 << 16);
            }
          }
        } else {
          const uint16_t* src = reinterpret_cast<const uint16_t*>(e->A) + static_cast<int64_t>(c.m0 + row) * lda;
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const uint32_t lo16 = (live && 2 * j < r) ? __ldg(src + 2 * j) : 0u;
            const uint32_t hi16 = (live && 2 * j + 1 < r) ? __ldg(src + 2 * j + 1) : 0u;
            w[j] = lo16 | (hi16 << 16);
          }
        }
        // every thread has its row in registers: the staging buffer can take the next strip row's block now
        named_barrier_sync(2, kMgRepackThreads);
        prefetch_next_item();
        mbar_wait(a_empty, ae_phase ^ 1);   // the UMMAs of the previous row of tiles have read sA
        ae_phase ^= 1;
#pragma unroll
        for (int ch = 0; ch < 8; ++ch)
          *reinterpret_cast<uint4*>(sA + row * 128 + ((ch ^ (row & 7)) << 4)) =
              make_uint4(w[4 * ch], w[4 * ch + 1], w[4 * ch + 2], w[4 * ch + 3]);
        fence_proxy_async_smem();  // generic-proxy smem writes -> visible to the tensor core (async proxy)
        mbar_arrive(a_full);
      }
    }
  } else if (warp == 9) {
    if (lane == 0 && lo < hi) {
      // ===================== MMA issuer =====================
      constexpr uint32_t idesc = make_idesc(ab_format16<F16>(), kMgBM, kMgBN, 0, 1);
      MergeCursor c;
      c.init(tab, info, n_entries, lo);
      int acc = 0;
      uint32_t acc_phase = 0, af_phase = 0, b_phases = 0;
      const uint32_t sAu = smem_u32(sA), sBu = smem_u32(sBt);
      for (int tile = lo; tile < hi; ++tile) {
        c.seek(tile, lo, hi - 1);
        const int ksteps = (c.e->r + 15) >> 4;
        if (c.b_first_use) {
          mbar_wait(&b_full[c.j], (b_phases >> c.j) & 1u);
          b_phases ^= 1u << c.j;
        }
        if (c.new_item) {
          mbar_wait(a_full, af_phase);
          af_phase ^= 1;
        }
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t sB = sBu + c.j * kMgBBytes;
        for (int k = 0; k < ksteps; ++k) {
          const uint64_t ad = make_smem_desc(sAu + k * 32, 16, 1024);
          const uint64_t bd = make_smem_desc(sB + k * 2048, 8192, 1024);
          umma_bf16(tmem_base + acc * kMgBN, ad, bd, idesc, k > 0 ? 1u : 0u);
        }
        umma_commit(&tfull_bar[acc]);
        // sA / the B tiles may be overwritten once the UMMAs issued so far are done
        if (c.last_of_item) umma_commit(a_empty);
        if (c.b_last_use) umma_commit(&b_empty[c.j]);
        if (++acc == kMgAcc) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    }
  } else if (warp >= 14) {
    // ===================== store group =====================
    // Plain coalesced 16-byte stores (each warp instruction writes 2 rows x 256 contiguous bytes); measured 1-2 %
    // faster than a TMA store of the same tile, and it takes the write-back off the TMA unit that feeds the loads.
    if (lo < hi) {
      const int st = threadIdx.x - 448;          // 0..127
      const int sw = st >> 5;
      const int sub = lane >> 4;                 // which of the 2 rows of this warp instruction
      const int chunk16 = lane & 15;             // 16-byte chunk inside the 256-byte tile row
      const int half = chunk16 >> 3, ch = chunk16 & 7;
      MergeCursor c;
      c.init(tab, info, n_entries, lo);
      int slot = 0;
      uint32_t phase = 0;
      for (int tile = lo; tile < hi; ++tile) {
        c.seek(tile, lo, hi - 1);
        const MergeInfo* e = c.e;
        const uint8_t* sW = smem + slot * kMgSlotBytes + half * 16384;
        const int col = c.n0 + chunk16 * 8;
        const bool col_ok = col < e->out;        // out % 8 == 0: a 16-byte chunk never straddles the edge
        const int rows = min(kMgBM, e->in - c.m0);
        __nv_bfloat16* gbase = e->W + static_cast<int64_t>(c.m0) * e->out + col;
        mbar_wait(&wready_bar[slot], phase);
        if (st == 0) stamp(tile - lo, 6);
#pragma unroll
        for (int b = 0; b < 2; ++b) {
          uint4 v[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int row = ((b * 8 + i) * 4 + sw) * 2 + sub;
            v[i] = *reinterpret_cast<const uint4*>(sW + row * 128 + ((ch ^ (row & 7)) << 4));
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int row = ((b * 8 + i) * 4 + sw) * 2 + sub;
            if (col_ok && row < rows) {
              uint4* dst = reinterpret_cast<uint4*>(gbase + static_cast<int64_t>(row) * e->out);
              *dst = v[i];
            }
          }
        }
        if (st == 0) stamp(tile - lo, 7);
        mbar_arrive(&empty_bar[slot]);           // this thread's part of the slot is in registers / on its way
        if (++slot == kMgSlots) {
          slot = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp < 8) {
    // ===================== epilogue group =====================
    if (lo < hi) {
      const int q = warp & 3;            // TMEM lane quarter this warp may read
      const int half = warp >> 2;        // 64-column half of the tile (= one TMA box of the W slot)
      const int row = q * 32 + lane;
      MergeCursor c;
      c.init(tab, info, n_entries, lo);
      int slot = 0, acc = 0;
      uint32_t phase = 0, acc_phase = 0;
      float scale = 0.f;
      bool has_prev = false;
      for (int tile = lo; tile < hi; ++tile) {
        c.seek(tile, lo, hi - 1);
        if (c.entry_changed) {
          scale = c.e->scale;
          has_prev = c.e->has_prev != 0;
        }
        uint8_t* box = smem + slot * kMgSlotBytes + half * 16384 + row * 128;
        if (threadIdx.x == 0) stamp(tile - lo, 2);
        mbar_wait(&tfull_bar[acc], acc_phase);
        tc_fence_after();
        if (threadIdx.x == 0) stamp(tile - lo, 3);
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * kMgBN + half * 64;
        uint32_t v0[32], v1[32];
        tmem_ld32(taddr, v0);
        tmem_ld32(taddr + 32, v1);
        mbar_wait(&full_bar[slot], phase);  // W tile landed (acquire on the TMA barrier)
        if (threadIdx.x == 0) stamp(tile - lo, 4);
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive(&tempty_bar[acc]);      // accumulator is in registers: hand the TMEM stage back
#pragma unroll
        for (int ch = 0; ch < 8; ++ch) {
          uint4* p = reinterpret_cast<uint4*>(box + ((ch ^ (row & 7)) << 4));
          float f[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) f[j] = scale * __uint_as_float(ch < 4 ? v0[ch * 8 + j] : v1[(ch - 4) * 8 + j]);
          if (has_prev) {
            const uint4 old = *p;
            const uint32_t ow[4] = {old.x, old.y, old.z, old.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              f[2 * j] += lo16_to_f32<F16>(ow[j]);
              f[2 * j + 1] += hi16_to_f32<F16>(ow[j]);
            }
          }
          uint4 pk;
          pk.x = pack16x2<F16>(f[0], f[1]);
          pk.y = pack16x2<F16>(f[2], f[3]);
          pk.z = pack16x2<F16>(f[4], f[5]);
          pk.w = pack16x2<F16>(f[6], f[7]);
          *p = pk;
        }
        fence_proxy_async_smem();
        mbar_arrive(&wready_bar[slot]);
        if (threadIdx.x == 0) stamp(tile - lo, 5);
        if (++slot == kMgSlots) {
          slot = 0;
          phase ^= 1;
        }
        if (++acc == kMgAcc) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 9) tmem_dealloc(tmem_base, kMgTmemCols);
  if (dbg_ts != nullptr && threadIdx.x == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    dbg_ts[2048 + 2 * blockIdx.x + 1] = static_cast<long long>(t);
  }
}

// ------------------------------------------------------------------------------------------------
// fp32 variant (fp32 modules: the reference's GLUE fine-tunes keep W, A, B in fp32, run_glue.py:386-388; sow.py:131-153
// then accumulates in fp32).  Exact fp32 FMA on the CUDA cores: 2r flop per 8 bytes is far below the fp32 roof at the
// ranks those configs use (r = 8), and the merged W matches an fp32 evaluation to rounding -- a bf16 tensor-core product
// would cost the pretrained weights 16 mantissa bits at every merge.  One launch for all matrices: 32 x 128 tiles,
// thread = 4 rows x 4 columns (float4), A / B tiles staged in shared memory.
// ------------------------------------------------------------------------------------------------
struct MergeF32Entry {
  float* W;
  const float* W_prev;   // nullptr: first merge
  const float* A;        // (in, r)
  const float* B;        // (r, out)
  int in, out, r;
  float scale;
  int n_tiles;           // column tiles of 128
  int tile_begin;
};
constexpr int kMfBM = 32, kMfBN = 128, kMfMaxR = 64;

__global__ void __launch_bounds__(256)
sow_merge_f32_kernel(const MergeF32Entry* __restrict__ tab, int n_entries, int total_tiles) {
  __shared__ float sA[kMfBM][kMfMaxR + 1];
  __shared__ __align__(16) float sB[kMfMaxR][kMfBN];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;     // tx: float4 column group, ty: 4-row group
  for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
    int lo = 0, hi = n_entries - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (tab[mid].tile_begin <= tile) lo = mid; else hi = mid - 1;
    }
    const MergeF32Entry e = tab[lo];
    const int local = tile - e.tile_begin;
    const int m0 = (local / e.n_tiles) * kMfBM, n0 = (local % e.n_tiles) * kMfBN;
    for (int r0 = 0; r0 < e.r; r0 += kMfMaxR) {
      const int rc = min(kMfMaxR, e.r - r0);
      __syncthreads();
      for (int i = threadIdx.x; i < kMfBM * rc; i += 256) {
        const int row = i / rc, k = i % rc;
        sA[row][k] = (m0 + row < e.in) ? e.A[static_cast<int64_t>(m0 + row) * e.r + r0 + k] : 0.f;
      }
      for (int i = threadIdx.x; i < rc * kMfBN; i += 256) {
        const int k = i / kMfBN, col = i % kMfBN;
        sB[k][col] = (n0 + col < e.out) ? e.B[static_cast<int64_t>(r0 + k) * e.out + n0 + col] : 0.f;
      }
      __syncthreads();
      float acc[4][4];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
      for (int k = 0; k < rc; ++k) {
        const float4 b = *reinterpret_cast<const float4*>(&sB[k][tx * 4]);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float a = sA[ty * 4 + i][k];
          acc[i][0] = fmaf(a, b.x, acc[i][0]);
          acc[i][1] = fmaf(a, b.y, acc[i][1]);
          acc[i][2] = fmaf(a, b.z, acc[i][2]);
          acc[i][3] = fmaf(a, b.w, acc[i][3]);
        }
      }
      const int col = n0 + tx * 4;
      const bool vec = (e.out & 3) == 0 && col + 3 < e.out;
      const float* prev = (r0 == 0) ? e.W_prev : e.W;       // later rank chunks accumulate onto what this launch wrote
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int row = m0 + ty * 4 + i;
        if (row >= e.in) continue;
        const int64_t off = static_cast<int64_t>(row) * e.out + col;
        if (vec) {
          float4 w = make_float4(0.f, 0.f, 0.f, 0.f);
          if (prev != nullptr) w = *reinterpret_cast<const float4*>(prev + off);
          w.x = fmaf(e.scale, acc[i][0], w.x);
          w.y = fmaf(e.scale, acc[i][1], w.y);
          w.z = fmaf(e.scale, acc[i][2], w.z);
          w.w = fmaf(e.scale, acc[i][3], w.w);
          *reinterpret_cast<float4*>(e.W + off) = w;
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (col + j < e.out) e.W[off + j] = fmaf(e.scale, acc[i][j], prev != nullptr ? prev[off + j] : 0.f);
        }
      }
    }
  }
}

}  // namespace sowb

using namespace sowb;

// Host -> device upload of a descriptor table without blocking the host: the table is copied into one of a few cached
// PINNED staging buffers and sent with a truly asynchronous cudaMemcpyAsync (a pageable source of more than 64 KB makes
// the "async" copy synchronise the calling thread with the stream, and is illegal during stream capture).  A slot is
// reused only after the copy that last read it has completed (event per slot).
namespace {
struct PinnedRing {
  static constexpr int kSlots = 4;
  void* buf[kSlots] = {nullptr, nullptr, nullptr, nullptr};
  size_t cap[kSlots] = {0, 0, 0, 0};
  cudaEvent_t ev[kSlots] = {nullptr, nullptr, nullptr, nullptr};
  int next = 0;
  std::mutex mu;
};
PinnedRing g_ring;

int upload_table(void* dst_dev, const void* src_host, size_t bytes, cudaStream_t stream) {
  std::lock_guard<std::mutex> lk(g_ring.mu);
  const int s = g_ring.next;
  g_ring.next = (g_ring.next + 1) % PinnedRing::kSlots;
  if (g_ring.ev[s] == nullptr) SOWB_CHECK_CUDA(cudaEventCreateWithFlags(&g_ring.ev[s], cudaEventDisableTiming));
  else SOWB_CHECK_CUDA(cudaEventSynchronize(g_ring.ev[s]));
  if (g_ring.cap[s] < bytes) {
    if (g_ring.buf[s] != nullptr) SOWB_CHECK_CUDA(cudaFreeHost(g_ring.buf[s]));
    g_ring.buf[s] = nullptr;
    g_ring.cap[s] = 0;
    const size_t want = std::max(bytes, size_t(256) << 10);
    SOWB_CHECK_CUDA(cudaHostAlloc(&g_ring.buf[s], want, cudaHostAllocDefault));
    g_ring.cap[s] = want;
  }
  memcpy(g_ring.buf[s], src_host, bytes);
  SOWB_CHECK_CUDA(cudaMemcpyAsync(dst_dev, g_ring.buf[s], bytes, cudaMemcpyHostToDevice, stream));
  SOWB_CHECK_CUDA(cudaEventRecord(g_ring.ev[s], stream));
  return SOWB_OK;
}
}  // namespace

static long long* g_merge_ts = nullptr;   // debug timeline buffer (device), see sow_merge_debug_timeline

extern "C" {

// Debug aid (not part of the product ABI): device buffer of 256*8 int64 that CTA 0 of the next merge launches
// fills with clock64 stamps per tile; pass NULL to switch off.
int sow_merge_debug_timeline(void* buf) {
  g_merge_ts = static_cast<long long*>(buf);
  return SOWB_OK;
}

size_t sow_merge_table_stride(void) {
  // one device entry per 64-wide rank chunk; callers size the table for ceil(r/64) chunks per layer
  static_assert(sizeof(MergeF32Entry) <= sizeof(MergeDevEntry), "the fp32 table fits the same stride");
  return sizeof(MergeDevEntry);
}

static int merge_grouped_f32(const sowb_merge_entry* entries, int n, void* table_dev, size_t table_bytes, cudaStream_t stream) {
  if (table_bytes < size_t(n) * sizeof(MergeF32Entry))
    return set_error(SOWB_EWORKSPACE, "sow_merge_grouped: table %zu B < required %zu B", table_bytes, size_t(n) * sizeof(MergeF32Entry));
  std::vector<MergeF32Entry> host(n);
  int tiles = 0;
  double bytes = 0;
  for (int i = 0; i < n; ++i) {
    const sowb_merge_entry& e = entries[i];
    SOWB_REQUIRE(e.W && e.A && e.B, "sow_merge_grouped: entry %d has a null W/A/B pointer", i);
    SOWB_REQUIRE(e.in > 0 && e.out > 0 && e.r > 0, "sow_merge_grouped: entry %d has a non-positive dimension", i);
    MergeF32Entry& d = host[i];
    d.W = static_cast<float*>(e.W);
    d.W_prev = static_cast<const float*>(e.W_prev);
    d.A = static_cast<const float*>(e.A);
    d.B = static_cast<const float*>(e.B);
    d.in = e.in;
    d.out = e.out;
    d.r = e.r;
    d.scale = e.scale;
    d.n_tiles = ceil_div(e.out, kMfBN);
    d.tile_begin = tiles;
    tiles += ceil_div(e.in, kMfBM) * d.n_tiles;
    bytes += 4.0 * e.in * e.out * (1 + (e.W_prev != nullptr)) + 4.0 * e.r * (double(e.in) + e.out);
  }
  if (int rcu = upload_table(table_dev, host.data(), size_t(n) * sizeof(MergeF32Entry), stream)) return rcu;
  const int grid = std::min(tiles, num_sms() * 8);
  ProfileScope prof(stream, PROF_MERGE, bytes);
  sow_merge_f32_kernel<<<grid, 256, 0, stream>>>(static_cast<const MergeF32Entry*>(table_dev), n, tiles);
  SOWB_CHECK_CUDA(cudaGetLastError());
  return SOWB_OK;
}

int sow_merge_grouped(const sowb_merge_entry* entries, int n, int dtype, void* table_dev, size_t table_bytes,
                      void* stream_) {
  if (n <= 0) return SOWB_OK;
  if (dtype != SOWB_BF16 && dtype != SOWB_F32 && dtype != SOWB_F16) return set_error(SOWB_EINVAL, "sow_merge_grouped: unknown dtype %d", dtype);
  SOWB_REQUIRE(entries != nullptr && table_dev != nullptr, "sow_merge_grouped: null pointer argument");
  if (int rc0 = ensure_context_for(table_dev)) return rc0;
  if (dtype == SOWB_F32) {
    int rcf = require_sm100();
    if (rcf) return rcf;
    return merge_grouped_f32(entries, n, table_dev, table_bytes, static_cast<cudaStream_t>(stream_));
  }
  SOWB_REQUIRE((reinterpret_cast<uintptr_t>(table_dev) & 127) == 0, "sow_merge_grouped: table_dev must be 128-byte aligned");
  int rc = require_sm100();
  if (rc) return rc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const bool f16 = dtype == SOWB_F16;
  const CUtensorMapDataType t16 = map_type16(f16);
  auto kernel = f16 ? sow_merge_kernel<true> : sow_merge_kernel<false>;
  int max_chunks = 1;
  for (int i = 0; i < n; ++i) {
    const sowb_merge_entry& e = entries[i];
    SOWB_REQUIRE(e.W && e.A && e.B, "sow_merge_grouped: entry %d has a null W/A/B pointer", i);
    SOWB_REQUIRE(e.in > 0 && e.out > 0 && e.r > 0, "sow_merge_grouped: entry %d has a non-positive dimension", i);
    SOWB_REQUIRE(e.out % 8 == 0, "sow_merge_grouped: entry %d: out=%d must be a multiple of 8", i, e.out);
    max_chunks = std::max(max_chunks, ceil_div(e.r, 64));
  }
  if (table_bytes < size_t(n) * sizeof(MergeDevEntry))
    return set_error(SOWB_EWORKSPACE, "sow_merge_grouped: table %zu B < required %zu B", table_bytes,
                     size_t(n) * sizeof(MergeDevEntry));
  SOWB_CHECK_CUDA(set_max_smem_once(kernel, size_t(kMgSmemTotal)));
  const int sms = num_sms();
  // ranks above 64 are applied as successive 64-wide chunks (W_prev = W after the first chunk)
  for (int chunk = 0; chunk < max_chunks; ++chunk) {
    std::vector<MergeDevEntry> host;
    host.reserve(n);
    for (int i = 0; i < n; ++i) {
      const sowb_merge_entry& e = entries[i];
      const int r0 = chunk * 64;
      if (r0 >= e.r) continue;
      MergeDevEntry d;
      memset(&d, 0, sizeof(d));
      const void* prev = (chunk == 0) ? e.W_prev : e.W;
      d.has_prev = prev != nullptr;
      rc = make_tensor_map_2d(&d.tmWout, e.W, e.out, e.in, uint64_t(e.out) * 2, 64, kMgBM, t16);
      if (rc) return rc;
      d.tmWin = d.tmWout;
      if (prev != nullptr && prev != e.W) {
        rc = make_tensor_map_2d(&d.tmWin, prev, e.out, e.in, uint64_t(e.out) * 2, 64, kMgBM, t16);
        if (rc) return rc;
      }
      const int rc_rows = std::min(64, e.r - r0);
      const __nv_bfloat16* Bp = static_cast<const __nv_bfloat16*>(e.B) + size_t(r0) * e.out;
      rc = make_tensor_map_2d(&d.tmB, Bp, e.out, rc_rows, uint64_t(e.out) * 2, 64, 64, t16);
      if (rc) return rc;
      d.A = static_cast<const __nv_bfloat16*>(e.A) + r0;
      d.W = static_cast<__nv_bfloat16*>(e.W);
      d.lda = e.r;
      d.in = e.in;
      d.out = e.out;
      d.r = rc_rows;
      d.scale = e.scale;
      d.m_tiles = ceil_div(e.in, kMgBM);
      d.n_tiles = ceil_div(e.out, kMgBN);
      // bulk-copy staging of A needs contiguous, 16-byte aligned blocks whose length is a multiple of 16 bytes
      d.a_bulk = (e.r <= 64) && ((reinterpret_cast<uintptr_t>(e.A) & 15) == 0) &&
                 (((e.in % kMgBM) * e.r) % 8 == 0);
      host.push_back(d);
    }
    if (host.empty()) break;
    // the device table holds at most kMgMaxEntries entries per launch
    for (size_t first = 0; first < host.size(); first += kMgMaxEntries) {
      const size_t cnt = std::min(host.size() - first, size_t(kMgMaxEntries));
      int tiles = 0;
      double bytes = 0;   // algorithmic: W read (if any) + W write + A + B (SURVEY.md 8d)
      for (size_t j = first; j < first + cnt; ++j) {
        MergeDevEntry& d = host[j];
        d.tile_begin = tiles;
        tiles += d.m_tiles * d.n_tiles;
        bytes += 2.0 * d.in * d.out * (1 + d.has_prev) + 2.0 * d.r * (double(d.in) + d.out);
      }
      // stream-ordered: an earlier launch on this stream that still reads the table finishes before this copy
      rc = upload_table(table_dev, host.data() + first, cnt * sizeof(MergeDevEntry), stream);
      if (rc) return rc;
      const int grid = tiles < sms ? tiles : sms;
      ProfileScope prof(stream, PROF_MERGE, bytes);
      static const int prefetch = []() {
        const char* e = getenv("SOWB_MERGE_PREFETCH");   // tuning knob: tiles of L2 prefetch distance (0 = off)
        return e ? atoi(e) : kMgPrefetchDefault;
      }();
      kernel<<<grid, kMgThreads, kMgSmemTotal, stream>>>(static_cast<const MergeDevEntry*>(table_dev), static_cast<int>(cnt),
                                                         tiles, prefetch, g_merge_ts);
      SOWB_CHECK_CUDA(cudaGetLastError());
    }
  }
  return SOWB_OK;
}

}  // extern "C"
