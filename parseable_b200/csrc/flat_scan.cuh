// The flat scan kernels: decode -> predicate -> (selection bitmap | group-by accumulation) over the
// flat store (flat_store.cuh).  Same operator chain of the reference as k_scan
//   DataSourceExec(Parquet) -> FilterExec -> AggregateExec(Partial)
// (/root/reference/src/query/mod.rs:287; SURVEY.md §8 rows a10-a12), for the common case: every
// referenced column of a work item has pages with a flat copy (pages with NULLs carry a validity
// bitmap and one slot per ROW; a column missing from a file reads as all NULL).  A file whose value
// streams the flattener refuses is refused as corrupt at table open (PQB_FLAT_LENIENT keeps such
// pages on k_scan for debugging).
//
// Shape (both kernels): persistent CTAs, one PRODUCER warp and N consumer warps.  The producer's
// elected lane pulls work items from the queue, and for every slab of an item stages the slab's
// bytes of every referenced column with one TMA bulk copy per column (cp.async.bulk -> mbarrier
// complete_tx) into a ring of shared-memory stages; it runs up to `nstages` slabs ahead, across item
// boundaries.  Consumers wait on the stage's `full` mbarrier, work out of shared memory and hand the
// stage back through its `empty` mbarrier.  No block barrier inside the loop, no run directory, no
// header walk: value i of a page is bits [i*bw, (i+1)*bw).
//
// k_flat_filter<CONJ>: 4 consumer warps; a STAGE IS ONE WARP'S SLAB (2048 rows) and a consumer warp
//   draws the next stage in fill order with a shared-memory ticket, so no warp waits for a slower one
//   and the ring is 8-16 stages deep.  A thread owns two words of the selection bitmap per slab (32
//   consecutive rows each), evaluated by one rolled copy of the leaf code.  First leaf: all 32 indices
//   unpacked with compile-time shifts; a dictionary of <= 32 entries keeps its whole LUT in ONE REGISTER
//   (3 instructions per row: extract, rotate, funnel).  Later leaves of a conjunction run only on the
//   surviving rows.  HBM traffic = encoded bytes once + 1 bit per row.
// k_flat_agg<KR>: 31 consumer warps, one CTA per SM so that the hot part of the accumulator table
//   (group slots < plan.hot_slots; group ids are numbered hot-first; the very hottest own a cell per
//   lane) lives in shared memory next to the stages, in cells as narrow as their updates allow; cold
//   slots go to L2 with fire-and-forget reductions.  Rows are dealt to threads interleaved (lane L of a warp takes row base + L):
//   neighbouring lanes share their index words, and 8-byte values are read in place from the flat
//   store, fully coalesced.  Every pointer stays in ONE address space (a pointer that may be shared or
//   global makes every access through it generic: that cost 20-25 % on both kernels before it was
//   found in the SASS).
#pragma once
#include <cuda_runtime.h>

#include <type_traits>

#include "decode_core.cuh"
#include "device_structs.hpp"
#include "flat_store.cuh"
#include "ptx_utils.cuh"
#include "scan_kernel.cuh"   // acc_add / acc_apply / acc_merge

namespace pqb {

constexpr int kFlatStagesMax = 16;
constexpr int kFilterConsumerWarps = 4;
#ifndef PQB_WAIT_HINT
#define PQB_WAIT_HINT 0
#endif
#ifndef PQB_FILTER_ROLL
#define PQB_FILTER_ROLL 1   // 0: the two words of a thread unrolled (two copies of every leaf routine)
#endif
#ifndef PQB_FILTER_ILP
#define PQB_FILTER_ILP 1   // 0: the serial funnel chain / one survivor per trip (A/B builds: make EXTRA=-DPQB_FILTER_ILP=0)
#endif
#ifndef PQB_FILTER_WORDS
#define PQB_FILTER_WORDS 2
#endif
constexpr int kFilterWords = PQB_FILTER_WORDS;                     // 32-row bitmap words per consumer thread per slab
constexpr int kFilterThreads = 32 * (kFilterConsumerWarps + 1);
constexpr int kFilterSlabRows = 32 * 32 * kFilterWords;   // 2048: one WARP's slab (k_flat_filter's stages are taken warp by warp)
constexpr int kAggThreads = 1024;
constexpr int kAggConsumers = kAggThreads - 32;

struct FlatLayout {              // dynamic shared memory of the flat kernels (byte offsets), computed on the host
  uint32_t nstages;
  uint32_t stage_bytes;
  uint32_t stage0;               // first stage buffer
  uint32_t meta0, meta_stride;   // FlatStage records, one per stage, holding only the referenced columns
  uint32_t col_off[kMaxCols];    // values of column c inside a stage (16-byte aligned)
  uint32_t col_voff[kMaxCols];   // validity bits of column c inside a stage (columns that may hold NULLs)
  uint32_t acc;                  // hot accumulator table (k_flat_agg)
  uint32_t total;
};

constexpr uint32_t kColHasValid = 1u, kColAbsent = 2u, kColDirect = 4u;
struct FlatStageCol {
  uint64_t dict8;                // flat-store offset of the aligned numeric dictionary (~0: none)
  uint32_t bw;                   // bits per value (FK_PLAIN8: 64, FK_BITS: 1)
  uint32_t fkind;                // FlatKind
  uint32_t lut_base;
  uint32_t dict_n;
  uint32_t phase;                // bit of the staged bytes where row 0 of the slab starts (a piece may start inside a
                                 // page at a row that is not a multiple of 128: the copy starts at the 16 bytes below)
  uint32_t vphase;               // the same for the validity bits
  uint32_t flags;                // kColHasValid: the page holds NULLs (validity staged); kColAbsent: column missing from the file
  uint32_t _pad;
};
struct FlatStage {
  uint32_t item;                 // 0xffffffff: the queue is empty, consumers leave
  uint32_t R;                    // rows of this slab
  uint32_t r0;                   // first row of the slab inside the item
  uint32_t bitmap_word0;
  uint32_t regmask;              // bit l: leaf l's whole LUT is lutreg[l] (dictionary of <= 32 entries, index width <= 5)
  uint32_t lutreg[kMaxLeaves];   // periodic with 2^bw, so the bits above the index never matter
  FlatStageCol col[kMaxCols];
};
struct FlatCtl {
  uint64_t full[kFlatStagesMax];
  uint64_t empty[kFlatStagesMax];
  uint32_t ticket;               // k_flat_filter: the next stage (in fill order) nobody has taken yet
  uint32_t _pad[3];
};
// stage record s (the col[] tail is allocated for plan.ncols columns only: L.meta_stride)
__device__ __forceinline__ FlatStage& flat_stage(uint8_t* smem, const FlatLayout& L, uint32_t s) {
  return *reinterpret_cast<FlatStage*>(smem + L.meta0 + s * L.meta_stride);
}

__device__ __forceinline__ uint32_t flat_col_bytes(uint32_t phase, uint32_t bw, uint32_t rows) {
  const uint32_t nb = (phase + rows * bw + 7u) >> 3;
  return (nb + 15u) & ~15u;
}

// ---- producer: one warp; lane 0 owns the queue, the barriers and the TMA copies ------------------
// Wait with a real back-off.  mbarrier.try_wait's suspend-time hint does not park the thread for long: ptxas turns it
// into a four-instruction TRYWAIT / NANOSLEEP.SYNCS loop, and a waiting warp -- the producer waits for a free stage
// most of its life -- ran that loop 10^8 times per launch: 15-18 % of all executed instructions, taken from the
// scheduler it shares with seven or eight working warps (profiles/k_flat_agg_r2b, k_flat_filter_r2b).
__device__ __forceinline__ void mbar_wait_spin(uint64_t* bar, uint32_t parity, uint32_t max_ns) {
#if PQB_WAIT_HINT
  while (!mbar_try_wait_hint(bar, parity, 100000u)) {}   // A/B: the hint-only wait
  return;
#endif
  if (mbar_try_wait(bar, parity)) return;
  uint32_t ns = 64;
  do {
    __nanosleep(ns);
    if (ns < max_ns) ns <<= 1;
  } while (!mbar_try_wait(bar, parity));
}

// `takers`: how many consumers must see the end-of-queue record (k_flat_agg: 1, every warp reads every stage;
// k_flat_filter: one per consumer warp, every warp takes stages of its own)
__device__ __noinline__ void flat_producer(const DevPlan& plan, const FlatLayout& L, const DevScanArgs& a, FlatCtl& ctl,
                                           uint8_t* smem, uint32_t S, uint32_t takers, uint32_t wait_ns) {
  const uint32_t lane = threadIdx.x & 31;
  uint32_t stage = 0, par = 1;   // parity the next wait on empty[stage] needs; a fresh barrier counts as released
  const uint32_t ncols = plan.ncols;
  for (;;) {
    uint32_t id = 0;
    if (lane == 0) id = (uint32_t)atomicAdd(&a.counters[2], 1ull);
    id = __shfl_sync(0xffffffffu, id, 0);
    if (id >= plan.n_items) break;
    const DevItem& item = a.items[id];
    if (!(item.fast & kItemFlat)) continue;
    const uint32_t rg = item.rg;
    if (a.rg_live && !a.rg_live[rg]) continue;
    // lane c looks after column slot c
    FlatStageCol mycol{};
    uint64_t mysrc = 0, myvsrc = 0;
    uint32_t mypoff = 0;
    if (lane < ncols) {
      const DevChunk& ch = a.chunks[rg * ncols + lane];
      mycol.dict8 = ch.dict8_off;
      mycol.lut_base = ch.lut_base;
      mycol.dict_n = ch.dict_n;
      if ((item.absent >> lane) & 1u) {
        mycol.flags = kColAbsent;
        mycol.fkind = FK_NONE;
      } else {
        const FlatPageRec fp = a.fpages[item.page[lane]];
        mycol.bw = fp.bw;
        mycol.fkind = fp.fkind;
        if (fp.fkind == FK_BYTES) mycol.dict8 = fp.base;   // PLAIN byte arrays: arena offset of the page's values section
        mysrc = fp.off;
        mypoff = item.poff[lane];
        if (fp.voff != ~0ull) { mycol.flags = kColHasValid; myvsrc = fp.voff; }
      }
    }
    // register LUTs of this item's row group: every lane fetches one LUT byte, one ballot per leaf
    uint32_t regmask = 0, mylut = 0;
    for (uint32_t l = 0; l < plan.nleaves; l++) {
      const DevLeaf& lf = plan.leaves[l];
      const uint32_t bw = __shfl_sync(0xffffffffu, mycol.bw, lf.col), fk = __shfl_sync(0xffffffffu, mycol.fkind, lf.col);
      const uint32_t dn = __shfl_sync(0xffffffffu, mycol.dict_n, lf.col), lb = __shfl_sync(0xffffffffu, mycol.lut_base, lf.col);
      if (!((lf.kind == LK_CMP || lf.kind == LK_LIKE) && fk == FK_INDEX && bw <= 5 && dn <= 32)) continue;
      const uint8_t* lut = a.luts + lf.lut_off + lb;
      uint32_t r = __ballot_sync(0xffffffffu, lane < dn && lut[lane] != 0);
      for (uint32_t p = 1u << bw; p < 32; p <<= 1) r |= r << p;
      if (lane == l) mylut = r;
      regmask |= 1u << l;
    }
    const uint32_t nrows = item.nrows, bm0 = item.bitmap_word0;
    const bool staged = lane < ncols && plan.cols[lane].staged && !(mycol.flags & kColAbsent);
    for (uint32_t r0 = 0; r0 < nrows; r0 += S) {
      const uint32_t R = nrows - r0 < S ? nrows - r0 : S;
      if (lane == 0) mbar_wait_spin(&ctl.empty[stage], par, wait_ns);
      __syncwarp();
      FlatStage& st = flat_stage(smem, L, stage);
      // first bit of the slab in the page's flat copy; the copy starts at the 16-byte boundary below it
      const uint64_t bit0 = uint64_t(mypoff + r0) * mycol.bw, vbit0 = uint64_t(mypoff) + r0;
      mycol.phase = uint32_t(bit0 & 127u);
      mycol.vphase = uint32_t(vbit0 & 127u);
      // a column that is only projected is not staged: the gather after the scan reads its selected rows
      // plan.direct8 (k_flat_agg): 8-byte values are not staged -- a thread reads its rows' values straight from the flat
      // store (row-interleaved threads: fully coalesced, each value used once); dict8 then carries where row 0 of the slab is
      const bool direct = plan.direct8 && mycol.fkind == FK_PLAIN8;
      const uint32_t nb = (staged && !direct) ? flat_col_bytes(mycol.phase, mycol.bw, R) : 0u;
      const uint32_t vnb = (staged && (mycol.flags & kColHasValid)) ? flat_col_bytes(mycol.vphase, 1, R) : 0u;
      if (lane < ncols) {
        FlatStageCol sc = mycol;
        if (direct) { sc.dict8 = mysrc + uint64_t(mypoff + r0) * 8; sc.flags |= kColDirect; sc.phase = 0; }
        st.col[lane] = sc;
      }
      if (lane < plan.nleaves) st.lutreg[lane] = mylut;
      uint32_t bytes = nb + vnb;
      for (int o = 16; o; o >>= 1) bytes += __shfl_xor_sync(0xffffffffu, bytes, o);
      if (lane == 0) {
        st.item = id;
        st.R = R;
        st.r0 = r0;
        st.bitmap_word0 = bm0;
        st.regmask = regmask;
      }
      __syncwarp();
      if (lane == 0) mbar_arrive_expect_tx(&ctl.full[stage], bytes);
      __syncwarp();
      uint8_t* base = smem + L.stage0 + stage * L.stage_bytes;
      if (nb) tma_load_1d(base + L.col_off[lane], a.flat + mysrc + ((bit0 >> 7) << 4), nb, &ctl.full[stage]);
      if (vnb) tma_load_1d(base + L.col_voff[lane], a.flat + myvsrc + ((vbit0 >> 7) << 4), vnb, &ctl.full[stage]);
      if (++stage == L.nstages) { stage = 0; par ^= 1u; }
    }
  }
  if (lane == 0) {
    for (uint32_t t = 0; t < takers; t++) {
      mbar_wait_spin(&ctl.empty[stage], par, wait_ns);
      flat_stage(smem, L, stage).item = 0xffffffffu;
      mbar_arrive(&ctl.full[stage]);
      if (++stage == L.nstages) { stage = 0; par ^= 1u; }
    }
  }
}

__device__ __forceinline__ void flat_ctl_init(FlatCtl& ctl, uint32_t nstages, uint32_t consumer_warps) {
  if (threadIdx.x == 0) {
    for (uint32_t s = 0; s < nstages; s++) {
      mbar_init(&ctl.full[s], 1);
      mbar_init(&ctl.empty[s], consumer_warps);   // arrivals that hand a stage back
    }
    ctl.ticket = 0;
    mbar_fence_init();
  }
}

// ---- one staged column of the current slab ------------------------------------------------------
struct ColCtx {
  const uint32_t* colw;      // staged values (shared memory): flat bits / 8-byte slots, whole words of the phase folded in
  const uint64_t* v8;        // 8-byte values of a PLAIN8 page: the staged ones, or (k_flat_agg) the flat store's in global memory.
                             // Two pointers so that neither ever mixes address spaces (a mixed one makes every load generic)
  const uint32_t* vw;        // validity bits (nullptr: every row valid, unless `absent`)
  uint32_t phase, vphase;    // remaining bit phases (0..31) of row 0
  uint32_t bw, mask, dict_max, fkind;
  bool absent;               // column missing from this file: every row NULL
};
template <bool DIRECT8>
__device__ __forceinline__ void col_ctx(ColCtx& c, const FlatStage& st, const uint8_t* base, const FlatLayout& L, uint32_t col,
                                        const uint8_t* flat) {
  const FlatStageCol& sc = st.col[col];
  c.colw = reinterpret_cast<const uint32_t*>(base + L.col_off[col]) + (sc.phase >> 5);
  if (DIRECT8) c.v8 = reinterpret_cast<const uint64_t*>(flat + sc.dict8);   // k_flat_agg: 8-byte values read in place (only used on PLAIN8 pages)
  else c.v8 = reinterpret_cast<const uint64_t*>(c.colw);
  c.phase = sc.phase & 31u;
  c.vw = (sc.flags & kColHasValid) ? reinterpret_cast<const uint32_t*>(base + L.col_voff[col]) + (sc.vphase >> 5) : nullptr;
  c.vphase = sc.vphase & 31u;
  c.bw = sc.bw;
  c.mask = sc.bw >= 32 ? 0xffffffffu : ((1u << sc.bw) - 1u);
  c.dict_max = sc.dict_n ? sc.dict_n - 1 : 0u;   // a corrupt index must not leave the LUT (the reference's reader errors out)
  c.fkind = sc.fkind;
  c.absent = (sc.flags & kColAbsent) != 0;
}
__device__ __forceinline__ uint32_t col_index(const ColCtx& c, uint32_t row) {
  uint32_t v = bits32_at(c.colw, c.phase + row * c.bw) & c.mask;   // bw == 0: mask == 0
  return v < c.dict_max ? v : c.dict_max;
}
// validity of 32 consecutive rows starting at `row` / of one row
__device__ __forceinline__ uint32_t col_valid32(const ColCtx& c, uint32_t row) {
  if (c.absent) return 0u;
  return c.vw ? bits32_at(c.vw, c.vphase + row) : 0xffffffffu;
}
__device__ __forceinline__ bool col_valid(const ColCtx& c, uint32_t row) {
  if (c.absent) return false;
  if (!c.vw) return true;
  const uint32_t b = c.vphase + row;
  return (c.vw[b >> 5] >> (b & 31)) & 1u;
}

// ---- leaves -------------------------------------------------------------------------------------
// Everything a consumer needs about one leaf for the CURRENT slab; built once per slab (warp uniform)
// so that the row loops below carry no interpretation: the switch on the page kind sits outside them.
enum LeafMode : uint32_t { LM_FALSE = 0, LM_TRUE = 1, LM_REGLUT = 2, LM_MEMLUT = 3, LM_PLAIN8 = 4, LM_BITS = 5, LM_BYTES = 6 };
struct LeafCtx {
  ColCtx c;
  const uint8_t* lut;        // this leaf's LUT bytes for the chunk (global); LM_BYTES: the page's values section instead
                             // (PLAIN byte arrays: [len][bytes]...)
  const DevLeaf* lf;         // LM_BYTES: string literal / cooked LIKE pattern live in the plan + literal pool
  const uint8_t* lit_pool;
  uint32_t lutreg;           // LM_REGLUT: the whole LUT, periodic with 2^bw
  uint32_t mode;             // LeafMode: the answer for a NON-NULL row
  uint32_t cmp;
  uint32_t lkind;            // DevLeafKind
  int64_t lit;               // literal (i64, bool 0/1, or f64 order key for DK_F64)
  bool f64;
};

template <bool DIRECT8>
__device__ __forceinline__ void leaf_ctx(LeafCtx& x, const DevPlan& plan, const DevScanArgs& a, const FlatStage& st,
                                         const uint8_t* stage_base, const FlatLayout& L, uint32_t l) {
  const DevLeaf& lf = plan.leaves[l];
  const uint32_t c = lf.col;
  const FlatStageCol& sc = st.col[c];
  col_ctx<DIRECT8>(x.c, st, stage_base, L, c, a.flat);
  x.cmp = lf.cmp;
  x.lkind = lf.kind;
  x.f64 = plan.cols[c].kind == DK_F64;
  x.lit = (x.f64 && lf.kind == LK_CMP) ? f64_order_key(uint64_t(lf.lit_i64)) : lf.lit_i64;
  x.lut = a.luts + lf.lut_off + sc.lut_base;
  x.lutreg = st.lutreg[l];
  x.lf = &lf;
  x.lit_pool = a.lit_pool;
  if (lf.kind == LK_IS_NULL || lf.kind == LK_IS_NOT_NULL || x.c.absent) x.mode = LM_FALSE;   // answered by the validity alone
  else if (sc.fkind == FK_BYTES) { x.mode = LM_BYTES; x.lut = a.arena + sc.dict8; }
  else if (sc.fkind == FK_INDEX) {
    if ((st.regmask >> l) & 1u) x.mode = LM_REGLUT;
    else if (sc.bw == 0) x.mode = __ldg(x.lut) ? LM_TRUE : LM_FALSE;   // one-entry dictionary: no bits at all
    else x.mode = LM_MEMLUT;
  } else x.mode = sc.fkind == FK_PLAIN8 ? LM_PLAIN8 : LM_BITS;
}

__device__ __forceinline__ bool plain_cmp(uint64_t bits, const LeafCtx& x) {
  const int64_t v = x.f64 ? f64_order_key(bits) : int64_t(bits);
  return cmp_i64(v, x.lit, x.cmp);
}

// the comparison for ONE non-NULL row; x.mode is warp uniform, so the switch costs one predictable branch
__device__ __forceinline__ bool leaf_row(const LeafCtx& x, uint32_t row) {
  switch (x.mode) {
    case LM_FALSE: return false;
    case LM_TRUE: return true;
    case LM_REGLUT: return (__funnelshift_r(x.lutreg, x.lutreg, bits32_at(x.c.colw, x.c.phase + row * x.c.bw)) & 1u) != 0;
    case LM_MEMLUT: return __ldg(x.lut + col_index(x.c, row)) != 0;
    case LM_PLAIN8: return plain_cmp(x.c.v8[row], x);
    case LM_BYTES: {
      // the string itself (no dictionary to answer for it): arrow-ord / arrow-string semantics on the raw bytes
      const uint8_t* sp = x.lut + bits32_at(x.c.colw, x.c.phase + row * 32);
      const uint32_t len = load_u32_unaligned(sp - 4);
      const uint8_t* needle = x.lit_pool + x.lf->str_off;
      if (x.lkind == LK_CMP) return cmp_result(cmp_bytes(sp, len, needle, x.lf->str_len), x.cmp);
      const bool t = like_match(sp, len, needle, x.lf->str_len, x.cmp, (x.lf->flags & 2u) != 0);
      return (x.lf->flags & 1u) ? !t : t;
    }
    default: {
      const uint32_t pb = x.c.phase + row;
      return cmp_i64(int64_t((x.c.colw[pb >> 5] >> (pb & 31)) & 1u), x.lit, x.cmp);
    }
  }
}
// SQL truth of the leaf for one row: 1 TRUE, 0 FALSE, 2 NULL
__device__ __forceinline__ uint32_t leaf_row3(const LeafCtx& x, uint32_t row) {
  const bool v = col_valid(x.c, row);
  if (x.lkind == LK_IS_NULL) return v ? 0u : 1u;
  if (x.lkind == LK_IS_NOT_NULL) return v ? 1u : 0u;
  if (!v) return 2u;
  return leaf_row(x, row) ? 1u : 0u;
}

// knock the rows of `m` (bit k = row row0 + k, all non-NULL) out that fail the comparison: one trip per surviving row
__device__ __forceinline__ uint32_t leaf_survivors(const LeafCtx& x, uint32_t row0, uint32_t m) {
  uint32_t mm = m;
  if (x.mode == LM_MEMLUT) {
    const uint32_t bit0 = x.c.phase + row0 * x.c.bw;
#if PQB_FILTER_ILP
    // two survivors per trip: their index extractions and LUT probes overlap (one trip is a chain of
    // shared load -> funnel -> global LUT byte)
    while (mm) {
      const uint32_t k0 = __ffs(mm) - 1;
      mm &= mm - 1;
      const uint32_t k1 = mm ? __ffs(mm) - 1 : k0;
      mm &= mm - 1;   // mm == 0 stays 0
      uint32_t v0 = bits32_at(x.c.colw, bit0 + k0 * x.c.bw) & x.c.mask, v1 = bits32_at(x.c.colw, bit0 + k1 * x.c.bw) & x.c.mask;
      v0 = v0 < x.c.dict_max ? v0 : x.c.dict_max;
      v1 = v1 < x.c.dict_max ? v1 : x.c.dict_max;
      const uint32_t t0 = __ldg(x.lut + v0), t1 = __ldg(x.lut + v1);   // the LUTs, dictionaries and id tables are global and read-only: LDG, not a generic load
      m &= ~((t0 ? 0u : 1u) << k0);
      m &= ~((t1 ? 0u : 1u) << k1);   // k1 == k0 when there was only one: same answer twice
    }
#else
    while (mm) {
      const uint32_t k = __ffs(mm) - 1;
      mm &= mm - 1;
      uint32_t v = bits32_at(x.c.colw, bit0 + k * x.c.bw) & x.c.mask;
      v = v < x.c.dict_max ? v : x.c.dict_max;
      if (!__ldg(x.lut + v)) m ^= 1u << k;
    }
#endif
    return m;
  }
  if (x.mode == LM_TRUE) return m;
  if (x.mode == LM_FALSE) return 0u;
  while (mm) {
    const uint32_t k = __ffs(mm) - 1;
    mm &= mm - 1;
    if (!leaf_row(x, row0 + k)) m ^= 1u << k;
  }
  return m;
}

// 32 consecutive indices of BW bits starting at word w[0] -> 32 LUT answers, bit k = value k
template <int BW, bool REGLUT>
__device__ __forceinline__ uint32_t leaf_dense_bw(const uint32_t* __restrict__ w, uint32_t lutreg, const uint8_t* __restrict__ lut,
                                                  uint32_t dict_max) {
  uint32_t x[BW + 1];
#pragma unroll
  for (int i = 0; i < BW; i++) x[i] = w[i];
  x[BW] = 0;
  constexpr uint32_t mask = BW >= 32 ? 0xffffffffu : ((1u << BW) - 1u);
#if PQB_FILTER_ILP
  // four independent chains of eight (values 8c .. 8c+7 end up in the top byte of q[c]): the 32-step funnel chain was
  // the longest dependency of the kernel (`wait` stalls in the profile), three PRMTs put the bytes together
  uint32_t q[4] = {0, 0, 0, 0};
#pragma unroll
  for (int k = 0; k < 32; k++) {
    const int bit = k * BW, wi = bit >> 5, sh = bit & 31;
    uint32_t v = (sh + BW <= 32) ? (x[wi] >> sh) : __funnelshift_r(x[wi], x[wi + 1], sh);
    uint32_t t;
    if (REGLUT) t = __funnelshift_r(lutreg, lutreg, v);
    else {
      v &= mask;
      v = v < dict_max ? v : dict_max;
      t = __ldg(lut + v);
    }
    q[k >> 3] = __funnelshift_r(q[k >> 3], t, 1);
  }
  const uint32_t lo = __byte_perm(q[0], q[1], 0x0073), hi = __byte_perm(q[2], q[3], 0x7300);
  return __byte_perm(lo, hi, 0x7610);
#else
  uint32_t m = 0;
#pragma unroll
  for (int k = 0; k < 32; k++) {
    const int bit = k * BW, wi = bit >> 5, sh = bit & 31;
    uint32_t v = (sh + BW <= 32) ? (x[wi] >> sh) : __funnelshift_r(x[wi], x[wi + 1], sh);
    uint32_t t;
    if (REGLUT) t = __funnelshift_r(lutreg, lutreg, v);   // rotate: bit 0 = LUT[v mod 32], the LUT is periodic with 2^BW
    else {
      v &= mask;
      v = v < dict_max ? v : dict_max;
      t = __ldg(lut + v);
    }
    m = __funnelshift_r(m, t, 1);                          // shift the answer in from the top: after 32 steps bit k = value k
  }
  return m;
#endif
}

// dense comparison of one leaf over the thread's 32 rows [32*tc, 32*tc + 32) (blocked mapping); NULL rows
// hold slot value 0 and are masked by the caller
__device__ __forceinline__ uint32_t leaf_dense(const LeafCtx& x, uint32_t tc, uint32_t R, uint32_t need) {
  switch (x.mode) {
    case LM_FALSE: return 0u;
    case LM_TRUE: return 0xffffffffu;
    case LM_BYTES: {   // only the rows in `need` (in range, not NULL: a NULL row owns no bytes)
      uint32_t m = 0, mm = need;
      while (mm) {
        const uint32_t k = __ffs(mm) - 1;
        mm &= mm - 1;
        if (leaf_row(x, tc * 32 + k)) m |= 1u << k;
      }
      return m;
    }
    case LM_REGLUT:
    case LM_MEMLUT: {
      if (tc * 32 >= R) return 0u;   // a short slab (or a reduced slab size): nothing staged for this thread
      const uint32_t* w = x.c.colw + tc * x.c.bw;
      if (x.c.phase == 0) {
        if (x.mode == LM_REGLUT) {
          switch (x.c.bw) {
            case 0: return (x.lutreg & 1u) ? 0xffffffffu : 0u;
            case 1: return leaf_dense_bw<1, true>(w, x.lutreg, nullptr, 0);
            case 2: return leaf_dense_bw<2, true>(w, x.lutreg, nullptr, 0);
            case 3: return leaf_dense_bw<3, true>(w, x.lutreg, nullptr, 0);
            case 4: return leaf_dense_bw<4, true>(w, x.lutreg, nullptr, 0);
            default: return leaf_dense_bw<5, true>(w, x.lutreg, nullptr, 0);
          }
        }
        switch (x.c.bw) {
          case 1: return leaf_dense_bw<1, false>(w, 0, x.lut, x.c.dict_max);
          case 2: return leaf_dense_bw<2, false>(w, 0, x.lut, x.c.dict_max);
          case 3: return leaf_dense_bw<3, false>(w, 0, x.lut, x.c.dict_max);
          case 4: return leaf_dense_bw<4, false>(w, 0, x.lut, x.c.dict_max);
          case 5: return leaf_dense_bw<5, false>(w, 0, x.lut, x.c.dict_max);
          case 6: return leaf_dense_bw<6, false>(w, 0, x.lut, x.c.dict_max);
          case 7: return leaf_dense_bw<7, false>(w, 0, x.lut, x.c.dict_max);
          case 8: return leaf_dense_bw<8, false>(w, 0, x.lut, x.c.dict_max);
          case 9: return leaf_dense_bw<9, false>(w, 0, x.lut, x.c.dict_max);
          case 10: return leaf_dense_bw<10, false>(w, 0, x.lut, x.c.dict_max);
          case 11: return leaf_dense_bw<11, false>(w, 0, x.lut, x.c.dict_max);
          case 12: return leaf_dense_bw<12, false>(w, 0, x.lut, x.c.dict_max);
          default: break;
        }
      }
      // wide indices, or a piece that starts inside a page off the 32-bit grid: value by value
      uint32_t m = 0, bit = x.c.phase + tc * 32 * x.c.bw;
      if (x.mode == LM_REGLUT) {
#pragma unroll 4
        for (int k = 0; k < 32; k++, bit += x.c.bw) m = __funnelshift_r(m, __funnelshift_r(x.lutreg, x.lutreg, bits32_at(x.c.colw, bit)), 1);
      } else {
#pragma unroll 4
        for (int k = 0; k < 32; k++, bit += x.c.bw) {
          uint32_t v = bits32_at(x.c.colw, bit) & x.c.mask;
          v = v < x.c.dict_max ? v : x.c.dict_max;
          m = __funnelshift_r(m, uint32_t(__ldg(x.lut + v)), 1);
        }
      }
      return m;
    }
    case LM_BITS: {
      if (tc * 32 >= R) return 0u;
      const uint32_t word = bits32_at(x.c.colw, x.c.phase + tc * 32);
      const uint32_t r1 = cmp_i64(1, x.lit, x.cmp) ? word : 0u, r0 = cmp_i64(0, x.lit, x.cmp) ? ~word : 0u;
      return r1 | r0;
    }
    default: {
      // LM_PLAIN8: transposed over the warp (lane L reads row base + 32 j + L: conflict free), lane j keeps word j
      const uint32_t lane = threadIdx.x & 31, wbase = (tc - lane) * 32;   // the warp's 32 consecutive words: lane j owns word (tc - lane) + j
      const uint64_t* v8 = x.c.v8;
      uint32_t mine = 0;
#pragma unroll 4
      for (uint32_t j = 0; j < 32; j++) {
        const uint32_t r = wbase + j * 32 + lane;
        const bool t = r < R && plain_cmp(v8[r], x);
        const uint32_t wj = __ballot_sync(0xffffffffu, t);
        if (lane == j) mine = wj;
      }
      return mine;
    }
  }
}

// SQL three-valued logic on bit planes: t = TRUE rows, n = NULL rows (FALSE = neither); arrow's Kleene and / or
struct Tri32 { uint32_t t, n; };
__device__ __forceinline__ Tri32 tri_leaf(const LeafCtx& x, uint32_t V, uint32_t dense) {
  if (x.lkind == LK_IS_NULL) return {~V, 0u};
  if (x.lkind == LK_IS_NOT_NULL) return {V, 0u};
  return {dense & V, ~V};
}
__device__ __forceinline__ Tri32 tri_and(Tri32 a, Tri32 b) {
  const uint32_t fa = ~(a.t | a.n), fb = ~(b.t | b.n);
  return {a.t & b.t, (a.n | b.n) & ~fa & ~fb};
}
__device__ __forceinline__ Tri32 tri_or(Tri32 a, Tri32 b) {
  const uint32_t t = a.t | b.t;
  return {t, (a.n | b.n) & ~t};
}
__device__ __forceinline__ Tri32 tri_not(Tri32 a) { return {~(a.t | a.n), a.n}; }

// ---- k_flat_filter ------------------------------------------------------------------------------
// CONJ: the predicate is a pure conjunction of leaves (or there is none) -- its own instantiation, without the
// three-valued evaluation stack of general programs (registers, local memory and instruction-cache footprint)
template <bool CONJ>
__global__ void __launch_bounds__(kFilterThreads, 6)
k_flat_filter(const __grid_constant__ DevPlan plan, const __grid_constant__ FlatLayout L, const __grid_constant__ DevScanArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];
  FlatCtl& ctl = *reinterpret_cast<FlatCtl*>(smem);
  flat_ctl_init(ctl, L.nstages, 1);
  __syncthreads();
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == kFilterConsumerWarps) {   // the last warp produces
    flat_producer(plan, L, a, ctl, smem, plan.flat_slab_rows, kFilterConsumerWarps, 512);   // a stage comes back every ~1.5 us
    return;
  }
  // A stage is ONE warp's slab (<= 2048 rows): a consumer warp draws the next stage in fill order with a ticket,
  // works through it alone and hands it back alone -- no warp ever waits for a slower one, and the ring is as deep as
  // shared memory allows (L.nstages is a power of two).  Thread: bitmap words h * 32 + lane (h = 0, 1) of the slab.
  uint32_t word[kFilterWords];
#pragma unroll
  for (int h = 0; h < kFilterWords; h++) word[h] = h * 32 + lane;
  const uint32_t stage_mask = L.nstages - 1, stage_shift = 31u - __clz(L.nstages);
  for (;;) {
    uint32_t ticket = 0;
    if (lane == 0) ticket = atomicAdd(&ctl.ticket, 1u);
    ticket = __shfl_sync(0xffffffffu, ticket, 0);
    const uint32_t stage = ticket & stage_mask, par = (ticket >> stage_shift) & 1u;
    mbar_wait_spin(&ctl.full[stage], par, 256);
    const FlatStage& st = flat_stage(smem, L, stage);
    if (st.item == 0xffffffffu) break;
    const uint32_t R = st.R;
    const uint8_t* base = smem + L.stage0 + stage * L.stage_bytes;
    uint32_t inr[kFilterWords], m[kFilterWords];
#pragma unroll
    for (int h = 0; h < kFilterWords; h++) {
      const uint32_t row0 = word[h] * 32;
      inr[h] = row0 >= R ? 0u : (R - row0 >= 32 ? 0xffffffffu : ((1u << (R - row0)) - 1u));
      m[h] = inr[h];
    }
    if (plan.npred && !(plan.dbg & 1u)) {
      if (CONJ) {
        // conjunction: a row passes when every leaf is TRUE (a NULL leaf drops it).  First leaf on every row,
        // the others on the survivors only (or dense when many survive)
        for (uint32_t l = 0; l < plan.nleaves; l++) {
          uint32_t pc = 0;
#pragma unroll
          for (int h = 0; h < kFilterWords; h++) pc += __popc(m[h]);
          const uint32_t mx = l ? __reduce_max_sync(0xffffffffu, pc) : 64u;
          if (mx == 0) break;
          LeafCtx x;
          leaf_ctx<false>(x, plan, a, st, base, L, l);
          const bool dense = mx > 12;
#if PQB_FILTER_ROLL
          // ONE copy of the leaf code for both words (the loop is not unrolled; the word in hand rotates through
          // registers): half the instruction-cache footprint of the hot path
#pragma unroll 1
          for (int h = 0; h < kFilterWords; h++) {
            const uint32_t wa = h * 32 + lane;
            uint32_t ma = m[0];
            const uint32_t V = wa * 32 < R ? col_valid32(x.c, wa * 32) : 0u;
            if (x.lkind == LK_IS_NULL) ma &= ~V;
            else {
              ma &= V;
              if (x.lkind != LK_IS_NOT_NULL) {
                if (dense) ma &= leaf_dense(x, wa, R, ma);
                else ma = leaf_survivors(x, wa * 32, ma);
              }
            }
#pragma unroll
            for (int k = 0; k + 1 < kFilterWords; k++) m[k] = m[k + 1];   // rotate: after kFilterWords trips every word is back in its place
            m[kFilterWords - 1] = ma;
          }
#else
#pragma unroll
          for (int h = 0; h < kFilterWords; h++) {
            const uint32_t V = inr[h] ? col_valid32(x.c, word[h] * 32) : 0u;
            if (x.lkind == LK_IS_NULL) { m[h] &= ~V; continue; }
            m[h] &= V;
            if (x.lkind == LK_IS_NOT_NULL) continue;
            if (dense) m[h] &= leaf_dense(x, word[h], R, m[h]);
            else m[h] = leaf_survivors(x, word[h] * 32, m[h]);
          }
#endif
        }
      } else {
        // general boolean program, SQL three-valued logic (NULLs come from validity bitmaps and NULL literals)
        Tri32 stk[kFilterWords][kPredStack];
        int sp = 0;
#pragma unroll 1
        for (uint32_t i = 0; i < plan.npred; i++) {
          const DevPredOp op = plan.pred[i];
          if (op.kind == PK_LEAF) {
            LeafCtx x;
            leaf_ctx<false>(x, plan, a, st, base, L, op.arg);
#pragma unroll
            for (int h = 0; h < kFilterWords; h++) {
              const uint32_t V = inr[h] ? col_valid32(x.c, word[h] * 32) : 0u;
              stk[h][sp] = tri_leaf(x, V, leaf_dense(x, word[h], R, inr[h] & V));
            }
            sp++;
          } else if (op.kind == PK_CONST) {
#pragma unroll
            for (int h = 0; h < kFilterWords; h++) stk[h][sp] = {op.arg == 1 ? 0xffffffffu : 0u, op.arg == 2 ? 0xffffffffu : 0u};
            sp++;
          } else if (op.kind == PK_NOT) {
#pragma unroll
            for (int h = 0; h < kFilterWords; h++) stk[h][sp - 1] = tri_not(stk[h][sp - 1]);
          } else {
            sp--;
#pragma unroll
            for (int h = 0; h < kFilterWords; h++)
              stk[h][sp - 1] = op.kind == PK_AND ? tri_and(stk[h][sp - 1], stk[h][sp]) : tri_or(stk[h][sp - 1], stk[h][sp]);
          }
        }
#pragma unroll
        for (int h = 0; h < kFilterWords; h++) m[h] = stk[h][0].t & inr[h];
      }
    }
    uint32_t pc = 0;
#pragma unroll
    for (int h = 0; h < kFilterWords; h++) {
      if (plan.write_bitmap && word[h] * 32 < R) a.bitmap[st.bitmap_word0 + (st.r0 >> 5) + word[h]] = m[h];
      pc += __popc(m[h]);
    }
    const uint32_t cnt = __reduce_add_sync(0xffffffffu, pc);
    const uint32_t item = st.item;
    __syncwarp();
    if (lane == 0) {
      mbar_arrive(&ctl.empty[stage]);
      if (cnt) atomicAdd(&a.item_counts[item], cnt);
    }
  }
}

// ---- k_flat_agg ---------------------------------------------------------------------------------
// A consumer thread owns up to kAggRowsMax rows of a slab, interleaved: row i of thread tc is
// tc + i * kAggConsumers.  The slab is processed operator by operator ("vectorised interpreter"):
// selection mask, then one pass per GROUP BY key into slot[], then one pass per aggregate.  Every
// decision that does not depend on the row (page kind, bit width, aggregate function, pointers) is
// made once per pass, outside the row loop.
constexpr int kAggRowsMax = 8;   // k_flat_agg<KR>: KR = 8, 4, 2 rows per thread and slab

// Shared-memory cells are as narrow as their updates allow (plan.hot_off): counts are u32 (a CTA sees < 2^32 rows),
// Int64 MIN / MAX whose range the footer statistics bound are u32 offsets, sums and f64 MIN / MAX keep 8 bytes.  The
// flush widens every cell into the 8-byte global table.
// `s` / `g`: the cell in the shared-memory table / in the global one, `hot` says which is meant.  Two pointers so
// that each atomic is compiled for its address space (a pointer chosen at run time makes them generic: an address-space
// test in front of every update, returning ATOM.E instead of RED for the cold cells).
__device__ __forceinline__ void cell_add_u64(unsigned long long* s, unsigned long long* g, bool hot, unsigned long long v) {
  if (hot) {
    uint32_t* w = reinterpret_cast<uint32_t*>(s);
    const uint32_t lo = uint32_t(v), hi = uint32_t(v >> 32);
    uint32_t carry = 0;
    if (lo) carry = uint32_t(atomicAdd(&w[0], lo) + lo) < lo ? 1u : 0u;
    if (hi + carry) atomicAdd(&w[1], hi + carry);
  } else atomicAdd(g, v);
}
__device__ __forceinline__ void cell_add_f64(unsigned long long* s, unsigned long long* g, bool hot, double v) {
  if (hot) atomicAdd(reinterpret_cast<double*>(s), v);   // no native shared-memory f64 add: a CAS loop
  else atomicAdd(reinterpret_cast<double*>(g), v);
}
__device__ __forceinline__ void cell_min_max(unsigned long long* s, unsigned long long* g, bool hot, bool is_min, long long k) {
  if (hot) {   // 64-bit min / max in shared memory are CAS loops: skip when the row cannot improve the cell
    const long long cur = *reinterpret_cast<volatile long long*>(s);
    if (is_min ? k >= cur : k <= cur) return;
    if (is_min) atomicMin(reinterpret_cast<long long*>(s), k);
    else atomicMax(reinterpret_cast<long long*>(s), k);
  } else if (is_min) atomicMin(reinterpret_cast<long long*>(g), k);
  else atomicMax(reinterpret_cast<long long*>(g), k);
}
// narrow Int64 MIN / MAX (plan.acc_narrow): one native 32-bit shared-memory atomic (ATOMS.MIN / MAX: no read, no CAS;
// a plain read in front of it to skip rows that cannot improve the cell measured 1 % slower).
// A value the statistics did not announce falls outside the window and goes to the global 8-byte cell `g` (the slot's
// cell, also for a per-lane cell), which the flush merges with: the answer never depends on the statistics being right.
constexpr uint64_t kNarrowSpan = 0xfffffffeull;   // offsets 0 .. kNarrowSpan (MAX stores offset + 1: 0 stays "empty")
__device__ __forceinline__ void cell_min_max32(uint32_t* s, unsigned long long* g, bool hot, bool is_min, long long k, long long base) {
  const uint64_t d = uint64_t(k) - uint64_t(base);
  if (hot && d <= kNarrowSpan) {
    if (is_min) atomicMin(s, uint32_t(d));
    else atomicMax(s, uint32_t(d) + 1u);
  } else if (is_min) atomicMin(reinterpret_cast<long long*>(g), k);
  else atomicMax(reinterpret_cast<long long*>(g), k);
}

// Cell index of a group slot inside the hot table.  The plan.lane_slots hottest groups (slots 0 .. T-1: the
// hot-first numbering puts them there) own one cell PER LANE, so that the lanes of a warp never meet on them: on
// skewed keys a fifth of a warp's rows belong to one group, and same-address shared-memory atomics (all the more the
// 64-bit CAS loops behind f64 SUM and i64 MIN / MAX) retire one lane at a time.
//   slot <  T : cell = slot * 32 + lane          slot >= T : cell = slot + 31 T
// Cold slots (cell >= hot cells) go to the global table at cell - 31 T = slot.
// HASHED instantiation: the cell of a group whose wide id (mixed radix with 64-bit strides) does not fit the dense
// table.  Open addressing, linear probing; keys only ever go from EMPTY to one value, so a stale EMPTY read is
// caught by the CAS.  A full table raises counters[1] = 100 (the host reports it, nothing is written out of bounds).
constexpr unsigned long long kHashEmpty = ~0ull;
__device__ __forceinline__ uint32_t agg_hash_slot(unsigned long long* __restrict__ keys, uint32_t mask, uint64_t wide, unsigned long long* counters) {
  uint32_t h = uint32_t(mix64(wide)) & mask;
  for (uint32_t probes = 0; probes <= mask; probes++) {
    const unsigned long long cur = *reinterpret_cast<volatile unsigned long long*>(keys + h);
    if (cur == wide) return h;
    if (cur == kHashEmpty) {
      const unsigned long long prev = atomicCAS(keys + h, kHashEmpty, (unsigned long long)wide);
      if (prev == kHashEmpty || prev == wide) return h;
    }
    h = (h + 1) & mask;
  }
  atomicExch(&counters[1], 100ull);
  return 0u;
}

template <int KR, bool HASHED>
__global__ void __launch_bounds__(kAggThreads, 1)
k_flat_agg(const __grid_constant__ DevPlan plan, const __grid_constant__ FlatLayout L, const __grid_constant__ DevScanArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];
  FlatCtl& ctl = *reinterpret_cast<FlatCtl*>(smem);
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t H = plan.hot_slots, nslots = plan.nslots, T = plan.lane_slots;
  const uint32_t Hs = H + 31u * T;   // cells per plane of the hot table
  const uint32_t cells = 1 + plan.n_acc + plan.n_nn;
  uint8_t* const hot = smem + L.acc;
  // plane p of the hot table, as 4-byte / 8-byte cells
  auto hot32 = [&](uint32_t p) { return reinterpret_cast<uint32_t*>(hot + plan.hot_off[p]); };
  auto hot64 = [&](uint32_t p) { return reinterpret_cast<unsigned long long*>(hot + plan.hot_off[p]); };
  // this CTA's copy of the global table (plan.replicas copies spread same-address traffic over L2; k_acc_reduce merges them)
  unsigned long long* gacc = a.acc + size_t(blockIdx.x % plan.replicas) * cells * nslots;
  flat_ctl_init(ctl, L.nstages, kAggConsumers / 32);
  for (uint32_t i = threadIdx.x; i < cells * Hs; i += kAggThreads) {
    const uint32_t arr = i / Hs, c = i - arr * Hs;
    if (arr >= 1 && arr < 1 + plan.n_acc) {
      const uint8_t k = plan.acc_init[arr - 1];
      if ((plan.acc_narrow >> (arr - 1)) & 1u) hot32(arr)[c] = k == 2 ? 0xffffffffu : 0u;
      else hot64(arr)[c] = k == 2 ? 0x7fffffffffffffffull : (k == 3 ? 0x8000000000000000ull : 0ull);
    } else hot32(arr)[c] = 0u;   // rows, non-null counters
  }
  __syncthreads();
  const uint32_t S = plan.flat_slab_rows;
  // Warps with (warp & 7) >= smem_share send even their hot slots to L2 (experiment switch; default: all use shared memory).
  const bool smem_warp = (warp & 7u) < plan.smem_share;
  const uint32_t Hw = smem_warp ? Hs : 0u, Tw = smem_warp ? T : 0u;
  unsigned long long* gadj = gacc - 31u * Tw;   // indexed by cell: gadj[cell] == gacc[slot] for a cold slot
  if (warp == kAggConsumers / 32) {
    flat_producer(plan, L, a, ctl, smem, S, 1, 512);
  } else {
    const uint32_t tc = threadIdx.x;
    uint32_t stage = 0, par = 0;
    for (;;) {
      mbar_wait_spin(&ctl.full[stage], par, 256);
      const FlatStage& st = flat_stage(smem, L, stage);
      if (st.item == 0xffffffffu) break;
      const uint32_t R = st.R;
      const uint8_t* base = smem + L.stage0 + stage * L.stage_bytes;
      // ---- rows of this thread, selection ----
      uint32_t sel = 0;
#pragma unroll
      for (int i = 0; i < KR; i++) sel |= (tc + i * kAggConsumers < R ? 1u : 0u) << i;
      if (plan.dbg & 2u) sel = 0;   // PQB_AGG_NOWORK: every slab handed back untouched (what producer + TMA can supply)
      if (plan.npred && sel) {
        if (plan.conj) {
          for (uint32_t l = 0; l < plan.nleaves; l++) {
            LeafCtx x;
            leaf_ctx<true>(x, plan, a, st, base, L, l);
            uint32_t m = 0;
            if (!x.c.absent && !x.c.vw && x.lkind != LK_IS_NULL && x.lkind != LK_IS_NOT_NULL) {   // no NULLs in this slab: plain comparison
#pragma unroll
              for (int i = 0; i < KR; i++)
                if ((sel >> i) & 1u) m |= (leaf_row(x, tc + i * kAggConsumers) ? 1u : 0u) << i;
            } else {
#pragma unroll
              for (int i = 0; i < KR; i++)
                if ((sel >> i) & 1u) m |= (leaf_row3(x, tc + i * kAggConsumers) == 1u ? 1u : 0u) << i;
            }
            sel = m;
          }
        } else {
          Tri32 stk[kPredStack];
          int sp = 0;
#pragma unroll 1
          for (uint32_t i = 0; i < plan.npred; i++) {
            const DevPredOp op = plan.pred[i];
            if (op.kind == PK_LEAF) {
              LeafCtx x;
              leaf_ctx<true>(x, plan, a, st, base, L, op.arg);
              Tri32 v{0u, 0u};
#pragma unroll
              for (int j = 0; j < KR; j++)
                if ((sel >> j) & 1u) {
                  const uint32_t t3 = leaf_row3(x, tc + j * kAggConsumers);
                  v.t |= (t3 == 1u ? 1u : 0u) << j;
                  v.n |= (t3 == 2u ? 1u : 0u) << j;
                }
              stk[sp++] = v;
            } else if (op.kind == PK_CONST) stk[sp++] = {op.arg == 1 ? 0xffu : 0u, op.arg == 2 ? 0xffu : 0u};
            else if (op.kind == PK_NOT) stk[sp - 1] = tri_not(stk[sp - 1]);
            else { sp--; stk[sp - 1] = op.kind == PK_AND ? tri_and(stk[sp - 1], stk[sp]) : tri_or(stk[sp - 1], stk[sp]); }
          }
          sel &= stk[0].t;
        }
      }
      // ---- group slot of every selected row: one pass per key; NULL is its own group (id == card) ----
      // HASHED: the mixed radix of the group ids is wider than the dense table (64-bit strides); the row's group
      // finds its cell through the open-addressing table a.hkeys (agg_hash_slot)
      using slot_t = typename std::conditional<HASHED, uint64_t, uint32_t>::type;
      slot_t slot[KR];
#pragma unroll
      for (int i = 0; i < KR; i++) slot[i] = 0;
      for (uint32_t k = 0; k < plan.nkeys; k++) {
        const DevKey& key = plan.keys[k];
        ColCtx c;
        col_ctx<true>(c, st, base, L, key.col, a.flat);
        const slot_t stride = HASHED ? slot_t(key.wstride) : slot_t(key.stride), nullslot = slot_t(key.card) * stride;
        const bool nullable = c.absent || c.vw != nullptr;
        if (key.kind == KK_BOOL) {
#pragma unroll
          for (int i = 0; i < KR; i++)
            if ((sel >> i) & 1u) {
              const uint32_t r = tc + i * kAggConsumers;
              if (nullable && !col_valid(c, r)) { slot[i] += nullslot; continue; }
              const uint32_t pb = c.phase + r;
              slot[i] += ((c.colw[pb >> 5] >> (pb & 31)) & 1u) * stride;
            }
        } else if (key.kind == KK_BIN) {
          // DATE_BIN: the key is computed from the value.  value - bin_base >= 0 and < 2^53 (checked on the host from the
          // footer statistics), so one double multiply and a fix-up replace a 64-bit division
          const bool plain = c.fkind == FK_PLAIN8;
          const uint64_t* __restrict__ dict = reinterpret_cast<const uint64_t*>(a.flat + st.col[key.col].dict8);
          const uint64_t* v8 = c.v8;
          const double inv = 1.0 / double(key.bin_width);
          const long long w = key.bin_width, b0 = key.bin_base;
#pragma unroll
          for (int i = 0; i < KR; i++)
            if ((sel >> i) & 1u) {
              const uint32_t r = tc + i * kAggConsumers;
              if (nullable && !col_valid(c, r)) { slot[i] += nullslot; continue; }
              const long long x = (long long)__ldg(plain ? v8 + r : dict + col_index(c, r)) - b0;
              long long q = (long long)(double(x) * inv);
              long long rem = x - q * w;
              if (rem < 0) { q--; rem += w; }
              if (rem >= w) q++;
              const uint32_t g = (q < 0 || q >= (long long)key.card) ? key.card - 1 : uint32_t(q);   // statistics were wrong: clamp, never out of the table
              slot[i] += g * stride;
            }
        } else {
          const uint32_t* __restrict__ gid = key.gid + st.col[key.col].lut_base;
          if (c.fkind == FK_IDS) {   // a page without a dictionary: its rows were interned when the table column became a key, the staged words ARE the ids
#pragma unroll
            for (int i = 0; i < KR; i++)
              if ((sel >> i) & 1u) {
                const uint32_t r = tc + i * kAggConsumers;
                if (nullable && !col_valid(c, r)) { slot[i] += nullslot; continue; }
                const uint32_t g = bits32_at(c.colw, c.phase + r * 32u);
                slot[i] += (g < key.card ? g : key.card - 1u) * stride;   // never out of the table
              }
          } else if (!nullable) {   // the loads of all rows in flight together
            uint32_t g[KR];
#pragma unroll
            for (int i = 0; i < KR; i++) g[i] = ((sel >> i) & 1u) ? __ldg(gid + col_index(c, tc + i * kAggConsumers)) : 0u;
#pragma unroll
            for (int i = 0; i < KR; i++) slot[i] += g[i] * stride;
          } else {
#pragma unroll
            for (int i = 0; i < KR; i++)
              if ((sel >> i) & 1u) {
                const uint32_t r = tc + i * kAggConsumers;
                if (!col_valid(c, r)) { slot[i] += nullslot; continue; }
                slot[i] += __ldg(gid + col_index(c, r)) * stride;
              }
          }
        }
      }
      // ---- slot -> cell (the hottest groups own a cell per lane; HASHED: the group's place in the hash table) ----
      uint32_t cell[KR];
#pragma unroll
      for (int i = 0; i < KR; i++) {
        if (HASHED) cell[i] = ((sel >> i) & 1u) ? agg_hash_slot(a.hkeys, plan.hmask, uint64_t(slot[i]), a.counters) : 0u;
        else cell[i] = uint32_t(slot[i]) < Tw ? uint32_t(slot[i]) * 32u + lane : uint32_t(slot[i]) + 31u * Tw;
      }
      // ---- COUNT(*) cell ----
      uint32_t* const srows = hot32(0);
#pragma unroll
      for (int i = 0; i < KR; i++)
        if ((sel >> i) & 1u) {
          if (cell[i] < Hw) atomicAdd(&srows[cell[i]], 1u);
          else atomicAdd(&gadj[cell[i]], 1ull);
        }
      // ---- one pass per aggregate (NULL inputs contribute nothing) ----
      for (uint32_t g = 0; g < plan.naggs; g++) {
        const DevAgg& ag = plan.aggs[g];
        if (ag.fn == AG_COUNT_STAR) continue;
        ColCtx c;
        col_ctx<true>(c, st, base, L, ag.col, a.flat);
        if (c.absent) continue;
        uint32_t vsel = sel;   // selected rows whose input is not NULL
        if (c.vw) {
#pragma unroll
          for (int i = 0; i < KR; i++)
            if (((sel >> i) & 1u) && !col_valid(c, tc + i * kAggConsumers)) vsel &= ~(1u << i);
        }
        if (ag.update_nn) {
          const uint32_t arr = 1 + plan.n_acc + ag.nn_slot;
          uint32_t* const snn = hot32(arr);
#pragma unroll
          for (int i = 0; i < KR; i++)
            if ((vsel >> i) & 1u) {
              if (cell[i] < Hw) atomicAdd(&snn[cell[i]], 1u);
              else atomicAdd(&gadj[size_t(arr) * nslots + cell[i]], 1ull);
            }
        }
        if (ag.fn == AG_COUNT) continue;
        const bool plain = c.fkind == FK_PLAIN8;
        const uint64_t* __restrict__ dict = reinterpret_cast<const uint64_t*>(a.flat + st.col[ag.col].dict8);
        const uint64_t* v8 = c.v8;
        unsigned long long* scell = hot64(1 + ag.acc_slot);
        unsigned long long* gcell = gadj + size_t(1 + ag.acc_slot) * nslots;
        const bool f64 = ag.kind == DK_F64;
        const uint32_t fn = ag.fn;
        // f64 sums have no native shared-memory atomic (a CAS loop that retires one colliding lane per trip): only the
        // per-lane cells, where the lanes of a warp never meet, keep them in shared memory; every other hot slot sends
        // them to L2 as fire-and-forget reductions (plan.f64_smem: all hot slots, plan.f64_global: none)
        const bool f64_add = fn == AG_AVG || (fn == AG_SUM && f64);
        const uint32_t Hc = !f64_add ? Hw : plan.f64_global ? 0u : plan.f64_smem ? Hw : 32u * Tw;
        // the values first (all loads in flight together: a dictionary value is an L2 round trip), then the updates,
        // one straight-line loop per aggregate function
        uint64_t bits[KR];
        if (plain) {
#pragma unroll
          for (int i = 0; i < KR; i++) bits[i] = ((vsel >> i) & 1u) ? __ldg(v8 + tc + i * kAggConsumers) : 0ull;   // in place in the flat store (global)
        } else {
#pragma unroll
          for (int i = 0; i < KR; i++) bits[i] = ((vsel >> i) & 1u) ? __ldg(dict + col_index(c, tc + i * kAggConsumers)) : 0ull;
        }
        if (fn == AG_SUM && !f64) {   // wrapping, like DataFusion's SUM(Int64)
#pragma unroll
          for (int i = 0; i < KR; i++)
            if ((vsel >> i) & 1u) cell_add_u64(scell + cell[i], gcell + cell[i], cell[i] < Hc, bits[i]);
        } else if (fn == AG_SUM || fn == AG_AVG) {
#pragma unroll
          for (int i = 0; i < KR; i++)
            if ((vsel >> i) & 1u) {
              const double v = (f64 || fn == AG_SUM) ? __longlong_as_double((long long)bits[i]) : double((long long)bits[i]);
              cell_add_f64(scell + cell[i], gcell + cell[i], cell[i] < Hc, v);
            }
        } else {
          const bool is_min = fn == AG_MIN;
          // MIN(x), MAX(x) next to each other: one pass over the values feeds both cells (the second aggregate of a
          // column never owns the non-null counter, so nothing else of its pass is left)
          const DevAgg& nx = plan.aggs[g + 1 < plan.naggs ? g + 1 : g];
          const bool narrow = (plan.acc_narrow >> ag.acc_slot) & 1u;   // decided per column: MIN and MAX of it agree
          const bool pair = g + 1 < plan.naggs && nx.col == ag.col && (nx.fn == AG_MIN || nx.fn == AG_MAX) && !nx.update_nn &&
                            narrow == (((plan.acc_narrow >> nx.acc_slot) & 1u) != 0);
          unsigned long long* gcell2 = gadj + size_t(1 + nx.acc_slot) * nslots;
          const bool is_min2 = nx.fn == AG_MIN;
          if (narrow) {
            uint32_t* s32 = hot32(1 + ag.acc_slot);
            uint32_t* s32b = hot32(1 + nx.acc_slot);
            const long long base = plan.acc_base[ag.acc_slot], base2 = plan.acc_base[nx.acc_slot];
#pragma unroll
            for (int i = 0; i < KR; i++)
              if ((vsel >> i) & 1u) {
                const uint32_t gc = cell[i] < 32u * Tw ? (cell[i] >> 5) + 31u * Tw : cell[i];   // the slot's global cell
                cell_min_max32(s32 + cell[i], gcell + gc, cell[i] < Hc, is_min, (long long)bits[i], base);
                if (pair) cell_min_max32(s32b + cell[i], gcell2 + gc, cell[i] < Hc, is_min2, (long long)bits[i], base2);
              }
          } else {
            unsigned long long* scell2 = hot64(1 + nx.acc_slot);
#pragma unroll
            for (int i = 0; i < KR; i++)
              if ((vsel >> i) & 1u) {
                const long long k = f64 ? (long long)f64_order_key(bits[i]) : (long long)bits[i];
                cell_min_max(scell + cell[i], gcell + cell[i], cell[i] < Hc, is_min, k);
                if (pair) cell_min_max(scell2 + cell[i], gcell2 + cell[i], cell[i] < Hc, is_min2, k);
              }
          }
          if (pair) g++;
        }
      }
      const uint32_t cnt = __reduce_add_sync(0xffffffffu, __popc(sel));
      const uint32_t item = st.item;
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&ctl.empty[stage]);
        if (cnt) atomicAdd(&a.item_counts[item], cnt);
      }
      if (++stage == L.nstages) { stage = 0; par ^= 1u; }
    }
  }
  // ---- flush the hot table ----
  __syncthreads();
  for (uint32_t cell = threadIdx.x; cell < Hs; cell += kAggThreads) {
    const uint32_t rows = hot32(0)[cell];
    if (rows == 0) continue;
    const uint32_t slot = cell < 32u * T ? cell >> 5 : cell - 31u * T;
    atomicAdd(&gacc[slot], (unsigned long long)rows);
    for (uint32_t arr = 0; arr < plan.n_acc; arr++) {
      const uint8_t how = plan.acc_init[arr];
      unsigned long long* g = &gacc[(1 + arr) * nslots + slot];
      if ((plan.acc_narrow >> arr) & 1u) {
        const uint32_t v = hot32(1 + arr)[cell];
        if (how == 2 ? v != 0xffffffffu : v != 0u)   // empty: every value of the slot went to the global cell (or was NULL)
          acc_merge(g, how, uint64_t(plan.acc_base[arr]) + v - (how == 2 ? 0u : 1u));
      } else acc_merge(g, how, hot64(1 + arr)[cell]);
    }
    for (uint32_t k = 0; k < plan.n_nn; k++) {
      const uint32_t v = hot32(1 + plan.n_acc + k)[cell];
      if (v) atomicAdd(&gacc[(1 + plan.n_acc + k) * nslots + slot], (unsigned long long)v);
    }
  }
}

// merge the copies 1 .. replicas-1 of the accumulator table into copy 0
__global__ void k_acc_reduce(unsigned long long* __restrict__ acc, uint32_t nslots, uint32_t cells, uint32_t replicas,
                             const __grid_constant__ DevPlan plan) {
  const uint64_t n = uint64_t(nslots) * cells;
  for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < n; i += uint64_t(gridDim.x) * blockDim.x) {
    const uint32_t arr = uint32_t(i / nslots);
    const uint8_t how = (arr >= 1 && arr < 1 + plan.n_acc) ? plan.acc_init[arr - 1] : 0;
    unsigned long long v = acc[i];
    for (uint32_t r = 1; r < replicas; r++) {
      const unsigned long long o = acc[uint64_t(r) * n + i];
      if (how == 0) v += o;
      else if (how == 1) v = (unsigned long long)__double_as_longlong(__longlong_as_double((long long)v) + __longlong_as_double((long long)o));
      else if (how == 2) v = (long long)o < (long long)v ? o : v;
      else v = (long long)o > (long long)v ? o : v;
    }
    acc[i] = v;
  }
}

}  // namespace pqb
