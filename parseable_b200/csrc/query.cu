// Query planning and execution: the C-ABI PqQueryDesc becomes a DevPlan; work items, chunk tables
// and the per-column side tables (string entry offsets, interned GROUP BY ids) come from the
// table's caches; then  k_leaf_luts -> k_flat_filter | k_flat_agg (+ k_scan for the items the flat
// store does not cover) -> k_item_prefix / k_compact_row_ids | k_agg_compact  run on one stream.
//
// Reference behaviour restated here (all /root/reference paths):
//   * predicate pushed into the scan AND re-applied (Inexact pushdown,
//     src/query/stream_schema_provider.rs:665-683): one fused evaluation gives the
//     same rows;
//   * row-group pruning from footer min/max (ParquetFormat::with_enable_pruning,
//     :146): pruning never changes results, only rows_scanned;
//   * SQL three-valued logic, NULL group keys, COUNT -> Int64, SUM(Int64) wrapping,
//     float totalOrder (SURVEY.md §8 rows a11, a12).
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <map>
#include <set>
#include <string_view>
#include <unordered_map>

#include "engine.hpp"
#include "prep_kernels.cuh"
#include "scan_kernel.cuh"
#include "flat_scan.cuh"
#include "json_egress.cuh"
#include "egress_kernels.cuh"

namespace pqb {

namespace {

template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  cudaStream_t s = nullptr;
  void alloc(size_t count, cudaStream_t stream) {
    if (p) { cudaFreeAsync(p, s); p = nullptr; }   // a second alloc (a retry with a larger capacity) replaces the first
    n = count;
    s = stream;
    if (count) PQB_CUDA(cudaMallocAsync((void**)&p, count * sizeof(T), stream));
  }
  void upload(const std::vector<T>& v, cudaStream_t stream) {
    alloc(v.size(), stream);
    if (!v.empty()) PQB_CUDA(cudaMemcpyAsync(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, stream));
  }
  void zero() { if (n) PQB_CUDA(cudaMemsetAsync(p, 0, n * sizeof(T), s)); }
  ~DevBuf() { if (p) cudaFreeAsync(p, s); }
};

constexpr uint64_t kKeepDeviceResult = 1ull << 30;   // result blocks up to this size stay on the device until the query closes

struct Timer {
  cudaEvent_t a, b;
  Timer() { cudaEventCreate(&a); cudaEventCreate(&b); }
  ~Timer() { cudaEventDestroy(a); cudaEventDestroy(b); }
};

// ---- LIKE pattern classification (arrow-string like.rs fast paths) ----
struct LikePlan { uint32_t kind; std::string needle; };
LikePlan classify_like(const std::string& pat) {
  // unescaped structure: sequence of literal chars and wildcards
  std::string lit;
  std::vector<int> tokens;  // -1 '%', -2 '_', >=0 literal byte
  for (size_t i = 0; i < pat.size(); i++) {
    char c = pat[i];
    if (c == '\\' && i + 1 < pat.size()) { tokens.push_back((unsigned char)pat[++i]); }
    else if (c == '%') tokens.push_back(-1);
    else if (c == '_') tokens.push_back(-2);
    else tokens.push_back((unsigned char)c);
  }
  bool has_us = false;
  int npct = 0;
  for (int t : tokens) { has_us |= t == -2; npct += t == -1; }
  auto literal_of = [&](size_t b, size_t e) { std::string s; for (size_t i = b; i < e; i++) s.push_back(char(tokens[i])); return s; };
  if (!has_us) {
    if (npct == 0) return {LIKE_EQ, literal_of(0, tokens.size())};
    // collapse leading / trailing runs of '%'
    size_t b = 0, e = tokens.size();
    while (b < e && tokens[b] == -1) b++;
    while (e > b && tokens[e - 1] == -1) e--;
    bool inner = false;
    for (size_t i = b; i < e; i++) inner |= tokens[i] == -1;
    if (!inner) {
      bool lead = b > 0, trail = e < tokens.size();
      std::string n = literal_of(b, e);
      if (lead && trail) return {LIKE_CONTAINS, n};
      if (trail) return {LIKE_PREFIX, n};
      if (lead) return {LIKE_SUFFIX, n};
    }
  }
  return {LIKE_GENERAL, pat};
}

uint64_t f64_bits(double d) { uint64_t b; std::memcpy(&b, &d, 8); return b; }
double bits_f64(uint64_t b) { double d; std::memcpy(&d, &b, 8); return d; }

// tri-state for pruning
enum Tri { TRI_FALSE = 0, TRI_TRUE = 1, TRI_MAYBE = 2 };

struct HostLeaf {
  DevLeaf d{};
  int qcol = -1;
  std::string str;
};

// Can `col <cmp> lit` be decided for a whole chunk from its min/max statistics?
Tri leaf_from_stats(const HostLeaf& lf, uint8_t kind, const TableChunk& ch, uint32_t rg_rows) {
  if (!ch.present) {
    // column absent: all NULL
    if (lf.d.kind == LK_IS_NULL) return TRI_TRUE;
    return TRI_FALSE;  // NULL compare is never TRUE; IS NOT NULL is FALSE
  }
  const ColumnStats& st = ch.meta->stats;
  bool no_nulls = st.null_count == 0;
  bool all_nulls = st.null_count >= 0 && uint64_t(st.null_count) == uint64_t(ch.meta->num_values);
  if (lf.d.kind == LK_IS_NULL) return no_nulls ? TRI_FALSE : (all_nulls ? TRI_TRUE : TRI_MAYBE);
  if (lf.d.kind == LK_IS_NOT_NULL) return no_nulls ? TRI_TRUE : (all_nulls ? TRI_FALSE : TRI_MAYBE);
  if (all_nulls) return TRI_FALSE;
  if (lf.d.kind != LK_CMP || !st.has_min || !st.has_max) return TRI_MAYBE;
  int lo_c, hi_c;  // sign of compare(min, lit), compare(max, lit)
  if (kind == DK_I64) {
    if (st.min.size() != 8 || st.max.size() != 8) return TRI_MAYBE;
    int64_t mn, mx;
    std::memcpy(&mn, st.min.data(), 8);
    std::memcpy(&mx, st.max.data(), 8);
    lo_c = mn < lf.d.lit_i64 ? -1 : (mn > lf.d.lit_i64 ? 1 : 0);
    hi_c = mx < lf.d.lit_i64 ? -1 : (mx > lf.d.lit_i64 ? 1 : 0);
  } else if (kind == DK_F64) {
    if (st.min.size() != 8 || st.max.size() != 8) return TRI_MAYBE;
    double mn, mx, lit = bits_f64(uint64_t(lf.d.lit_i64));
    std::memcpy(&mn, st.min.data(), 8);
    std::memcpy(&mx, st.max.data(), 8);
    // footer statistics ignore NaN and may fold -0.0/+0.0: only decide on clean finite bounds
    if (std::isnan(mn) || std::isnan(mx) || std::isnan(lit)) return TRI_MAYBE;
    if (mn == 0.0 || mx == 0.0 || lit == 0.0) return TRI_MAYBE;
    lo_c = mn < lit ? -1 : (mn > lit ? 1 : 0);
    hi_c = mx < lit ? -1 : (mx > lit ? 1 : 0);
    // a chunk may still hold NaN (greater than everything in totalOrder) outside [min,max]
    // -> never claim TRI_TRUE/FALSE on the upper side
    switch (lf.d.cmp) {
      case PQ_LT: case PQ_LE: return (lf.d.cmp == PQ_LT ? lo_c >= 0 : lo_c > 0) ? TRI_FALSE : TRI_MAYBE;
      case PQ_EQ: return (lo_c > 0) ? TRI_FALSE : TRI_MAYBE;
      default: return TRI_MAYBE;
    }
  } else if (kind == DK_STR) {
    auto cmpb = [&](const std::string& a) {
      int c = cmp_bytes((const uint8_t*)a.data(), uint32_t(a.size()), (const uint8_t*)lf.str.data(), uint32_t(lf.str.size()));
      return c;
    };
    lo_c = cmpb(st.min);
    hi_c = cmpb(st.max);
    // string max statistics may be truncated upper bounds: only use them to rule rows OUT
    switch (lf.d.cmp) {
      case PQ_EQ: return (lo_c > 0 || hi_c < 0) ? TRI_FALSE : TRI_MAYBE;
      case PQ_LT: return lo_c >= 0 ? TRI_FALSE : TRI_MAYBE;
      case PQ_LE: return lo_c > 0 ? TRI_FALSE : TRI_MAYBE;
      case PQ_GT: return hi_c <= 0 ? TRI_FALSE : TRI_MAYBE;
      case PQ_GE: return hi_c < 0 ? TRI_FALSE : TRI_MAYBE;
      default: return TRI_MAYBE;
    }
  } else {
    return TRI_MAYBE;
  }
  (void)rg_rows;
  Tri r = TRI_MAYBE;
  switch (lf.d.cmp) {
    case PQ_EQ: r = (lo_c > 0 || hi_c < 0) ? TRI_FALSE : ((lo_c == 0 && hi_c == 0) ? TRI_TRUE : TRI_MAYBE); break;
    case PQ_NE: r = (lo_c > 0 || hi_c < 0) ? TRI_TRUE : ((lo_c == 0 && hi_c == 0) ? TRI_FALSE : TRI_MAYBE); break;
    case PQ_LT: r = hi_c < 0 ? TRI_TRUE : (lo_c >= 0 ? TRI_FALSE : TRI_MAYBE); break;
    case PQ_LE: r = hi_c <= 0 ? TRI_TRUE : (lo_c > 0 ? TRI_FALSE : TRI_MAYBE); break;
    case PQ_GT: r = lo_c > 0 ? TRI_TRUE : (hi_c <= 0 ? TRI_FALSE : TRI_MAYBE); break;
    case PQ_GE: r = lo_c >= 0 ? TRI_TRUE : (hi_c < 0 ? TRI_FALSE : TRI_MAYBE); break;
  }
  if (r == TRI_TRUE && !no_nulls) r = TRI_MAYBE;  // NULL rows evaluate to NULL, not TRUE
  return r;
}

Tri tri_and(Tri a, Tri b) { return (a == TRI_FALSE || b == TRI_FALSE) ? TRI_FALSE : ((a == TRI_TRUE && b == TRI_TRUE) ? TRI_TRUE : TRI_MAYBE); }
Tri tri_or(Tri a, Tri b) { return (a == TRI_TRUE || b == TRI_TRUE) ? TRI_TRUE : ((a == TRI_FALSE && b == TRI_FALSE) ? TRI_FALSE : TRI_MAYBE); }
// NOT of "certainly not TRUE" is not "certainly TRUE" under NULLs: keep MAYBE
Tri tri_not(Tri a) { (void)a; return TRI_MAYBE; }

const char* type_name(int t) {
  switch (t) { case PQ_T_BOOL: return "Boolean"; case PQ_T_I64: return "Int64"; case PQ_T_F64: return "Float64";
    case PQ_T_UTF8: return "Utf8"; case PQ_T_TS_MS: return "Timestamp(ms)"; default: return "Null"; }
}

uint32_t align_up(uint32_t v, uint32_t a) { return (v + a - 1) & ~(a - 1); }

}  // namespace

Query::Query(const PqQueryDesc& d) {
  run(d);
}
Query::~Query() {
  for (auto& b : dev_blocks_)
    if (b && b->dev) { cudaFree(b->dev); b->dev = nullptr; }
}

void launch_slab_index(const uint8_t* arena, const DevPage* pages, uint32_t n_pages, const uint32_t* col_caps, DevSlabRec* recs,
                       DirEntry* dirs, uint8_t* page_fast, cudaStream_t stream) {
  if (!n_pages) return;
  k_slab_index<<<(n_pages + 63) / 64, 64, 0, stream>>>(arena, pages, n_pages, col_caps, recs, dirs, page_fast);
  PQB_CUDA(cudaGetLastError());
}

void launch_flatten_pages(const uint8_t* arena, const DevPage* pages, const void* jobs, uint32_t n_jobs, uint8_t* side,
                          DevSlabRec* recs, DirEntry* dirs, uint8_t* page_fast, cudaStream_t stream) {
  if (!n_jobs) return;
  k_flatten_pages<<<(n_jobs + 31) / 32, 32, 0, stream>>>(arena, pages, static_cast<const FlatJob*>(jobs), n_jobs, side, recs, dirs, page_fast);
  PQB_CUDA(cudaGetLastError());
}

void launch_flat_store(const uint8_t* arena, const DevPage* pages, const void* jobs, uint32_t n_jobs, uint8_t* flat, uint8_t* ok,
                       uint32_t* maxlen, cudaStream_t stream) {
  if (!n_jobs) return;
  k_flat_store<<<(n_jobs + 3) / 4, 128, 0, stream>>>(arena, pages, static_cast<const FlatStoreJob*>(jobs), n_jobs, flat, ok, maxlen);
  PQB_CUDA(cudaGetLastError());
}

// ---- table-level side tables (called under Table::side_mu) -----------------------------------------
static std::vector<EntChunk> column_chunks(const Table& t, int tcol) {
  std::vector<EntChunk> v(t.row_groups.size());
  for (size_t g = 0; g < t.row_groups.size(); g++) {
    const TableChunk& tc = t.row_groups[g].chunks[tcol];
    v[g] = EntChunk{tc.dict_off, tc.dict_len, tc.dict_n, t.sides[tcol].base_per_rg[g], tc.present ? 1u : 0u};
  }
  return v;
}

void launch_dba_lengths(const uint8_t* arena, const DevPage* pages, const DbaJob* jobs, uint32_t n_jobs, uint8_t* scratch, DbaInfo* info, cudaStream_t stream) {
  if (!n_jobs) return;
  k_dba_lengths<<<(n_jobs + 3) / 4, 128, 0, stream>>>(arena, pages, jobs, n_jobs, scratch, info);
  PQB_CUDA(cudaGetLastError());
}
void launch_dba_materialise(const uint8_t* arena, const DevPage* pages, const DbaJob* jobs, const DbaInfo* info, uint32_t n_jobs,
                            const uint8_t* scratch, uint8_t* mat, cudaStream_t stream) {
  if (!n_jobs) return;
  k_dba_materialise<<<(n_jobs + 3) / 4, 128, 0, stream>>>(arena, pages, jobs, info, n_jobs, scratch, mat);
  PQB_CUDA(cudaGetLastError());
}
void launch_check_flat_indices(const uint8_t* flat, const FlatPageRec* fpages, const uint32_t* dict_n, uint32_t n_pages, uint32_t* first_bad, cudaStream_t stream) {
  if (!n_pages) return;
  k_check_flat_indices<<<(n_pages + 3) / 4, 128, 0, stream>>>(flat, fpages, dict_n, n_pages, first_bad);
  PQB_CUDA(cudaGetLastError());
}
void launch_page_has_nulls(const uint8_t* arena, const DevPage* pages, uint32_t n_pages, uint8_t* out, cudaStream_t stream) {
  if (!n_pages) return;
  k_page_has_nulls<<<(n_pages + 127) / 128, 128, 0, stream>>>(arena, pages, n_pages, out);
  PQB_CUDA(cudaGetLastError());
}

void launch_delta_to_plain8(const uint8_t* arena, const DevPage* pages, const void* jobs, uint32_t n_jobs, uint8_t* flat_base, uint8_t* ok,
                            cudaStream_t stream) {
  if (!n_jobs) return;
  k_delta_to_plain8<<<(n_jobs + 3) / 4, 128, 0, stream>>>(arena, pages, static_cast<const DeltaJob*>(jobs), n_jobs, flat_base, ok);
  PQB_CUDA(cudaGetLastError());
}

void launch_entry_offsets(const Table& t, int tcol, uint64_t* d_out, uint32_t* max_len, cudaStream_t stream) {
  std::vector<EntChunk> ch = column_chunks(t, tcol);
  if (ch.empty()) return;
  DevBuf<EntChunk> d_ch; d_ch.upload(ch, stream);
  DevBuf<unsigned int> d_err; d_err.alloc(2, stream); d_err.zero();
  k_dict_entry_offsets<<<uint32_t((ch.size() + 3) / 4), 128, 0, stream>>>(t.d_arena, d_ch.p, uint32_t(ch.size()), t.columns[tcol].kind, d_out, d_err.p);
  PQB_CUDA(cudaGetLastError());
  unsigned int errs[2] = {0, 0};
  PQB_CUDA(cudaMemcpyAsync(errs, d_err.p, 8, cudaMemcpyDeviceToHost, stream));
  PQB_CUDA(cudaStreamSynchronize(stream));
  const unsigned int err = errs[0];
  if (max_len) *max_len = t.columns[tcol].kind == DK_STR ? errs[1] : 8u;
  if (err) throw Error(PQ_ERR_CORRUPT, "column '" + t.columns[tcol].name + "': a string dictionary page runs past its end");
}

// GROUP BY key interning of one table column: every dictionary entry of every row group gets the
// dense id of its VALUE (DataFusion's GroupValues, SURVEY §8 a12), ids numbered hot-first from a
// sample of the column, and the distinct values are packed for the result batches.
void build_key_side(const Table& t, int tcol, ColSide& side, cudaStream_t stream) {
  const uint8_t kkind = t.columns[tcol].kind;
  std::vector<EntChunk> ch = column_chunks(t, tcol);
  const uint32_t nrg = uint32_t(ch.size());
  const uint32_t n = side.total_entries;
  // ---- pages without a dictionary: their rows are entries too ----
  std::vector<RowPage> rowpages;
  side.key_row_pages.clear();
  side.n_dict_pad = (n + 3u) & ~3u;
  uint64_t row_entries = 0;
  for (uint32_t g = 0; g < nrg; g++) {
    const TableChunk& tc = t.row_groups[g].chunks[tcol];
    if (!tc.present) continue;
    for (uint32_t k = 0; k < tc.pages.n_pages; k++) {
      const uint32_t pi = tc.pages.first_page + k;
      const DevPage& dp = t.pages[pi];
      if (dp.enc == DE_DICT || dp.enc == DE_RLE_BOOL) continue;
      const FlatPageRec* fr = pi < t.flat_pages.size() ? &t.flat_pages[pi] : nullptr;
      if (!fr || (fr->fkind != FK_PLAIN8 && fr->fkind != FK_BYTES))
        throw Error(PQ_ERR_UNSUPPORTED, "GROUP BY column '" + t.columns[tcol].name + "': a page without a dictionary has no flat-store copy to take the keys from");
      rowpages.push_back(RowPage{fr->off, fr->voff, fr->base, fr->rows, uint32_t(row_entries), fr->fkind, 0u});
      side.key_row_pages.push_back({pi, uint32_t(row_entries)});
      row_entries += (uint64_t(fr->rows) + 3u) & ~3ull;
    }
  }
  if (uint64_t(side.n_dict_pad) + row_entries > 0xfffffff0ull) throw Error(PQ_ERR_UNSUPPORTED, "GROUP BY column '" + t.columns[tcol].name + "': more than 2^32 key entries");
  const uint32_t n_all = rowpages.empty() ? n : uint32_t(side.n_dict_pad + row_entries);
  side.key_entries = n_all;
  PQB_CUDA(cudaMallocAsync((void**)&side.d_gid, std::max<uint64_t>(n_all, 1) * 4, stream));
  PQB_CUDA(cudaMemsetAsync(side.d_gid, 0, std::max<uint64_t>(n_all, 1) * 4, stream));
  side.card = 0;
  side.kd = KeyDict{};
  side.kd.offs.assign(1, 0);
  if (!n_all || !nrg) { PQB_CUDA(cudaStreamSynchronize(stream)); return; }
  DevBuf<EntChunk> d_ch; d_ch.upload(ch, stream);
  DevBuf<RowPage> d_rp;
  if (!rowpages.empty()) {
    d_rp.upload(rowpages, stream);
    PQB_CUDA(cudaMallocAsync((void**)&side.d_row_ent, row_entries * 8, stream));
    PQB_CUDA(cudaMemsetAsync(side.d_row_ent, 0xff, row_entries * 8, stream));   // padding between pages: no entry
    k_row_entries<<<uint32_t(std::min<size_t>(rowpages.size(), 65535)), 256, 0, stream>>>(t.d_flat, d_rp.p, uint32_t(rowpages.size()),
                                                                                         uint64_t(t.d_flat) - uint64_t(t.d_arena), side.d_row_ent);
    PQB_CUDA(cudaGetLastError());
  }
  const EntView ent{side.d_ent_off, side.d_row_ent, rowpages.empty() ? n : side.n_dict_pad};
  const uint32_t maxn = std::max<uint32_t>(side.max_dict_n, 1);
  uint64_t cap = 64;
  while (cap < 4ull * maxn) cap <<= 1;
  while (cap < std::min<uint64_t>(2 * row_entries, 1ull << 22)) cap <<= 1;   // rows: start where a column of mostly distinct values needs few redos
  DevBuf<uint32_t> rep;
  uint32_t card = 0;
  for (;;) {
    DevBuf<unsigned long long> slots; slots.alloc(cap, stream); slots.zero();
    DevBuf<uint32_t> gid_of_slot; gid_of_slot.alloc(cap, stream);
    DevBuf<uint32_t> rep_try; rep_try.alloc(cap, stream);
    DevBuf<uint32_t> counter; counter.alloc(2, stream); counter.zero();
    DevKeyTable kt{slots.p, gid_of_slot.p, rep_try.p, counter.p, uint32_t(cap - 1), kkind, ent, side.d_gid};
    const uint32_t gy = std::min<uint32_t>((maxn + 255) / 256, 64);
    for (int mode = 0; mode < 2; mode++) {
      for (uint32_t c0 = 0; n && c0 < nrg; c0 += 32768) {
        dim3 grid(std::min<uint32_t>(32768, nrg - c0), gy);
        k_key_intern<<<grid, 256, 0, stream>>>(t.d_arena, d_ch.p, c0, kt, mode);
      }
      if (!rowpages.empty())
        k_row_intern<<<uint32_t(std::min<size_t>(rowpages.size(), 65535)), 256, 0, stream>>>(t.d_arena, d_rp.p, uint32_t(rowpages.size()), kt, mode);
    }
    PQB_CUDA(cudaGetLastError());
    uint32_t cnt[2];
    PQB_CUDA(cudaMemcpyAsync(cnt, counter.p, 8, cudaMemcpyDeviceToHost, stream));
    PQB_CUDA(cudaStreamSynchronize(stream));
    if (cnt[1] == 1 || cnt[0] * 2ull > cap) {  // table too full: grow and redo
      if (cap > (1ull << 30)) throw Error(PQ_ERR_UNSUPPORTED, "GROUP BY key table overflow");
      cap <<= 2;
      continue;
    }
    if (cnt[1]) throw Error(PQ_ERR_CUDA, "group key lookup failed");
    card = cnt[0];
    rep.alloc(std::max<uint32_t>(card, 1), stream);
    PQB_CUDA(cudaMemcpyAsync(rep.p, rep_try.p, size_t(card) * 4, cudaMemcpyDeviceToDevice, stream));
    PQB_CUDA(cudaStreamSynchronize(stream));
    break;
  }
  side.card = card;
  // ---- hot-first numbering: occurrences of every id over a sample of the column's flat pages ----
  if (card > 1 && t.d_flat_pages) {
    std::vector<KeySamplePage> sp;
    std::vector<uint32_t> cand;
    for (uint32_t g = 0; g < nrg; g++) {
      const TableChunk& tc = t.row_groups[g].chunks[tcol];
      if (!tc.present) continue;
      for (uint32_t k = 0; k < tc.pages.n_pages; k++)
        if (t.flat_pages[tc.pages.first_page + k].fkind == FK_INDEX) { cand.push_back(g); cand.push_back(tc.pages.first_page + k); }
    }
    const size_t npg = cand.size() / 2, want = std::min<size_t>(npg, 192);
    for (size_t i = 0; i < want; i++) {
      const size_t j = i * npg / want;
      const uint32_t g = cand[2 * j], pi = cand[2 * j + 1];
      const FlatPageRec& fr = t.flat_pages[pi];
      sp.push_back({fr.off, std::min<uint32_t>(fr.rows, 2048), fr.bw, side.base_per_rg[g], t.row_groups[g].chunks[tcol].dict_n});
    }
    if (!sp.empty()) {
      DevBuf<KeySamplePage> d_sp; d_sp.upload(sp, stream);
      DevBuf<uint32_t> d_cnt; d_cnt.alloc(card, stream); d_cnt.zero();
      k_key_sample<<<uint32_t(sp.size()), 256, 0, stream>>>(t.d_flat, d_sp.p, uint32_t(sp.size()), side.d_gid, d_cnt.p);
      PQB_CUDA(cudaGetLastError());
      std::vector<uint32_t> cnt(card), hrep(card);
      PQB_CUDA(cudaMemcpyAsync(cnt.data(), d_cnt.p, size_t(card) * 4, cudaMemcpyDeviceToHost, stream));
      PQB_CUDA(cudaMemcpyAsync(hrep.data(), rep.p, size_t(card) * 4, cudaMemcpyDeviceToHost, stream));
      PQB_CUDA(cudaStreamSynchronize(stream));
      std::vector<uint32_t> order(card);
      for (uint32_t i = 0; i < card; i++) order[i] = i;
      // hot first; ties by the representative entry (deterministic for a given table)
      std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return cnt[a] != cnt[b] ? cnt[a] > cnt[b] : hrep[a] < hrep[b]; });
      std::vector<uint32_t> remap(card), nrep(card);
      for (uint32_t i = 0; i < card; i++) { remap[order[i]] = i; nrep[i] = hrep[order[i]]; }
      DevBuf<uint32_t> d_remap; d_remap.upload(remap, stream);
      k_gid_remap<<<std::min<uint32_t>(1024, (n_all + 255) / 256), 256, 0, stream>>>(side.d_gid, side.d_gid, n_all, d_remap.p, card);
      PQB_CUDA(cudaMemcpyAsync(rep.p, nrep.data(), size_t(card) * 4, cudaMemcpyHostToDevice, stream));
      PQB_CUDA(cudaStreamSynchronize(stream));
    }
  }
  // ---- pack the distinct values: lengths -> offsets (host) -> bytes ----
  KeyDict& loc = side.kd;
  loc.offs.assign(size_t(card) + 1, 0);
  if (card) {
    DevBuf<uint32_t> lens;
    lens.alloc(card, stream);
    k_key_lens<<<(card + 255) / 256, 256, 0, stream>>>(t.d_arena, ent, rep.p, card, kkind, lens.p);
    std::vector<uint32_t> hl(card);
    PQB_CUDA(cudaMemcpyAsync(hl.data(), lens.p, card * 4ull, cudaMemcpyDeviceToHost, stream));
    PQB_CUDA(cudaStreamSynchronize(stream));
    uint64_t tot = 0;
    for (uint32_t g = 0; g < card; g++) { loc.offs[g] = uint32_t(tot); tot += hl[g]; }
    loc.offs[card] = uint32_t(tot);
    if (tot > 0x7fffffffull) throw Error(PQ_ERR_UNSUPPORTED, "group key strings exceed 2 GiB");
    DevBuf<uint32_t> doffs;
    doffs.upload(loc.offs, stream);
    DevBuf<uint8_t> dbytes;
    dbytes.alloc(std::max<uint64_t>(tot, 1), stream);
    k_key_bytes<<<card, 64, 0, stream>>>(t.d_arena, ent, rep.p, card, kkind, doffs.p, dbytes.p);
    loc.bytes.resize(tot);
    if (tot) PQB_CUDA(cudaMemcpyAsync(loc.bytes.data(), dbytes.p, tot, cudaMemcpyDeviceToHost, stream));
    // the result assembly reads the dictionary on the device
    PQB_CUDA(cudaMallocAsync((void**)&side.d_kd_offs, (size_t(card) + 1) * 4, stream));
    PQB_CUDA(cudaMallocAsync((void**)&side.d_kd_bytes, std::max<uint64_t>(tot, 1), stream));
    PQB_CUDA(cudaMemcpyAsync(side.d_kd_offs, doffs.p, (size_t(card) + 1) * 4, cudaMemcpyDeviceToDevice, stream));
    if (tot) PQB_CUDA(cudaMemcpyAsync(side.d_kd_bytes, dbytes.p, tot, cudaMemcpyDeviceToDevice, stream));
    PQB_CUDA(cudaStreamSynchronize(stream));
    for (uint32_t g = 0; g < card; g++) side.kd_max_len = std::max(side.kd_max_len, hl[g]);
  }
}

// Collective: every rank of the communicator calls it for the same key column at the same time.
void unify_key_side(const Table& t, int tcol, ColSide& cs, cudaStream_t stream) {
  const KeyDict& loc = cs.kd;
  const uint32_t card_l = cs.card;
  const int nr = comm_nranks(), me = comm_rank();
  std::vector<unsigned long long> sizes(size_t(nr) * 2);
  {
    unsigned long long mine[2] = {card_l, loc.bytes.size()};
    DevBuf<unsigned long long> dsend, drecv;
    dsend.alloc(2, stream);
    drecv.alloc(size_t(nr) * 2, stream);
    PQB_CUDA(cudaMemcpyAsync(dsend.p, mine, 16, cudaMemcpyHostToDevice, stream));
    comm_allgather_bytes(dsend.p, drecv.p, 16, stream);
    PQB_CUDA(cudaMemcpyAsync(sizes.data(), drecv.p, size_t(nr) * 16, cudaMemcpyDeviceToHost, stream));
    PQB_CUDA(cudaStreamSynchronize(stream));
  }
  unsigned long long cardmax = 0, bytesmax = 0;
  for (int r = 0; r < nr; r++) { cardmax = std::max(cardmax, sizes[2 * r]); bytesmax = std::max(bytesmax, sizes[2 * r + 1]); }
  const size_t per_rank = ((4 * (cardmax + 1) + bytesmax) + 15) & ~size_t(15);
  std::vector<uint8_t> sendbuf(per_rank, 0), recvbuf(per_rank * nr);
  std::memcpy(sendbuf.data(), loc.offs.data(), loc.offs.size() * 4);
  if (!loc.bytes.empty()) std::memcpy(sendbuf.data() + 4 * (cardmax + 1), loc.bytes.data(), loc.bytes.size());
  {
    DevBuf<uint8_t> dsend, drecv;
    dsend.upload(sendbuf, stream);
    drecv.alloc(per_rank * nr, stream);
    comm_allgather_bytes(dsend.p, drecv.p, per_rank, stream);
    PQB_CUDA(cudaMemcpyAsync(recvbuf.data(), drecv.p, per_rank * nr, cudaMemcpyDeviceToHost, stream));
    PQB_CUDA(cudaStreamSynchronize(stream));
  }
  // ids by first occurrence in rank order: identical content + identical order on every rank.  Views into the received
  // bytes (no copies), one hash probe per value
  std::unordered_map<std::string_view, uint32_t> ids;
  {
    size_t total = 0;
    for (int r = 0; r < nr; r++) total += size_t(sizes[2 * r]);
    ids.reserve(total);
  }
  std::vector<uint32_t> remap(std::max<uint32_t>(card_l, 1), 0);
  KeyDict& glob = cs.glob_kd;
  glob.offs.assign(1, 0);
  glob.bytes.clear();
  for (int r = 0; r < nr; r++) {
    const uint8_t* base = recvbuf.data() + per_rank * r;
    const uint32_t* offs = reinterpret_cast<const uint32_t*>(base);
    const uint8_t* bytes = base + 4 * (cardmax + 1);
    for (unsigned long long i = 0; i < sizes[2 * r]; i++) {
      const std::string_view v(reinterpret_cast<const char*>(bytes + offs[i]), offs[i + 1] - offs[i]);
      auto it = ids.find(v);
      if (it == ids.end()) {
        it = ids.emplace(v, uint32_t(ids.size())).first;
        glob.bytes.insert(glob.bytes.end(), v.begin(), v.end());
        glob.offs.push_back(uint32_t(glob.bytes.size()));
      }
      if (r == me) remap[i] = it->second;
    }
  }
  cs.glob_card = uint32_t(ids.size());
  auto renew = [&](auto*& p, size_t bytes) {
    if (p) PQB_CUDA(cudaFreeAsync(p, stream));
    p = nullptr;
    PQB_CUDA(cudaMallocAsync((void**)&p, std::max<size_t>(bytes, 16), stream));
  };
  const uint32_t n_ent = cs.key_entries ? cs.key_entries : cs.total_entries;   // rows of pages without a dictionary are entries too
  renew(cs.d_glob_gid, size_t(n_ent) * 4);
  renew(cs.d_glob_kd_offs, glob.offs.size() * 4);
  renew(cs.d_glob_kd_bytes, glob.bytes.size());
  PQB_CUDA(cudaMemcpyAsync(cs.d_glob_kd_offs, glob.offs.data(), glob.offs.size() * 4, cudaMemcpyHostToDevice, stream));
  if (!glob.bytes.empty()) PQB_CUDA(cudaMemcpyAsync(cs.d_glob_kd_bytes, glob.bytes.data(), glob.bytes.size(), cudaMemcpyHostToDevice, stream));
  cs.glob_max_len = 0;
  for (size_t g = 0; g + 1 < glob.offs.size(); g++) cs.glob_max_len = std::max(cs.glob_max_len, glob.offs[g + 1] - glob.offs[g]);
  if (card_l && n_ent) {
    DevBuf<uint32_t> dremap;
    dremap.upload(remap, stream);
    k_gid_remap<<<std::min<uint32_t>(1024, (n_ent + 255) / 256), 256, 0, stream>>>(cs.d_gid, cs.d_glob_gid, n_ent, dremap.p, card_l);
    PQB_CUDA(cudaGetLastError());
  }
  PQB_CUDA(cudaStreamSynchronize(stream));
  (void)t; (void)tcol;
  cs.glob_epoch = comm_epoch();
  cs.glob_ready = true;
}

void Query::run(const PqQueryDesc& d) {
  const auto t_begin = std::chrono::steady_clock::now();
  const char* vb = getenv("PQB_VERBOSE"); const bool verbose = vb && vb[0] && vb[0] != '0';
  auto mark = [&](const char* what) {   // PQB_VERBOSE: host timeline of this query
    if (verbose)
      fprintf(stderr, "[pqb] +%.3f ms %s\n", std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count(), what);
  };
  struct HostTimer {
    std::chrono::steady_clock::time_point t0;
    PqMetrics* m;
    ~HostTimer() { m->host_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(); }
  } host_timer{t_begin, &metrics};
  Context& ctx = Context::get();
  ctx.ensure();
  if (d.n_columns > (uint32_t)kMaxCols) throw Error(PQ_ERR_UNSUPPORTED, "too many referenced columns");
  if (d.n_aggs > (uint32_t)kMaxAggs) throw Error(PQ_ERR_UNSUPPORTED, "too many aggregates");
  if (d.n_group_by > (uint32_t)kMaxKeys) throw Error(PQ_ERR_UNSUPPORTED, "too many GROUP BY columns");
  if (d.n_pred > (uint32_t)kMaxPredOps) throw Error(PQ_ERR_UNSUPPORTED, "predicate program too long");
  if (d.n_group_by && !d.n_aggs) throw Error(PQ_ERR_INVALID_ARG, "GROUP BY without aggregates");

  cudaStream_t stream;
  PQB_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
  struct StreamGuard { cudaStream_t s; ~StreamGuard() { cudaStreamDestroy(s); } } sg{stream};

  // ---- input: resident table, or upload the referenced columns of a file list ----
  const Table* table = reinterpret_cast<const Table*>(d.table);
  std::vector<int> tcol(d.n_columns, -1);  // query column -> table column
  if (!table) {
    if (!d.files || !d.n_files) throw Error(PQ_ERR_INVALID_ARG, "query has neither a table nor files");
    std::vector<std::string> names;
    for (uint32_t c = 0; c < d.n_columns; c++) names.push_back(d.columns[c].name ? d.columns[c].name : "");
    owned_table_ = std::make_unique<Table>();
    owned_table_->open(d.files, d.n_files, names, d.shard_index, d.shard_count, stream);
    metrics.upload_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
    table = owned_table_.get();
    metrics.h2d_bytes += table->h2d_bytes;
  }
  for (uint32_t c = 0; c < d.n_columns; c++) {
    if (!d.columns[c].name) throw Error(PQ_ERR_INVALID_ARG, "column without a name");
    tcol[c] = table->find_column(d.columns[c].name);
    if (tcol[c] < 0) throw Error(PQ_ERR_INVALID_ARG, std::string("column '") + d.columns[c].name + "' is not part of the resident table");
  }

  // ---- column kinds vs the plan's expectation ----
  DevPlan plan{};
  plan.ncols = d.n_columns;
  for (uint32_t c = 0; c < d.n_columns; c++) {
    const TableColumn& tc = table->columns[tcol[c]];
    uint8_t kind = tc.kind;
    int want = d.columns[c].type;
    if (kind == 0xfe) {  // in no file: all NULL, take the plan's type
      kind = want == PQ_T_F64 ? DK_F64 : want == PQ_T_UTF8 ? DK_STR : want == PQ_T_BOOL ? DK_BOOL : DK_I64;
    } else {
      bool ok = (want == PQ_T_I64 && kind == DK_I64 && !tc.is_ts) || (want == PQ_T_TS_MS && kind == DK_I64 && tc.is_ts) ||
                (want == PQ_T_F64 && kind == DK_F64) || (want == PQ_T_UTF8 && kind == DK_STR) ||
                (want == PQ_T_BOOL && kind == DK_BOOL) || want == PQ_T_NULL;
      // Int64 plan type also accepts a timestamp column and vice versa (same physical values)
      if (!ok && kind == DK_I64 && (want == PQ_T_I64 || want == PQ_T_TS_MS)) ok = true;
      if (!ok) throw Error(PQ_ERR_INVALID_ARG, std::string("column '") + tc.name + "' is not " + type_name(want) + " in the Parquet files");
    }
    plan.cols[c].kind = kind;
    plan.cols[c].max_def = tc.max_def;
  }
  auto out_type_of = [&](uint32_t c) -> int {
    const TableColumn& tc = table->columns[tcol[c]];
    if (d.columns[c].type != PQ_T_NULL) return d.columns[c].type;
    switch (plan.cols[c].kind) { case DK_F64: return PQ_T_F64; case DK_STR: return PQ_T_UTF8; case DK_BOOL: return PQ_T_BOOL;
      default: return tc.is_ts ? PQ_T_TS_MS : PQ_T_I64; }
  };

  // ---- predicate compile ----
  std::vector<HostLeaf> leaves;
  std::vector<DevPredOp> prog;
  std::vector<uint8_t> lit_pool(16, 0);
  bool has_null_const = false;
  {
    int depth = 0;
    for (uint32_t i = 0; i < d.n_pred; i++) {
      const PqPredOp& op = d.pred[i];
      switch (op.kind) {
        case PQ_OP_CMP: case PQ_OP_IS_NULL: case PQ_OP_IS_NOT_NULL: case PQ_OP_LIKE: {
          if (op.col < 0 || uint32_t(op.col) >= d.n_columns) throw Error(PQ_ERR_INVALID_ARG, "predicate column out of range");
          if (leaves.size() >= (size_t)kMaxLeaves) throw Error(PQ_ERR_UNSUPPORTED, "too many leaf predicates");
          HostLeaf lf;
          lf.qcol = op.col;
          lf.d.col = uint8_t(op.col);
          uint8_t kind = plan.cols[op.col].kind;
          if (op.kind == PQ_OP_IS_NULL) lf.d.kind = LK_IS_NULL;
          else if (op.kind == PQ_OP_IS_NOT_NULL) lf.d.kind = LK_IS_NOT_NULL;
          else if (op.kind == PQ_OP_LIKE) {
            if (kind != DK_STR) throw Error(PQ_ERR_INVALID_ARG, "LIKE needs a Utf8 column");
            if (op.lit.type != PQ_T_UTF8) throw Error(PQ_ERR_INVALID_ARG, "LIKE needs a Utf8 pattern");
            LikePlan lp = classify_like(std::string(op.lit.str ? op.lit.str : "", op.lit.str_len));
            lf.d.kind = LK_LIKE;
            lf.d.cmp = uint8_t(lp.kind);
            lf.d.flags = op.flags;
            lf.str = lp.needle;
          } else {
            lf.d.kind = LK_CMP;
            if (op.cmp < PQ_EQ || op.cmp > PQ_GE) throw Error(PQ_ERR_INVALID_ARG, "bad comparison operator");
            lf.d.cmp = uint8_t(op.cmp);
            // literal coercion as DataFusion's type coercion does for column-vs-literal (SURVEY §8 a11)
            switch (kind) {
              case DK_I64:
                if (op.lit.type == PQ_T_I64 || op.lit.type == PQ_T_TS_MS) lf.d.lit_i64 = op.lit.i64;
                else if (op.lit.type == PQ_T_F64 && std::nearbyint(op.lit.f64) == op.lit.f64 && op.lit.f64 >= -9223372036854775808.0 && op.lit.f64 < 9223372036854775808.0)
                  lf.d.lit_i64 = int64_t(op.lit.f64);
                else if (op.lit.type == PQ_T_F64) {
                  // DataFusion coerces the COLUMN to Float64 and compares there.  Against a literal that is no int64 this
                  // has an exact integer restatement (a non-integer double is < 2^52 in magnitude, where the cast of
                  // any int64 at or beyond it cannot cross it):  v > 100.5  <=>  v > 100,  v < 100.5  <=>  v < 101,
                  // v = 100.5 never, v != 100.5 always (for non-NULL v).  NaN is the greatest value (totalOrder).
                  const double L = op.lit.f64;
                  const int64_t kMin = std::numeric_limits<int64_t>::min();
                  auto never = [&] { lf.d.cmp = PQ_LT; lf.d.lit_i64 = kMin; };    // v < INT64_MIN
                  auto always = [&] { lf.d.cmp = PQ_GE; lf.d.lit_i64 = kMin; };   // v >= INT64_MIN
                  const bool above = std::isnan(L) || L >= 9223372036854775808.0;   // greater than every int64
                  const bool below = L < -9223372036854775808.0;                     // less than every int64
                  if (above || below) {
                    const bool lt = op.cmp == PQ_LT || op.cmp == PQ_LE, gt = op.cmp == PQ_GT || op.cmp == PQ_GE;
                    if (op.cmp == PQ_EQ) never();
                    else if (op.cmp == PQ_NE) always();
                    else if ((above && lt) || (below && gt)) always();
                    else never();
                  } else {
                    const int64_t fl = int64_t(std::floor(L)), ce = fl + 1;   // |L| < 2^52
                    switch (op.cmp) {
                      case PQ_EQ: never(); break;
                      case PQ_NE: always(); break;
                      case PQ_GT: case PQ_GE: lf.d.cmp = PQ_GT; lf.d.lit_i64 = fl; break;
                      default: lf.d.cmp = PQ_LT; lf.d.lit_i64 = ce; break;   // PQ_LT, PQ_LE
                    }
                  }
                } else throw Error(PQ_ERR_INVALID_ARG, "Int64 column compared with a non-numeric literal");
                break;
              case DK_F64:
                if (op.lit.type == PQ_T_F64) lf.d.lit_i64 = int64_t(f64_bits(op.lit.f64));
                else if (op.lit.type == PQ_T_I64) lf.d.lit_i64 = int64_t(f64_bits(double(op.lit.i64)));  // `status = 200` on a Float64 column
                else throw Error(PQ_ERR_INVALID_ARG, "Float64 column compared with a non-numeric literal");
                break;
              case DK_BOOL:
                if (op.lit.type != PQ_T_BOOL) throw Error(PQ_ERR_INVALID_ARG, "Boolean column compared with a non-boolean literal");
                lf.d.lit_i64 = op.lit.i64 ? 1 : 0;
                break;
              case DK_STR:
                if (op.lit.type != PQ_T_UTF8) throw Error(PQ_ERR_INVALID_ARG, "Utf8 column compared with a non-string literal");
                lf.str.assign(op.lit.str ? op.lit.str : "", op.lit.str_len);
                break;
              default: throw Error(PQ_ERR_UNSUPPORTED, "comparison on this column type");
            }
          }
          if (kind == DK_STR && (lf.d.kind == LK_CMP || lf.d.kind == LK_LIKE)) {
            lf.d.str_off = uint32_t(lit_pool.size());
            lf.d.str_len = uint32_t(lf.str.size());
            lit_pool.insert(lit_pool.end(), lf.str.begin(), lf.str.end());
            lit_pool.resize(align_up(uint32_t(lit_pool.size()) + 8, 8), 0);
          }
          prog.push_back({PK_LEAF, uint8_t(leaves.size())});
          leaves.push_back(lf);
          depth++;
          break;
        }
        case PQ_OP_AND: case PQ_OP_OR:
          if (depth < 2) throw Error(PQ_ERR_INVALID_ARG, "predicate program underflow");
          prog.push_back({uint8_t(op.kind == PQ_OP_AND ? PK_AND : PK_OR), 0});
          depth--;
          break;
        case PQ_OP_NOT:
          if (depth < 1) throw Error(PQ_ERR_INVALID_ARG, "predicate program underflow");
          prog.push_back({PK_NOT, 0});
          break;
        case PQ_OP_CONST:
          prog.push_back({PK_CONST, uint8_t(op.lit.type == PQ_T_NULL ? 2 : (op.lit.i64 ? 1 : 0))});
          has_null_const |= op.lit.type == PQ_T_NULL;
          depth++;
          break;
        default: throw Error(PQ_ERR_INVALID_ARG, "unknown predicate op");
      }
      if (depth > kPredStack) throw Error(PQ_ERR_UNSUPPORTED, "predicate nesting too deep");
    }
    if (d.n_pred && depth != 1) throw Error(PQ_ERR_INVALID_ARG, "predicate program does not reduce to one value");
  }

  // ---- row-group pruning + constant folding of leaves that statistics decide everywhere ----
  const uint32_t nrg_table = uint32_t(table->row_groups.size());
  std::vector<uint8_t> rg_live(std::max<uint32_t>(nrg_table, 1), 0);
  uint32_t nrg = 0;   // surviving row groups
  std::vector<int> leaf_const(leaves.size(), -1);  // -1 unknown; else Tri over all survivors
  metrics.row_groups_total = nrg_table;
  {
    std::vector<Tri> lt(leaves.size()), st;
    for (uint32_t g = 0; g < nrg_table; g++) {
      const TableRowGroup& rg = table->row_groups[g];
      for (size_t l = 0; l < leaves.size(); l++) {
        const TableChunk& ch = rg.chunks[tcol[leaves[l].qcol]];
        lt[l] = leaf_from_stats(leaves[l], plan.cols[leaves[l].qcol].kind, ch, rg.num_rows);
      }
      Tri root = TRI_TRUE;
      if (!prog.empty()) {
        st.clear();
        for (const DevPredOp& op : prog) {
          if (op.kind == PK_LEAF) st.push_back(lt[op.arg]);
          else if (op.kind == PK_CONST) st.push_back(op.arg == 1 ? TRI_TRUE : TRI_FALSE);
          else if (op.kind == PK_NOT) st.back() = tri_not(st.back());
          else { Tri b = st.back(); st.pop_back(); st.back() = op.kind == PK_AND ? tri_and(st.back(), b) : tri_or(st.back(), b); }
        }
        root = st[0];
      }
      if (root == TRI_FALSE) { metrics.row_groups_pruned++; continue; }
      for (size_t l = 0; l < leaves.size(); l++) {
        if (leaf_const[l] == -1) leaf_const[l] = lt[l];
        else if (leaf_const[l] != lt[l]) leaf_const[l] = TRI_MAYBE;
      }
      rg_live[g] = 1;
      nrg++;
      metrics.rows_scanned += rg.num_rows;
    }
  }
  // a leaf that is TRUE in every surviving row group is replaced by a constant: the injected
  // p_timestamp range filter (src/query/mod.rs:774-833) usually disappears here and its column
  // is then never read.  (A NOT above it is fine: TRUE means "TRUE for every row, no NULLs".)
  std::vector<bool> leaf_live(leaves.size(), true);
  for (DevPredOp& op : prog)
    if (op.kind == PK_LEAF && leaf_const[op.arg] == TRI_TRUE) { leaf_live[op.arg] = false; op = {PK_CONST, 1}; }

  // ---- which columns does the kernel really read? ----
  std::vector<bool> col_used(d.n_columns, false);
  for (size_t l = 0; l < leaves.size(); l++) if (leaf_live[l]) col_used[leaves[l].qcol] = true;
  for (uint32_t k = 0; k < d.n_group_by; k++) {
    if (d.group_by[k] < 0 || uint32_t(d.group_by[k]) >= d.n_columns) throw Error(PQ_ERR_INVALID_ARG, "group-by column out of range");
    col_used[d.group_by[k]] = true;
  }
  for (uint32_t a = 0; a < d.n_aggs; a++) {
    if (d.aggs[a].fn == PQ_AGG_COUNT_STAR) continue;
    if (d.aggs[a].col < 0 || uint32_t(d.aggs[a].col) >= d.n_columns) throw Error(PQ_ERR_INVALID_ARG, "aggregate column out of range");
    col_used[d.aggs[a].col] = true;
  }
  std::vector<bool> col_staged = col_used;   // predicate / key / aggregate inputs: staged per slab by the flat kernels
  const bool want_rows = d.n_aggs == 0 && !(d.flags & PQ_QUERY_COUNT_ONLY);
  for (uint32_t i = 0; want_rows && i < d.n_projection; i++) {
    if (d.projection[i] < 0 || uint32_t(d.projection[i]) >= d.n_columns) throw Error(PQ_ERR_INVALID_ARG, "projection column out of range");
    col_used[d.projection[i]] = true;        // only gathered for the selected rows
  }
  // compact to kernel column slots
  std::vector<int> slot_of(d.n_columns, -1);
  std::vector<uint32_t> qcol_of_slot;
  for (uint32_t c = 0; c < d.n_columns; c++)
    if (col_used[c]) { slot_of[c] = int(qcol_of_slot.size()); qcol_of_slot.push_back(c); }
  const uint32_t ncols = uint32_t(qcol_of_slot.size());
  {
    DevPlan p2 = plan;
    for (uint32_t s = 0; s < ncols; s++) p2.cols[s] = plan.cols[qcol_of_slot[s]];
    plan = p2;
    plan.ncols = ncols;
  }
  std::vector<int> shape_cols(ncols);
  for (uint32_t s = 0; s < ncols; s++) {
    shape_cols[s] = tcol[qcol_of_slot[s]];
    plan.cols[s].staged = col_staged[qcol_of_slot[s]] ? 1 : 0;
    // the VALUES of a DELTA_BINARY_PACKED column are needed (a range that cuts row groups, a projection of
    // p_timestamp): its pages get row-addressable 8-byte copies, once per table
    if (table->sides[shape_cols[s]].has_delta) table->ensure_plain8(shape_cols[s], stream);
  }
  std::shared_ptr<Shape> shape = table->shape_for(shape_cols, stream);
  const std::vector<DevItem>& items = shape->items;

  // is the predicate a pure conjunction of leaves (folded TRUE constants are neutral)?
  bool conj = true;
  for (const DevPredOp& op : prog)
    if (!(op.kind == PK_LEAF || op.kind == PK_AND || (op.kind == PK_CONST && op.arg == 1))) conj = false;
  // renumber live leaves; a conjunction evaluates its cheapest leaves first (narrow dictionary indices:
  // the whole LUT in a register), the later ones only see the survivors
  std::vector<int> leaf_slot(leaves.size(), -1);
  uint32_t nleaves = 0;
  {
    std::vector<size_t> order;
    for (size_t l = 0; l < leaves.size(); l++) if (leaf_live[l]) order.push_back(l);
    if (conj)
      std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) {
        auto cost = [&](size_t l) {
          const uint32_t s = uint32_t(slot_of[leaves[l].qcol]);
          if (leaves[l].d.kind == LK_IS_NULL || leaves[l].d.kind == LK_IS_NOT_NULL) return 0u;
          if (plan.cols[s].kind == DK_STR && shape->has_plain[s]) return 200u;   // PLAIN byte arrays: compared string by string, last
          return shape->flat_plain8[s] ? 64u : std::max<uint32_t>(shape->flat_max_bw[s], shape->max_bw[s]);
        };
        return cost(a) < cost(b);
      });
    for (size_t l : order) {
      leaf_slot[l] = int(nleaves);
      plan.leaves[nleaves] = leaves[l].d;
      plan.leaves[nleaves].col = uint8_t(slot_of[leaves[l].qcol]);
      nleaves++;
    }
  }
  plan.nleaves = nleaves;
  plan.conj = conj ? 1 : 0;
  // per column: the leaves a dictionary LUT answers (k_scan fuses up to two into the unpack)
  for (uint32_t c = 0; c < (uint32_t)kMaxCols; c++) { plan.col_nlut[c] = 0; plan.col_l0[c] = -1; plan.col_l1[c] = -1; }
  for (uint32_t l = 0; l < nleaves; l++) {
    const DevLeaf& lf = plan.leaves[l];
    if (lf.kind != LK_CMP && lf.kind != LK_LIKE) continue;
    if (plan.col_nlut[lf.col] == 0) plan.col_l0[lf.col] = int8_t(l);
    else if (plan.col_nlut[lf.col] == 1) plan.col_l1[lf.col] = int8_t(l);
    plan.col_nlut[lf.col]++;
  }
  {
    const char* rm = getenv("PQB_ROW_MAJOR");  // experiment switch: register-only row-major pass for no-NULL slabs
    plan.row_major = rm && rm[0] == '1';
  }
  {
    // k_scan: conjunction of 1-4 CMP/LIKE leaves: specialised octet pass over slab-indexed pages
    bool c4 = conj && nleaves >= 1 && nleaves <= 4;
    for (uint32_t l = 0; l < nleaves; l++) c4 &= plan.leaves[l].kind == LK_CMP || plan.leaves[l].kind == LK_LIKE;
    const char* fa = getenv("PQB_FAST_AND");
    plan.fast_and = c4 && !(fa && fa[0] == '0');
  }
  plan.npred = uint32_t(prog.size());
  for (size_t i = 0; i < prog.size(); i++) {
    plan.pred[i] = prog[i];
    if (prog[i].kind == PK_LEAF) plan.pred[i].arg = uint8_t(leaf_slot[prog[i].arg]);
  }

  // ---- aggregates ----
  const bool has_aggs = d.n_aggs > 0;
  bool only_count_star = has_aggs && d.n_group_by == 0;
  for (uint32_t a = 0; a < d.n_aggs; a++) only_count_star &= d.aggs[a].fn == PQ_AGG_COUNT_STAR;
  const bool agg_kernel = has_aggs && !only_count_star;
  plan.mode = agg_kernel ? SM_AGG : SM_FILTER;
  std::vector<int> agg_out_type(d.n_aggs, PQ_T_I64);
  if (has_aggs) {
    uint32_t n_acc = 0;
    plan.naggs = d.n_aggs;
    for (uint32_t a = 0; a < d.n_aggs; a++) {
      DevAgg& ag = plan.aggs[a];
      ag = DevAgg{};
      ag.fn = uint8_t(d.aggs[a].fn);
      if (ag.fn == AG_COUNT_STAR) { agg_out_type[a] = PQ_T_I64; continue; }
      if (ag.fn > AG_AVG) throw Error(PQ_ERR_INVALID_ARG, "unknown aggregate function");
      uint32_t qc = uint32_t(d.aggs[a].col);
      ag.col = uint8_t(slot_of[qc]);
      ag.kind = plan.cols[ag.col].kind;
      if (ag.fn != AG_COUNT && ag.kind != DK_I64 && ag.kind != DK_F64)
        throw Error(PQ_ERR_UNSUPPORTED, std::string("SUM/MIN/MAX/AVG over ") + type_name(out_type_of(qc)) + " is not on the GPU path");
      if (ag.fn == AG_COUNT) { agg_out_type[a] = PQ_T_I64; continue; }
      ag.acc_slot = uint8_t(n_acc);
      uint8_t how = 0;
      if (ag.fn == AG_SUM) how = ag.kind == DK_F64 ? 1 : 0;
      else if (ag.fn == AG_AVG) how = 1;
      else how = ag.fn == AG_MIN ? 2 : 3;
      plan.acc_init[n_acc++] = how;
      agg_out_type[a] = ag.fn == AG_AVG ? PQ_T_F64 : out_type_of(qc);
    }
    plan.n_acc = n_acc;
  }

  mark("plan compiled");
  // ---- what this query reads: bytes, NULL presence, encodings the kernels cannot take ----
  std::vector<uint8_t> col_needs_ent(ncols, 0);  // entry offsets (string leaf)
  for (uint32_t l = 0; l < nleaves; l++) {
    const DevLeaf& lf = plan.leaves[l];
    if ((lf.kind == LK_CMP || lf.kind == LK_LIKE) && plan.cols[lf.col].kind == DK_STR) col_needs_ent[lf.col] = 1;
  }
  uint64_t algo_bytes = 0, scanned_bytes = 0;
  std::vector<uint8_t> col_has_nulls(std::max<uint32_t>(ncols, 1), 0);   // statistics cannot rule NULLs out
  for (uint32_t g = 0; g < nrg_table; g++) {
    if (!rg_live[g]) continue;
    const TableRowGroup& rg = table->row_groups[g];
    for (uint32_t s = 0; s < ncols; s++) {
      const TableChunk& tc = rg.chunks[shape_cols[s]];
      if (!tc.present || tc.meta->stats.null_count != 0) col_has_nulls[s] = 1;   // absent column: every row NULL
      if (!tc.present) continue;
      scanned_bytes += tc.bytes;
      algo_bytes += uint64_t(tc.meta->total_uncompressed_size);
    }
  }
  for (uint32_t s = 0; s < ncols; s++) {
    const std::string& cname = table->columns[shape_cols[s]].name;
    plan.cols[s].has_delta = shape->has_delta[s];
    plan.cols[s].has_dict = shape->has_dict[s];
    plan.cols[s].has_plain = shape->has_plain[s];
    plan.cols[s].max_bw = shape->max_bw[s];
    if (shape->has_delta[s] && plan.cols[s].kind != DK_I64)
      throw Error(PQ_ERR_UNSUPPORTED, "column '" + cname + "': DELTA_BINARY_PACKED is decoded for INT64 columns only");
    if (shape->has_plain[s] && plan.cols[s].kind == DK_STR && shape->n_general)
      throw Error(PQ_ERR_UNSUPPORTED, "column '" + cname + "': PLAIN (dictionary-fallback) string pages without a flat-store copy are not decoded on the GPU");
  }
  plan.n_items = uint32_t(items.size());
  metrics.bytes_scanned = scanned_bytes;
  const bool allreduce = (d.flags & PQ_QUERY_ALLREDUCE) != 0;
  if (allreduce && !comm_active()) throw Error(PQ_ERR_INVALID_ARG, "PQ_QUERY_ALLREDUCE without pq_comm_init_rank");
  const bool multi = agg_kernel && allreduce && comm_nranks() > 1;
  // an aggregated column whose footers promise null_count == 0 in every row group read: its non-null
  // counter equals the group's row count, so the scan skips that atomic (and the table is 4 cells per group
  // narrower on C4).  Under PQ_QUERY_ALLREDUCE the cells are summed across ranks and every rank must make the same
  // choice: the per-rank footer verdicts are summed over the ranks first (a rank whose row groups were all pruned
  // contributes zeros).  The same tiny all-reduce carries whether every rank still holds the agreed numbering of the
  // GROUP BY key values (kept with the table column, tagged with the communicator's epoch; a rank may have reopened its
  // table): ONE collective and one round trip per query for both agreements.
  bool keys_agreed = true;
  if (multi) {
    std::vector<unsigned long long> f(1 + ncols, 0ull);
    for (uint32_t k = 0; k < d.n_group_by; k++) {
      if (d.group_exprs && d.group_exprs[k].kind == PQ_KEY_DATE_BIN) continue;
      const uint32_t s = uint32_t(slot_of[d.group_by[k]]);
      if (plan.cols[s].kind == DK_BOOL) continue;
      const ColSide& cs = table->sides[shape_cols[s]];
      if (!cs.glob_ready || cs.glob_epoch != comm_epoch()) f[0] = 1;   // this rank lacks an agreement
    }
    for (uint32_t s = 0; s < ncols; s++) f[1 + s] = col_has_nulls[s] ? 1ull : 0ull;
    DevBuf<unsigned long long> df;
    df.upload(f, stream);
    comm_allreduce_u64(df.p, f.size(), 0 /*sum*/, stream);
    PQB_CUDA(cudaMemcpyAsync(f.data(), df.p, f.size() * 8, cudaMemcpyDeviceToHost, stream));
    PQB_CUDA(cudaStreamSynchronize(stream));
    keys_agreed = f[0] == 0;
    for (uint32_t s = 0; s < ncols; s++) col_has_nulls[s] = f[1 + s] != 0;
  }
  std::vector<uint8_t> nn_is_rows(kMaxAggs, 0);
  {
    std::map<int, int> nn_of_col;   // one non-null counter array per aggregated column that may hold NULLs
    for (uint32_t a = 0; a < d.n_aggs; a++) {
      DevAgg& ag = plan.aggs[a];
      if (ag.fn == AG_COUNT_STAR) continue;
      ag.update_nn = 0;
      if (!col_has_nulls[ag.col]) { nn_is_rows[a] = 1; continue; }
      auto it = nn_of_col.find(int(ag.col));
      if (it == nn_of_col.end()) { it = nn_of_col.emplace(int(ag.col), int(nn_of_col.size())).first; ag.update_nn = 1; }
      ag.nn_slot = uint8_t(it->second);
    }
    plan.n_nn = uint32_t(nn_of_col.size());
  }
  // columns whose dictionary indices the row phase of k_scan needs (GROUP BY keys, aggregate inputs)
  for (uint32_t k = 0; k < d.n_group_by; k++) plan.cols[slot_of[d.group_by[k]]].need_idx = 1;
  for (uint32_t a = 0; a < d.n_aggs; a++)
    if (d.aggs[a].fn != PQ_AGG_COUNT_STAR) plan.cols[slot_of[d.aggs[a].col]].need_idx = 1;

  // ---- side tables: string entry offsets, per-leaf LUT regions ----
  DevPrepArgs pa{};
  uint64_t lut_total = 0;
  for (uint32_t s = 0; s < ncols; s++)
    if (col_needs_ent[s]) { table->ensure_ent_off(shape_cols[s], stream); pa.ent[s] = table->sides[shape_cols[s]].d_ent_off; }
  bool any_lut = false;
  uint32_t max_dict_n = 1;
  for (uint32_t l = 0; l < nleaves; l++) {
    DevLeaf& lf = plan.leaves[l];
    lf.lut_off = 0;
    if (lf.kind != LK_CMP && lf.kind != LK_LIKE) continue;
    const ColSide& cs = table->sides[shape_cols[lf.col]];
    if (lut_total + cs.total_entries > 0xfffffff0ull) throw Error(PQ_ERR_UNSUPPORTED, "leaf LUTs too large");
    lf.lut_off = uint32_t(lut_total);
    lut_total += cs.total_entries;
    any_lut |= cs.total_entries != 0;
    max_dict_n = std::max(max_dict_n, cs.max_dict_n);
  }

  // ---- GROUP BY keys: interned per table column (cached with the table) ----
  struct QKey { const KeyDict* kd = nullptr; uint32_t card = 0; bool is_bin = false; };
  std::vector<QKey> qk(d.n_group_by);
  std::vector<uint8_t> row_keys(d.n_group_by, 0);   // the key column has pages without a dictionary: per-row ids (FK_IDS pages)
  plan.nkeys = d.n_group_by;
  uint64_t launches = 0;
  for (uint32_t k = 0; agg_kernel && k < d.n_group_by; k++) {
    DevKey& key = plan.keys[k];
    key.col = uint8_t(slot_of[d.group_by[k]]);
    const uint8_t kind = plan.cols[key.col].kind;
    if (d.group_exprs && d.group_exprs[k].kind == PQ_KEY_DATE_BIN) {
      // ---- DATE_BIN(width, column, origin) (the counts / histogram API, src/query/mod.rs:623-680): the key is
      // computed from the value; the bins any scanned row can fall into come from the footer statistics ----
      const PqKeyExpr& gx = d.group_exprs[k];
      const std::string& cname = table->columns[tcol[d.group_by[k]]].name;
      if (kind != DK_I64) throw Error(PQ_ERR_INVALID_ARG, "DATE_BIN needs a Timestamp / Int64 column, '" + cname + "' is neither");
      if (gx.width_ms <= 0) throw Error(PQ_ERR_INVALID_ARG, "DATE_BIN needs a positive stride");
      int64_t vmin = INT64_MAX, vmax = INT64_MIN;
      for (uint32_t g = 0; g < nrg_table; g++) {
        if (!rg_live[g]) continue;
        const TableChunk& tc = table->row_groups[g].chunks[shape_cols[key.col]];
        if (!tc.present) continue;
        const ColumnStats& st = tc.meta->stats;
        if (st.null_count >= 0 && uint64_t(st.null_count) == uint64_t(tc.meta->num_values)) continue;   // all NULL: no bins
        if (!st.has_min || !st.has_max || st.min.size() != 8 || st.max.size() != 8)
          throw Error(PQ_ERR_UNSUPPORTED, "DATE_BIN over '" + cname + "' needs min / max statistics in the file footers");
        int64_t mn, mx;
        std::memcpy(&mn, st.min.data(), 8);
        std::memcpy(&mx, st.max.data(), 8);
        vmin = std::min(vmin, mn);
        vmax = std::max(vmax, mx);
      }
      auto floordiv = [](int64_t a, int64_t b) { int64_t q = a / b; return (a % b != 0 && ((a < 0) != (b < 0))) ? q - 1 : q; };
      int64_t bmin = 0, bmax = 0;
      if (vmin <= vmax) {
        if (vmin < gx.origin_ms - (int64_t(1) << 52) || vmax > gx.origin_ms + (int64_t(1) << 52))
          throw Error(PQ_ERR_UNSUPPORTED, "DATE_BIN: values more than 2^52 ms away from the origin");
        bmin = floordiv(vmin - gx.origin_ms, gx.width_ms);
        bmax = floordiv(vmax - gx.origin_ms, gx.width_ms);
      }
      if (multi) {   // every rank needs the same bin 0 and the same number of bins
        long long mm[2] = {(long long)bmin, -(long long)bmax};
        if (vmin > vmax) { mm[0] = INT64_MAX; mm[1] = INT64_MAX; }
        DevBuf<unsigned long long> dmm;
        dmm.alloc(2, stream);
        PQB_CUDA(cudaMemcpyAsync(dmm.p, mm, 16, cudaMemcpyHostToDevice, stream));
        comm_allreduce_u64(dmm.p, 2, 1 /*signed min*/, stream);
        PQB_CUDA(cudaMemcpyAsync(mm, dmm.p, 16, cudaMemcpyDeviceToHost, stream));
        PQB_CUDA(cudaStreamSynchronize(stream));
        if (mm[0] == INT64_MAX) { bmin = bmax = 0; } else { bmin = mm[0]; bmax = -mm[1]; }
      }
      if (bmax - bmin + 1 > (int64_t(1) << 24)) throw Error(PQ_ERR_UNSUPPORTED, "DATE_BIN: more than 2^24 bins in the scanned range");
      key.kind = KK_BIN;
      key.bin_width = gx.width_ms;
      key.bin_base = gx.origin_ms + bmin * gx.width_ms;
      qk[k].card = uint32_t(bmax - bmin + 1);
      qk[k].is_bin = true;
      continue;
    }
    key.kind = kind == DK_BOOL ? KK_BOOL : KK_DICT_LUT;
    if (key.kind == KK_BOOL) { qk[k].card = 2; continue; }
    if (plan.cols[key.col].has_plain || plan.cols[key.col].has_delta) {
      // Pages without a dictionary (PLAIN fallback of an overflowed dictionary, PLAIN / DELTA numerics): ensure_key interns
      // their ROWS next to the dictionary entries; the aggregate kernel then stages the pages' ids instead of their values,
      // so nothing else of this query may read the column's values
      for (uint32_t l = 0; l < nleaves; l++)
        if (plan.leaves[l].col == key.col && (plan.leaves[l].kind == LK_CMP || plan.leaves[l].kind == LK_LIKE))
          throw Error(PQ_ERR_UNSUPPORTED, "GROUP BY column '" + table->columns[tcol[d.group_by[k]]].name + "' has pages without a dictionary and is also filtered on: not on the GPU path");
      for (uint32_t a = 0; a < d.n_aggs; a++)
        if (plan.aggs[a].fn >= AG_SUM && plan.aggs[a].col == key.col)
          throw Error(PQ_ERR_UNSUPPORTED, "GROUP BY column '" + table->columns[tcol[d.group_by[k]]].name + "' has pages without a dictionary and is also aggregated: not on the GPU path");
      row_keys[k] = 1;
    }
    const int tc_i = shape_cols[key.col];
    table->ensure_key(tc_i, stream);
    const ColSide& cs = table->sides[tc_i];
    key.gid = cs.d_gid;
    qk[k].kd = &cs.kd;
    qk[k].card = cs.card;
  }
  if (multi && d.n_group_by) {
    // ---- multi-GPU: every rank must use ONE numbering of the key values.  The agreement (all-gather of the
    // packed distinct values, numbered by first occurrence in rank order: identical on every rank, and hot-first
    // because rank 0's ids are) is kept with the table column; `keys_agreed` (above) says whether EVERY rank holds it ----
    const uint32_t have = keys_agreed ? 1u : 0u;
    for (uint32_t k = 0; k < d.n_group_by; k++) {
      DevKey& key = plan.keys[k];
      if (key.kind != KK_DICT_LUT) continue;
      const int tc_i = shape_cols[key.col];
      if (!have) table->unify_key(tc_i, stream);
      const ColSide& cs = table->sides[tc_i];
      key.gid = cs.d_glob_gid;
      qk[k].kd = &cs.glob_kd;
      qk[k].card = cs.glob_card;
    }
  }
  // ---- id pages of key columns with pages that have no dictionary: this query's copy of the flat page table, with
  // those pages pointing into the column's id array (local or agreed numbering) ----
  DevBuf<FlatPageRec> d_kpages;
  std::vector<uint32_t> key_bw32(ncols, 0);
  {
    bool any = false;
    for (uint32_t k = 0; k < d.n_group_by; k++) any = any || row_keys[k];
    if (any) {
      std::vector<FlatPageRec> fp;
      {
        std::lock_guard<std::mutex> lk(table->side_mu);
        fp = table->flat_pages;
        for (uint32_t k = 0; k < d.n_group_by; k++) {
          if (!row_keys[k]) continue;
          const DevKey& key = plan.keys[k];
          const ColSide& cs = table->sides[shape_cols[key.col]];
          key_bw32[key.col] = 32;
          for (const ColSide::KeyRowPage& rp : cs.key_row_pages) {
            FlatPageRec& r = fp[rp.page];
            r.fkind = FK_IDS;
            r.bw = 32;
            // relative to d_flat like every flat page (the subtraction may wrap, base + offset does not); 16-byte aligned: ebase is a multiple of 4
            r.off = uint64_t(key.gid) + 4ull * (uint64_t(cs.n_dict_pad) + rp.ebase) - uint64_t(table->d_flat);
          }
        }
      }
      d_kpages.upload(fp, stream);
      metrics.h2d_bytes += fp.size() * sizeof(FlatPageRec);
    }
  }
  // mixed-radix group slot: the smallest key varies fastest, so that with hot-first ids of the largest key
  // "slot < hot_slots" is "one of the hottest values of the largest key" (flat aggregate kernel)
  uint64_t nslots64 = 1;
  {
    std::vector<uint32_t> korder(d.n_group_by);
    for (uint32_t k = 0; k < d.n_group_by; k++) korder[k] = k;
    std::stable_sort(korder.begin(), korder.end(), [&](uint32_t a, uint32_t b) { return qk[a].card < qk[b].card; });
    for (uint32_t k : korder) {
      plan.keys[k].card = qk[k].card;
      plan.keys[k].stride = uint32_t(nslots64);
      plan.keys[k].wstride = nslots64;
      if (nslots64 > (1ull << 62) / (uint64_t(qk[k].card) + 1)) throw Error(PQ_ERR_UNSUPPORTED, "GROUP BY key space wider than 2^62 combinations");
      nslots64 *= uint64_t(qk[k].card) + 1;
    }
  }
  // A key space wider than the dense table (2^26 slots): the groups that actually occur are found through a hash
  // table on the wide id (DataFusion's GroupValues hashes the key tuple, SURVEY §8 a12); its capacity is twice the
  // groups that can occur (<= rows scanned, <= combinations), so it never runs full below the 2^27-slot ceiling.
  plan.hashed = 0;
  plan.hmask = 0;
  if (nslots64 > (1ull << 26)) {
    if (allreduce || multi)
      throw Error(PQ_ERR_UNSUPPORTED, "GROUP BY key space too large for the dense accumulator table the ranks all-reduce (hashed tables are per rank)");
    uint64_t rows_bound = 0;
    for (uint32_t g = 0; g < nrg_table; g++) if (rg_live[g]) rows_bound += table->row_groups[g].num_rows;
    uint64_t cap = 1024;
    while (cap < 2 * std::min<uint64_t>(nslots64, std::max<uint64_t>(rows_bound, 1)) && cap < (1ull << 27)) cap <<= 1;
    if (cap * (1 + plan.n_acc + plan.n_nn) * 8 > (24ull << 30)) throw Error(PQ_ERR_UNSUPPORTED, "GROUP BY: the hashed accumulator table would exceed 24 GiB");
    plan.hashed = 1;
    plan.hmask = uint32_t(cap - 1);
    nslots64 = cap;
  }
  plan.nslots = uint32_t(nslots64);
  const uint32_t cells = 1 + plan.n_acc + plan.n_nn;
  // An Int64 MIN / MAX keeps 4-byte offsets from a base in the flat aggregate kernel's hot table when the footer
  // statistics of every row group read bound the column to fewer than 2^32 - 1 values (one native shared-memory atomic per
  // update instead of a read and a CAS loop).  Statistics that understate the range cost speed, never the answer: a value
  // outside the window updates the global 8-byte cell (cell_min_max32).  PQB_AGG_WIDE_CELLS=1: 8-byte cells (A/B switch).
  plan.acc_narrow = 0;
  if (agg_kernel && !plan.hashed && !(getenv("PQB_AGG_WIDE_CELLS") && atoi(getenv("PQB_AGG_WIDE_CELLS")))) {
    for (uint32_t a = 0; a < d.n_aggs; a++) {
      const DevAgg& ag = plan.aggs[a];
      if ((ag.fn != AG_MIN && ag.fn != AG_MAX) || ag.kind != DK_I64) continue;
      int64_t vmin = INT64_MAX, vmax = INT64_MIN;
      bool bounded = true;
      for (uint32_t g = 0; g < nrg_table && bounded; g++) {
        if (!rg_live[g]) continue;
        const TableChunk& tc = table->row_groups[g].chunks[shape_cols[ag.col]];
        if (!tc.present) continue;
        const ColumnStats& st = tc.meta->stats;
        if (st.null_count >= 0 && uint64_t(st.null_count) == uint64_t(tc.meta->num_values)) continue;   // all NULL: no values
        if (!st.has_min || !st.has_max || st.min.size() != 8 || st.max.size() != 8) { bounded = false; break; }
        int64_t mn, mx;
        std::memcpy(&mn, st.min.data(), 8);
        std::memcpy(&mx, st.max.data(), 8);
        vmin = std::min(vmin, mn);
        vmax = std::max(vmax, mx);
      }
      if (!bounded || vmin > vmax || uint64_t(vmax) - uint64_t(vmin) > kNarrowSpan) continue;
      // the window [base, base + kNarrowSpan] must not wrap past INT64_MAX
      plan.acc_base[ag.acc_slot] = std::min<int64_t>(vmin, INT64_MAX - int64_t(kNarrowSpan));
      plan.acc_narrow |= 1u << ag.acc_slot;
    }
  }
  plan.hot_cell_bytes = 4 * (1 + plan.n_nn);
  for (uint32_t a = 0; a < plan.n_acc; a++) plan.hot_cell_bytes += ((plan.acc_narrow >> a) & 1u) ? 4 : 8;

  // ---- which kernels run ----
  (void)has_null_const;   // the flat kernels evaluate SQL three-valued logic, NULL literals included
  const bool flat_ok = !(getenv("PQB_FLAT_SCAN") && getenv("PQB_FLAT_SCAN")[0] == '0');
  plan.no_flat = flat_ok ? 0 : 1;
  const uint32_t n_flat = flat_ok ? shape->n_flat : 0;
  const uint32_t n_general = flat_ok ? shape->n_general : uint32_t(items.size());
  const uint32_t n_fast_items = shape->n_slab_fast;

  for (uint32_t k = 0; agg_kernel && k < d.n_group_by; k++)
    if (plan.keys[k].kind == KK_BIN && n_general)
      throw Error(PQ_ERR_UNSUPPORTED, "DATE_BIN keys need a flat-store copy of every page the query reads: " + shape->why_general);
  if (agg_kernel && plan.hashed && n_general)
    throw Error(PQ_ERR_UNSUPPORTED, "a hashed GROUP BY needs a flat-store copy of every page the query reads: " + shape->why_general);
  mark("side tables ready");
  // ---- shared-memory layout of k_scan (items the flat kernels do not take) ----
  SmemLayout L{};
  size_t smem_fixed = 0;
  if (n_general) {
    uint32_t off = align_up(uint32_t(sizeof(ScanCtl)), 128);
    for (uint32_t s = 0; s < ncols; s++) {
      // window = bytes of one slab at the widest index + one header per 8 values + alignment slop;
      // anything denser makes the kernel shrink the slab (always correct, only slower)
      L.defwin_cap[s] = plan.cols[s].max_def ? align_up(kSlabRows / 8 + kSlabRows / 16 + 64, 16) : 0;
      L.valwin_cap[s] = plan.cols[s].has_dict ? valwin_cap_for_bw(plan.cols[s].max_bw) : 0;
      // the slab index holds window-relative bit offsets: stage at least the window it was built for
      if (n_fast_items && plan.cols[s].has_dict) L.valwin_cap[s] = std::max(L.valwin_cap[s], table->col_valwin_cap[shape_cols[s]]);
      if (plan.cols[s].has_delta) L.valwin_cap[s] = std::max<uint32_t>(L.valwin_cap[s], align_up(kDeltaWindowBytes, 16));
      for (int b = 0; b < 2; b++) { L.defwin[s][b] = off; off += align_up(L.defwin_cap[s] + 16, 128); }
      for (int b = 0; b < 2; b++) { L.valwin[s][b] = off; off += align_up(L.valwin_cap[s] + 16, 128); }
      L.valid[s] = off; off += align_up((kSlabWords + 2) * 4, 16);
      L.rank[s] = off; off += kSlabWords * 4;
      // staging: u32 dictionary indices, or i64 values of DELTA_BINARY_PACKED pages
      L.idx[s] = (plan.cols[s].has_dict || plan.cols[s].has_delta) ? off : 0;
      off += plan.cols[s].has_delta ? kSlabRows * 8 : (plan.cols[s].has_dict ? kSlabRows * 4 : 0);
      L.defdir[s] = off; off += kMaxDirEntries * sizeof(DirEntry);
      for (int b = 0; b < 2; b++) {   // bulk-copy destination for prebuilt directories: 16-byte aligned
        off = align_up(off, 16);
        L.valdir[s][b] = off;
        off += std::max<uint32_t>(kMaxDirEntries * sizeof(DirEntry), plan.cols[s].has_delta ? kMaxDeltaEntries * sizeof(DeltaEntry) : 0);
      }
    }
    off = align_up(off, 16);
    L.recs = off; off += uint32_t(kRecBatch * std::max<uint32_t>(ncols, 1) * sizeof(DevSlabRec));
    L.leafT = off; off += std::max<uint32_t>(nleaves, 1) * kLeafWords * 4;
    L.sel = off; off += kSlabWords * 4;
    L.lutc = off; if (plan.fast_and) off += nleaves * kLutCacheBytes;
    off = align_up(off, 128);
    L.acc = off;
    smem_fixed = off;
  }

  // ---- shared-memory layout of the flat kernels ----
  FlatLayout FL{};
  if (n_flat) {
    // barriers, then one FlatStage record per stage (with plan.ncols column entries), then the stage buffers
    const uint32_t meta_stride = align_up(uint32_t(offsetof(FlatStage, col) + ncols * sizeof(FlatStageCol)), 16);
    const uint32_t ctl_bytes = align_up(uint32_t(sizeof(FlatCtl)), 128) + 128;   // + alignment slack of the first stage buffer
    FL.meta0 = align_up(uint32_t(sizeof(FlatCtl)), 16);
    FL.meta_stride = meta_stride;
    plan.direct8 = 0;
    plan.dbg = (getenv("PQB_FILTER_NOWORK") ? 1u : 0u) | (getenv("PQB_AGG_NOWORK") ? 2u : 0u);   // measurement: how fast can the producer + TMA feed the consumers?
    if (agg_kernel) plan.direct8 = 1;   // k_flat_agg reads 8-byte values in place (measured: 4 % faster than staging them, and room for twice the rows per slab)
    auto stage_bytes_for = [&](uint32_t S) {
      uint32_t off = 0;
      for (uint32_t s = 0; s < ncols; s++) {
        FL.col_off[s] = off;
        FL.col_voff[s] = off;
        if (!plan.cols[s].staged) continue;
        const uint32_t cap = std::max<uint32_t>((shape->flat_plain8[s] && !plan.direct8) ? S * 8 : 0, (S * std::max(shape->flat_max_bw[s], key_bw32[s]) + 7) / 8);
        off += align_up(cap + 48, 128);   // + the bit phase of a piece that starts inside a page, + over-read slack
        if (shape->flat_nullable[s]) { FL.col_voff[s] = off; off += align_up(S / 8 + 48, 128); }   // validity bits of pages with NULLs
      }
      return std::max<uint32_t>(off, 128);
    };
    const uint32_t avail = uint32_t(ctx.smem_optin()) - ctl_bytes - 256 - (agg_kernel ? 3 * meta_stride : 0);
    if (!agg_kernel) {
      // six CTAs per SM (160 threads, 64 registers): a CTA may use a sixth of the SM's shared memory.  A stage is one
      // warp's slab (<= 2048 rows); the ring is a power of two and at least as deep as there are consumer warps (a
      // ticket must never meet the stage's previous fill still pending: the barrier's parity has one bit)
      uint32_t ctas = 6;
      if (const char* e = getenv("PQB_FILTER_CTAS")) ctas = std::max(1, std::min(8, atoi(e)));   // experiment switch
      const uint32_t budget = (228u * 1024 - ctas * 1024) / ctas - ctl_bytes;
      uint32_t S = kFilterSlabRows;
      while (S > 128 && uint32_t(kFilterConsumerWarps) * (stage_bytes_for(S) + meta_stride) > budget) S >>= 1;
      FL.stage_bytes = stage_bytes_for(S);
      const uint32_t per = FL.stage_bytes + meta_stride;
      if (uint32_t(kFilterConsumerWarps) * per > avail) throw Error(PQ_ERR_UNSUPPORTED, "query needs more shared memory than one SM has");
      uint32_t n = std::max<uint32_t>(budget, uint32_t(kFilterConsumerWarps) * per) / per;
      if (const char* e = getenv("PQB_FILTER_STAGES")) n = std::min<uint32_t>(n, uint32_t(std::max(1, atoi(e))));   // experiment switch
      n = std::max<uint32_t>(uint32_t(kFilterConsumerWarps), std::min<uint32_t>(n, uint32_t(kFlatStagesMax)));
      while (n & (n - 1)) n &= n - 1;   // largest power of two
      FL.nstages = n;
      plan.flat_slab_rows = S;
      plan.hot_slots = 0;
    } else {
      // one CTA per SM: the hot part of the accumulator table next to the stages
      const uint32_t cell_bytes = plan.hot_cell_bytes;
      const uint64_t full = plan.hashed ? 0 : uint64_t(plan.nslots) * cell_bytes;   // hashed: no hot table in shared memory
      uint32_t krows = plan.hashed ? 4 : 8;   // the hashed instantiation exists for 4 rows per thread (64-bit slots: registers)
      if (const char* e = plan.hashed ? nullptr : getenv("PQB_AGG_KROWS")) krows = std::max(1, std::min(8, atoi(e)));   // experiment switch
      while (krows & (krows - 1)) krows &= krows - 1;
      while (krows > 1 && 2 * stage_bytes_for(kAggConsumers * krows) + std::min<uint64_t>(full, 96 * 1024) > avail) krows >>= 1;
      const uint32_t S = kAggConsumers * krows;
      FL.stage_bytes = stage_bytes_for(S);
      if (2 * FL.stage_bytes + cell_bytes > avail) throw Error(PQ_ERR_UNSUPPORTED, "query needs more shared memory than one SM has");
      FL.nstages = 2;
      uint32_t left = avail - 2 * FL.stage_bytes;
      if (full + FL.stage_bytes <= left && FL.nstages < (uint32_t)kFlatStagesMax) { FL.nstages = 3; left -= FL.stage_bytes; }
      if (const char* e = getenv("PQB_AGG_STAGES")) {   // experiment switch: a deeper ring at the price of hot slots
        const uint32_t want = uint32_t(std::max(2, std::min(int(kFlatStagesMax), atoi(e))));
        while (FL.nstages < want && left >= FL.stage_bytes + meta_stride + 64 * cell_bytes) { FL.nstages++; left -= FL.stage_bytes + meta_stride; }
      }
      // the hottest groups own a cell per lane (no same-address lanes inside a warp): 31 more cells each
      const uint32_t cap = left / cell_bytes;
      uint32_t T = 16;   // C4 with the narrow cells: 16 beats 8 by 2.4 %, 32 by 1 % more (profiles/probe_ab_summary_r3.md)
      if (const char* e = getenv("PQB_LANE_SLOTS")) T = uint32_t(std::max(0, atoi(e)));   // experiment switch
      if (const char* e = getenv("PQB_F64_GLOBAL")) if (atoi(e)) T = 0;   // that experiment sends hot f64 cells to L2 by SLOT: no per-lane cells
      T = std::min<uint32_t>(T, plan.nslots);
      while (T && cap < 64u * T) T >>= 1;
      if (plan.hashed) T = 0;
      plan.lane_slots = T;
      plan.hot_slots = plan.hashed ? 0u : uint32_t(std::min<uint64_t>(plan.nslots, cap - 31u * T));
      if (const char* hs = plan.hashed ? nullptr : getenv("PQB_HOT_SLOTS")) plan.hot_slots = std::max(T, std::min<uint32_t>(plan.hot_slots, uint32_t(atoi(hs))));   // experiment switch
      plan.flat_slab_rows = S;
      plan.flat_krows = krows;
      // hot table planes: the 8-byte ones first, so that every cell is aligned to its width
      const uint32_t Hs = plan.hot_slots + 31u * T;
      uint32_t off = 0;
      for (int pass = 0; pass < 2; pass++)
        for (uint32_t p = 0; p < cells; p++) {
          const bool w8 = p >= 1 && p <= plan.n_acc && !((plan.acc_narrow >> (p - 1)) & 1u);
          if (w8 != (pass == 0)) continue;
          plan.hot_off[p] = off;
          off += Hs * (w8 ? 8u : 4u);
        }
    }
    FL.stage0 = align_up(FL.meta0 + FL.nstages * meta_stride, 128);
    FL.acc = align_up(FL.stage0 + FL.nstages * FL.stage_bytes, 128);
    FL.total = FL.acc + (agg_kernel ? (plan.hot_slots + 31u * plan.lane_slots) * plan.hot_cell_bytes : 0);
    if (FL.total > ctx.smem_optin()) throw Error(PQ_ERR_UNSUPPORTED, "query needs more shared memory than one SM has");
  }

  // ---- per-query device state ----
  Timer t_all, t_scan;
  PQB_CUDA(cudaEventRecord(t_all.a, stream));
  DevBuf<uint8_t> d_lit; d_lit.upload(lit_pool, stream);
  DevBuf<uint8_t> d_live;
  const bool pruned = nrg < nrg_table;
  if (pruned) d_live.upload(rg_live, stream);
  DevBuf<uint8_t> d_luts; d_luts.alloc(std::max<uint64_t>(lut_total, 16), stream);
  DevBuf<unsigned long long> d_counters; d_counters.alloc(8, stream); d_counters.zero();
  metrics.h2d_bytes += lit_pool.size() + (pruned ? rg_live.size() : 0);

  pa.arena = table->d_arena;
  pa.chunks = shape->d_chunks;
  pa.n_chunks = nrg_table * ncols;
  pa.ncols = ncols;
  pa.rg_live = pruned ? d_live.p : nullptr;
  pa.luts = d_luts.p;
  pa.lit_pool = d_lit.p;
  pa.counters = d_counters.p;
  if (nrg && ncols && any_lut) {
    dim3 grid(pa.n_chunks, std::min<uint32_t>((max_dict_n + 255) / 256, 64));
    k_leaf_luts<<<grid, 256, 0, stream>>>(pa, plan);
    launches++;
  }

  // ---- accumulators ----
  DevBuf<unsigned long long> d_acc, d_hkeys;
  size_t smem_total = smem_fixed;
  plan.replicas = 1;
  plan.smem_share = 8;
  plan.f64_global = 0;
  if (const char* e = getenv("PQB_SMEM_SHARE")) plan.smem_share = uint32_t(atoi(e));
  if (const char* e = getenv("PQB_F64_GLOBAL")) plan.f64_global = uint32_t(atoi(e));
  plan.f64_smem = 0;
  if (const char* e = getenv("PQB_F64_SMEM")) plan.f64_smem = uint32_t(atoi(e));   // A/B switch: f64 sums of every hot slot in shared memory
  if (agg_kernel) {
    bool f64_add = false;   // an f64 SUM / AVG: the hot slots without per-lane cells send it to L2
    for (uint32_t a = 0; a < plan.naggs; a++)
      f64_add |= plan.aggs[a].fn == AG_AVG || (plan.aggs[a].fn == AG_SUM && plan.aggs[a].kind == DK_F64);
    const bool f64_l2 = f64_add && !plan.f64_smem && plan.hot_slots > plan.lane_slots;
    // Cold group slots go to L2 with fire-and-forget reductions; L2 serialises same-address atomics, so the
    // table is kept in a few copies (CTA b adds into copy b mod replicas) as long as all copies stay L2 resident.
    if (n_flat && (plan.hot_slots < plan.nslots || plan.smem_share < 8 || plan.f64_global || f64_l2)) {
      const uint64_t tbytes = uint64_t(plan.nslots) * cells * 8;
      uint32_t r = uint32_t(std::min<uint64_t>(32, (48ull << 20) / std::max<uint64_t>(tbytes, 1)));
      if (const char* e = getenv("PQB_REPLICAS")) r = uint32_t(atoi(e));
      plan.replicas = std::max<uint32_t>(1, std::min<uint32_t>(r, uint32_t(ctx.sm_count())));
    }
    if (plan.hashed) {
      plan.replicas = 1;
      d_hkeys.alloc(plan.nslots, stream);
      PQB_CUDA(cudaMemsetAsync(d_hkeys.p, 0xff, size_t(plan.nslots) * 8, stream));
    }
    d_acc.alloc(size_t(plan.nslots) * cells * plan.replicas, stream);
    {
      const uint64_t ncell = uint64_t(plan.nslots) * cells * plan.replicas;
      k_acc_init<<<uint32_t(std::min<uint64_t>(2048, (ncell + 255) / 256)), 256, 0, stream>>>(d_acc.p, plan.nslots, plan.n_acc, cells, plan.replicas, plan);
    }
    launches++;
    size_t acc_bytes = size_t(plan.nslots) * cells * 8;
    if (n_general && smem_fixed + acc_bytes + 1024 <= ctx.smem_optin()) { plan.smem_acc = 1; smem_total = smem_fixed + acc_bytes; }
  }
  L.total = uint32_t(smem_total);
  if (smem_total > ctx.smem_optin()) throw Error(PQ_ERR_UNSUPPORTED, "query needs more shared memory than one SM has");

  // ---- selection bitmap / counts ----
  const bool projecting = want_rows && d.n_projection > 0;
  if (projecting && n_general)
    throw Error(PQ_ERR_UNSUPPORTED, "projection of column values needs a flat-store copy of every page it reads: PLAIN (dictionary-fallback) "
                                    "string pages are not projected on the GPU yet: " + shape->why_general);
  plan.write_bitmap = want_rows ? 1 : 0;
  DevBuf<uint32_t> d_bitmap, d_item_counts;
  // k_scan ORs partial words into its bitmap regions: they start zeroed.  The flat filter kernel stores
  // every word of its items, no memset needed.
  if (want_rows) { d_bitmap.alloc(std::max<uint32_t>(shape->bitmap_words, 1), stream); if (n_general) d_bitmap.zero(); }
  d_item_counts.alloc(std::max<size_t>(items.size(), 1), stream);
  d_item_counts.zero();
  if (want_rows) algo_bytes += metrics.rows_scanned / 8;
  metrics.algorithmic_bytes = algo_bytes;

  mark("prep kernels queued");
  // ---- the fused scans ----
  DevScanArgs sa{};
  sa.arena = table->d_arena;
  sa.pages = table->d_pages;
  sa.chunks = shape->d_chunks;
  sa.items = shape->d_items;
  sa.luts = d_luts.p;
  sa.lit_pool = d_lit.p;
  sa.rg_live = pruned ? d_live.p : nullptr;
  sa.flat = table->d_flat;
  sa.fpages = d_kpages.p ? d_kpages.p : table->d_flat_pages;
  sa.bitmap = d_bitmap.p;
  sa.item_counts = d_item_counts.p;
  sa.acc = d_acc.p;
  sa.hkeys = d_hkeys.p;
  sa.counters = d_counters.p;
  sa.slab_recs = table->d_slab_recs;
  sa.slab_dirs = table->d_slab_dirs;
  PQB_CUDA(cudaEventRecord(t_scan.a, stream));
  if (n_flat && nrg) {
    uint32_t grid;
    if (agg_kernel) {
      grid = std::min<uint32_t>(n_flat, uint32_t(ctx.sm_count()));
      if (const char* g = getenv("PQB_GRID")) grid = std::max(1, atoi(g));
      auto go = [&](auto kern) {
        PQB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(ctx.smem_optin())));
        kern<<<grid, kAggThreads, FL.total, stream>>>(plan, FL, sa);
      };
      if (plan.hashed) go(k_flat_agg<4, true>);           // key space wider than the dense table: cells through the hash table
      else if (plan.flat_krows >= 8) go(k_flat_agg<8, false>);   // rows per thread and slab: the widest instantiation the stages leave room for
      else if (plan.flat_krows >= 4) go(k_flat_agg<4, false>);
      else go(k_flat_agg<2, false>);
    } else {
      auto go = [&](auto kern) {
        PQB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(ctx.smem_optin())));
        int occ = 1;
        PQB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kFilterThreads, FL.total));
        if (occ < 1) occ = 1;
        grid = std::min<uint32_t>(n_flat, uint32_t(ctx.sm_count() * occ));
        if (const char* g = getenv("PQB_GRID")) grid = std::max(1, atoi(g));
        kern<<<grid, kFilterThreads, FL.total, stream>>>(plan, FL, sa);
      };
      if (plan.conj || !plan.npred) go(k_flat_filter<true>);   // conjunctions: the instantiation without the Kleene stack
      else go(k_flat_filter<false>);
    }
    PQB_CUDA(cudaGetLastError());
    launches++;
    if (verbose)
      fprintf(stderr, "[pqb] %s: %u CTAs, %u B smem/CTA, %u stages x %u B, slab %u rows, hot slots %u of %u, %u copies, %u flat items\n",
              agg_kernel ? "k_flat_agg" : "k_flat_filter", grid, FL.total, FL.nstages, FL.stage_bytes, plan.flat_slab_rows, plan.hot_slots,
              plan.nslots, plan.replicas, n_flat);
  }
  if (n_general && nrg) {
    if (n_flat) { PQB_CUDA(cudaMemsetAsync(d_counters.p + 2, 0, 8, stream)); }   // the work-queue head
    PQB_CUDA(cudaFuncSetAttribute(k_scan, cudaFuncAttributeMaxDynamicSharedMemorySize, int(ctx.smem_optin())));
    int occ = 1;
    PQB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_scan, kScanThreads, smem_total));
    if (occ < 1) occ = 1;
    uint32_t grid = std::min<uint32_t>(uint32_t(items.size()), uint32_t(ctx.sm_count() * occ));
    if (const char* g = getenv("PQB_GRID")) grid = std::max(1, atoi(g));   // debugging aid: forces several items per CTA
    if (verbose)
      fprintf(stderr, "[pqb] k_scan: %u CTAs x %d threads, %zu B smem/CTA, %d CTAs/SM, %u of %zu items (%u slab-indexed)\n", grid,
              kScanThreads, size_t(smem_total), occ, n_general, items.size(), n_fast_items);
    k_scan<<<grid, kScanThreads, smem_total, stream>>>(plan, L, sa);
    PQB_CUDA(cudaGetLastError());
    launches++;
  }
  if (agg_kernel && plan.replicas > 1) {
    k_acc_reduce<<<std::min<uint32_t>(1024, (plan.nslots * cells + 255) / 256), 256, 0, stream>>>(d_acc.p, plan.nslots, cells, plan.replicas, plan);
    launches++;
  }
  PQB_CUDA(cudaEventRecord(t_scan.b, stream));

  if (getenv("PQB_DEBUG_ITEMS")) {
    std::vector<uint32_t> ic(items.size());
    PQB_CUDA(cudaMemcpyAsync(ic.data(), d_item_counts.p, ic.size() * 4, cudaMemcpyDeviceToHost, stream));
    PQB_CUDA(cudaStreamSynchronize(stream));
    for (size_t i = 0; i < ic.size(); i++)
      fprintf(stderr, "item %zu rg %u row0 %u nrows %u g0 %llu flags %u count %u\n", i, items[i].rg, items[i].row0, items[i].nrows,
              (unsigned long long)items[i].global_row0, items[i].fast, ic[i]);
  }
  mark("scan queued");

  // ---- results ----
  const uint32_t batch_rows = d.batch_size ? d.batch_size : 20000;
  batch_rows_ = batch_rows;
  unsigned long long h_counters[4] = {0, 0, 0, 0};
  if (agg_kernel) {
    // multi-GPU: the partial tables meet in ONE grouped all-reduce (SURVEY §8e): one NCCL launch,
    // per array the reduction its aggregate needs
    Timer t_ar;
    if (allreduce) {
      PQB_CUDA(cudaEventRecord(t_ar.a, stream));
      comm_group_begin();
      comm_allreduce_u64(d_acc.p, plan.nslots, 0, stream);
      for (uint32_t a = 0; a < plan.n_acc; a++) {
        uint8_t how = plan.acc_init[a];
        comm_allreduce_u64(d_acc.p + size_t(1 + a) * plan.nslots, plan.nslots, how == 0 ? 0 : how == 1 ? 3 : how == 2 ? 1 : 2, stream);
      }
      if (plan.n_nn) comm_allreduce_u64(d_acc.p + size_t(1 + plan.n_acc) * plan.nslots, size_t(plan.n_nn) * plan.nslots, 0, stream);
      comm_group_end();
      PQB_CUDA(cudaEventRecord(t_ar.b, stream));
    }
    // ---- non-empty groups in ascending slot order (deterministic: the mixed radix of the group ids) ----
    const uint32_t ntiles = (plan.nslots + kSlotTile - 1) / kSlotTile;
    const uint64_t out_cap = std::min<uint64_t>(plan.nslots, std::max<uint64_t>(allreduce ? plan.nslots : metrics.rows_scanned, 1));
    DevBuf<uint32_t> d_tile_counts, d_out_slot;
    DevBuf<unsigned long long> d_tile_base, d_totals;
    d_tile_counts.alloc(ntiles, stream);
    d_tile_base.alloc(ntiles, stream);
    d_totals.alloc(2, stream);
    d_out_slot.alloc(out_cap, stream);
    k_slot_tile_counts<<<ntiles, 256, 0, stream>>>(d_acc.p, plan.nslots, d_tile_counts.p);
    k_item_prefix<<<1, 1024, 0, stream>>>(d_tile_counts.p, ntiles, d_tile_base.p, d_totals.p);
    k_slot_compact<<<ntiles, 256, 0, stream>>>(d_acc.p, plan.nslots, d_tile_base.p, d_out_slot.p);
    // rows this rank selected (its own items)
    DevBuf<unsigned long long> d_item_base;
    d_item_base.alloc(std::max<size_t>(items.size(), 1), stream);
    if (!items.empty()) k_item_prefix<<<1, 1024, 0, stream>>>(d_item_counts.p, uint32_t(items.size()), d_item_base.p, d_totals.p + 1);
    else PQB_CUDA(cudaMemsetAsync(d_totals.p + 1, 0, 8, stream));
    launches += 4;
    unsigned long long totals[2] = {0, 0};
    PQB_CUDA(cudaMemcpyAsync(totals, d_totals.p, 16, cudaMemcpyDeviceToHost, stream));
    PQB_CUDA(cudaMemcpyAsync(h_counters, d_counters.p, sizeof(h_counters), cudaMemcpyDeviceToHost, stream));
    PQB_CUDA(cudaStreamSynchronize(stream));
    metrics.d2h_bytes += 16 + sizeof(h_counters);
    if (plan.hashed && h_counters[1] == 100) throw Error(PQ_ERR_UNSUPPORTED, "GROUP BY: more distinct groups than the hashed accumulator table holds (2^26)");
    if (h_counters[1]) throw Error(PQ_ERR_CORRUPT, "corrupt or unsupported page encoding met on the device (code " + std::to_string(h_counters[1]) + ")");
    const uint32_t n_out = uint32_t(totals[0]);
    metrics.rows_selected = totals[1];
    if (allreduce) { float ms = 0; cudaEventElapsedTime(&ms, t_ar.a, t_ar.b); metrics.allreduce_ms = ms; }
    static const char* fn_names[] = {"count(*)", "count", "sum", "min", "max", "avg"};
    auto agg_name = [&](uint32_t a) {
      const DevAgg& ag = plan.aggs[a];
      return ag.fn == AG_COUNT_STAR ? std::string("count(*)") : std::string(fn_names[ag.fn]) + "(" + d.columns[d.aggs[a].col].name + ")";
    };
    if (d.n_group_by == 0 && n_out == 0) {
      // SQL: a global aggregate over zero rows still yields one row: COUNT = 0, everything else NULL
      OutBatch ob;
      ob.rows = 1;
      for (uint32_t a = 0; a < d.n_aggs; a++) {
        OutColumn oc;
        oc.name = agg_name(a);
        oc.type = agg_out_type[a];
        oc.values.assign(8, 0);
        const bool is_count = plan.aggs[a].fn == AG_COUNT_STAR || plan.aggs[a].fn == AG_COUNT;
        if (!is_count) { oc.validity.assign(1, 0); oc.null_count = 1; }
        ob.cols.push_back(std::move(oc));
      }
      metrics.groups = 1;
      batches_.push_back(std::move(ob));
      PQB_CUDA(cudaEventRecord(t_all.b, stream));
      PQB_CUDA(cudaStreamSynchronize(stream));
    } else if (n_out == 0) {
      metrics.groups = 0;
      PQB_CUDA(cudaEventRecord(t_all.b, stream));
      PQB_CUDA(cudaStreamSynchronize(stream));
    } else {
      // ---- the result block: every buffer of every batch, assembled on the device ----
      FinishArgs fa{};
      const uint32_t nbatches = (n_out + batch_rows - 1) / batch_rows;
      const uint32_t wpb = (batch_rows + 31) / 32;
      const uint32_t ncolumns = d.n_group_by + d.n_aggs;
      uint64_t off = 0;
      auto take = [&](uint64_t bytes) { uint64_t o = off; off = (off + bytes + 63) & ~63ull; return o; };
      const uint64_t nulls_off = take(uint64_t(ncolumns) * nbatches * 4);
      for (uint32_t k = 0; k < d.n_group_by; k++) {
        FinishKey& fk = fa.keys[k];
        const uint8_t kind = plan.cols[plan.keys[k].col].kind;
        fk.kind = kind;
        fk.stride = plan.keys[k].stride;
        fk.wstride = plan.keys[k].wstride;
        fk.card = qk[k].card;
        fk.valid_off = take(uint64_t(nbatches) * wpb * 4);
        if (kind == DK_BOOL) fk.val_off = take(uint64_t(nbatches) * wpb * 4);
        else if (kind == DK_STR) fk.val_off = take((uint64_t(n_out) + 1) * 4);
        else fk.val_off = take(uint64_t(n_out) * 8);
        if (qk[k].is_bin) {
          fk.is_bin = 1;
          fk.bin_base = plan.keys[k].bin_base;
          fk.bin_width = plan.keys[k].bin_width;
        } else if (kind != DK_BOOL) {
          const ColSide& cs = table->sides[shape_cols[plan.keys[k].col]];
          if (multi) {   // the dictionary every rank agreed on
            fk.kd_offs = cs.d_glob_kd_offs;
            fk.kd_bytes = cs.d_glob_kd_bytes;
          } else {
            fk.kd_offs = cs.d_kd_offs;
            fk.kd_bytes = cs.d_kd_bytes;
          }
        }
      }
      for (uint32_t a = 0; a < d.n_aggs; a++) {
        fa.aggs[a] = plan.aggs[a];
        fa.nn_is_rows[a] = nn_is_rows[a];
        fa.valid_off[a] = take(uint64_t(nbatches) * wpb * 4);
        fa.val_off[a] = take(uint64_t(n_out) * 8);
      }
      // string key bytes: an upper bound (rows x the longest distinct value) keeps the copy to one round trip
      for (uint32_t k = 0; k < d.n_group_by; k++) {
        FinishKey& fk = fa.keys[k];
        if (fk.kind != DK_STR) continue;
        uint64_t max_len = 0;
        const KeyDict* kd = qk[k].kd;
        max_len = multi ? table->sides[shape_cols[plan.keys[k].col]].glob_max_len : table->sides[shape_cols[plan.keys[k].col]].kd_max_len;
        const uint64_t bound = std::min<uint64_t>(uint64_t(n_out) * max_len, uint64_t(n_out / std::max<uint32_t>(fk.card, 1) + 1) * kd->bytes.size());
        if (bound > 0x7fffffffull) throw Error(PQ_ERR_UNSUPPORTED, "group key strings of one result exceed 2 GiB");
        fk.data_off = take(bound);
      }
      const uint64_t copy_bytes = off;
      for (uint32_t k = 0; k < d.n_group_by; k++)
        if (fa.keys[k].kind == DK_STR) fa.keys[k].len_off = take(uint64_t(n_out) * 4);   // device-only scratch behind the copied part
      DevBuf<uint8_t> d_block;
      d_block.alloc(off, stream);
      PQB_CUDA(cudaMemsetAsync(d_block.p, 0, copy_bytes, stream));
      fa.acc = d_acc.p;
      fa.wide = plan.hashed ? d_hkeys.p : nullptr;
      fa.out_slot = d_out_slot.p;
      fa.out = d_block.p;
      fa.nulls = reinterpret_cast<uint32_t*>(d_block.p + nulls_off);
      fa.n_out = n_out;
      fa.nslots = plan.nslots;
      fa.n_acc = plan.n_acc;
      fa.naggs = d.n_aggs;
      fa.nkeys = d.n_group_by;
      fa.batch_rows = batch_rows;
      fa.words_per_batch = wpb;
      fa.nbatches = nbatches;
      k_agg_finish<<<(n_out + 255) / 256, 256, 0, stream>>>(fa);
      launches++;
      for (uint32_t k = 0; k < d.n_group_by; k++) {
        if (fa.keys[k].kind != DK_STR) continue;
        k_offsets_scan<<<1, 1024, 0, stream>>>(reinterpret_cast<const uint32_t*>(d_block.p + fa.keys[k].len_off), n_out,
                                               reinterpret_cast<int32_t*>(d_block.p + fa.keys[k].val_off));
        k_key_gather<<<uint32_t((uint64_t(n_out) * 32 + 255) / 256), 256, 0, stream>>>(fa, k);
        launches += 2;
      }
      PQB_CUDA(cudaGetLastError());
      auto block = std::make_shared<PinnedBlock>();
      block->p = ctx.pinned_acquire(copy_bytes);
      block->bytes = copy_bytes;
      PQB_CUDA(cudaMemcpyAsync(block->p, d_block.p, copy_bytes, cudaMemcpyDeviceToHost, stream));
      PQB_CUDA(cudaEventRecord(t_all.b, stream));
      PQB_CUDA(cudaStreamSynchronize(stream));
      if (copy_bytes <= kKeepDeviceResult) { block->dev = d_block.p; d_block.p = nullptr; dev_blocks_.push_back(block); }   // JSON egress formats it where it is
      metrics.d2h_bytes += copy_bytes;
      metrics.groups = n_out;
      const uint32_t* nulls = reinterpret_cast<const uint32_t*>(block->p + nulls_off);
      for (uint32_t b = 0; b < nbatches; b++) {
        const uint32_t r0 = b * batch_rows, nb = std::min(batch_rows, n_out - r0);
        OutBatch ob;
        ob.rows = nb;
        for (uint32_t c = 0; c < ncolumns; c++) {
          OutColumn oc;
          oc.ext = block;
          oc.ext_all = true;
          oc.null_count = nulls[c * nbatches + b];
          if (c < d.n_group_by) {
            const FinishKey& fk = fa.keys[c];
            const uint32_t qc = uint32_t(d.group_by[c]);
            oc.name = fk.is_bin ? std::string("date_bin(") + d.columns[qc].name + ")" : std::string(d.columns[qc].name);
            oc.type = fk.is_bin ? PQ_T_TS_MS : out_type_of(qc);
            oc.ext_validity_off = fk.valid_off + uint64_t(b) * wpb * 4;
            if (fk.kind == DK_STR) { oc.ext_offsets_off = fk.val_off + uint64_t(r0) * 4; oc.ext_off = fk.data_off; }
            else if (fk.kind == DK_BOOL) oc.ext_off = fk.val_off + uint64_t(b) * wpb * 4;
            else oc.ext_off = fk.val_off + uint64_t(r0) * 8;
          } else {
            const uint32_t a = c - d.n_group_by;
            oc.name = agg_name(a);
            oc.type = agg_out_type[a];
            oc.ext_validity_off = fa.valid_off[a] + uint64_t(b) * wpb * 4;
            oc.ext_off = fa.val_off[a] + uint64_t(r0) * 8;
          }
          ob.cols.push_back(std::move(oc));
        }
        batches_.push_back(std::move(ob));
      }
    }
  } else {
    // ---- filter / COUNT(*) ----
    // bitmap-driven stream compaction on the device: per-item prefix, then one CTA per item.  The
    // selected-row total is needed on the host to size the result; a repeat of the same query shape
    // sizes it from the previous answer and skips that round trip.
    DevBuf<unsigned long long> d_item_base, d_total, d_ids;
    std::shared_ptr<PinnedBlock> ids_block;   // selected row ordinals land in page-locked memory, batches alias it
    unsigned long long n_ids = 0, total = 0;
    d_total.alloc(1, stream);
    d_item_base.alloc(std::max<size_t>(items.size(), 1), stream);
    if (!items.empty()) {
      k_item_prefix<<<1, 1024, 0, stream>>>(d_item_counts.p, uint32_t(items.size()), d_item_base.p, d_total.p);
      launches++;
    } else {
      PQB_CUDA(cudaMemsetAsync(d_total.p, 0, 8, stream));
    }
    PQB_CUDA(cudaMemcpyAsync(h_counters, d_counters.p, sizeof(h_counters), cudaMemcpyDeviceToHost, stream));
    PQB_CUDA(cudaMemcpyAsync(&total, d_total.p, 8, cudaMemcpyDeviceToHost, stream));
    metrics.d2h_bytes += 8 + sizeof(h_counters);
    const unsigned long long lim = d.limit >= 0 ? (unsigned long long)d.limit : ~0ull;
    if (projecting) {
      // ---- TableProvider::scan(projection): gather the projected columns of the selected rows ----
      struct PC { uint32_t qcol; uint32_t slot; uint8_t kind; std::string name; int type; };
      std::vector<PC> pcs;
      for (uint32_t i = 0; i < d.n_projection; i++) {
        const uint32_t qc = uint32_t(d.projection[i]);
        pcs.push_back({qc, uint32_t(slot_of[qc]), plan.cols[slot_of[qc]].kind, d.columns[qc].name, out_type_of(qc)});
        if (pcs.back().kind == DK_STR) table->ensure_ent_off(shape_cols[slot_of[qc]], stream);
      }
      if (d.flags & PQ_QUERY_EMIT_ROW_IDS) pcs.push_back({0, 0xffffffffu, DK_I64, "__row_id", PQ_T_I64});
      const uint32_t npc = uint32_t(pcs.size());
      std::shared_ptr<PinnedBlock> block;
      ProjArgs pj{};
      uint64_t nulls_off = 0, copy_bytes = 0;
      uint32_t nbatches = 0;
      const uint32_t wpb = (batch_rows + 31) / 32;
      unsigned long long n_rows = 0;
      DevBuf<uint8_t> d_block;
      auto gather = [&](unsigned long long cap) {
        nbatches = uint32_t((cap + batch_rows - 1) / batch_rows);
        uint64_t off = 0;
        auto take = [&](uint64_t bytes) { uint64_t o = off; off = (off + bytes + 63) & ~63ull; return o; };
        nulls_off = take(uint64_t(npc) * nbatches * 4);
        for (uint32_t c = 0; c < npc; c++) {
          ProjCol& pc = pj.cols[c];
          pc = ProjCol{};
          pc.slot = pcs[c].slot;
          pc.kind = pcs[c].kind;
          pc.valid_off = take(uint64_t(nbatches) * wpb * 4);
          if (pc.kind == DK_BOOL) pc.val_off = take(uint64_t(nbatches) * wpb * 4);
          else if (pc.kind == DK_STR) pc.val_off = take((cap + 1) * 4);
          else pc.val_off = take(cap * 8);
        }
        for (uint32_t c = 0; c < npc; c++) {
          ProjCol& pc = pj.cols[c];
          if (pc.kind != DK_STR) continue;
          const ColSide& cs = table->sides[shape_cols[pc.slot]];
          pc.ent = cs.d_ent_off;
          const uint64_t bound = cap * uint64_t(std::max(cs.max_ent_len, cs.max_plain_len));
          if (bound > 0x7fffffffull) throw Error(PQ_ERR_UNSUPPORTED, "projected strings of one result exceed 2 GiB: add a LIMIT");
          pc.data_off = take(bound);
        }
        copy_bytes = off;
        for (uint32_t c = 0; c < npc; c++)
          if (pj.cols[c].kind == DK_STR) { pj.cols[c].src_off = take(cap * 8); pj.cols[c].len_off = take(cap * 4); }
        d_block.alloc(off, stream);
        PQB_CUDA(cudaMemsetAsync(d_block.p, 0, off, stream));
        pj.arena = table->d_arena;
        pj.flat = table->d_flat;
        pj.fpages = table->d_flat_pages;
        pj.chunks = shape->d_chunks;
        pj.items = shape->d_items;
        pj.bitmap = d_bitmap.p;
        pj.item_counts = d_item_counts.p;
        pj.item_base = d_item_base.p;
        pj.out = d_block.p;
        pj.nulls = reinterpret_cast<uint32_t*>(d_block.p + nulls_off);
        pj.n_out = cap;
        pj.n_items = uint32_t(items.size());
        pj.plan_ncols = ncols;
        pj.ncols = npc;
        pj.batch_rows = batch_rows;
        pj.words_per_batch = wpb;
        pj.nbatches = nbatches;
        const uint32_t grid = std::min<uint32_t>(uint32_t(items.size()), uint32_t(ctx.sm_count() * 8));
        k_project<<<grid, 256, 0, stream>>>(pj);
        launches++;
        for (uint32_t c = 0; c < npc; c++) {
          if (pj.cols[c].kind != DK_STR) continue;
          // rows beyond the selected total have length 0: the scan over `cap` rows is exact
          k_offsets_scan<<<1, 1024, 0, stream>>>(reinterpret_cast<const uint32_t*>(d_block.p + pj.cols[c].len_off), uint32_t(cap),
                                                 reinterpret_cast<int32_t*>(d_block.p + pj.cols[c].val_off));
          k_project_bytes<<<uint32_t((cap * 32 + 255) / 256), 256, 0, stream>>>(pj, c, cap);
          launches += 2;
        }
        PQB_CUDA(cudaGetLastError());
        block = std::make_shared<PinnedBlock>();
        block->p = ctx.pinned_acquire(copy_bytes);
        block->bytes = copy_bytes;
        PQB_CUDA(cudaMemcpyAsync(block->p, d_block.p, copy_bytes, cudaMemcpyDeviceToHost, stream));
      };
      if (!items.empty()) {
        const unsigned long long hint = shape->last_total.load();
        bool done = false;
        if (hint != ~0ull) {
          const unsigned long long cap = std::max<unsigned long long>(1, std::min(lim, hint + hint / 8 + 1024));
          if (cap > 0x7ffffff0ull) throw Error(PQ_ERR_UNSUPPORTED, "more than 2^31 projected rows in one result: add a LIMIT");
          gather(cap);
          PQB_CUDA(cudaStreamSynchronize(stream));
          if (std::min(total, lim) <= cap) { done = true; n_rows = std::min(total, lim); metrics.d2h_bytes += copy_bytes; }
          else block.reset();
        } else {
          PQB_CUDA(cudaStreamSynchronize(stream));
        }
        if (!done) {
          const unsigned long long keep = std::min(total, lim);
          if (keep > 0x7ffffff0ull) throw Error(PQ_ERR_UNSUPPORTED, "more than 2^31 projected rows in one result: add a LIMIT");
          if (keep) {
            gather(keep);
            PQB_CUDA(cudaStreamSynchronize(stream));
            metrics.d2h_bytes += copy_bytes;
          }
          n_rows = keep;
        }
        shape->last_total.store(total);
      }
      PQB_CUDA(cudaEventRecord(t_all.b, stream));
      PQB_CUDA(cudaStreamSynchronize(stream));
      if (h_counters[1]) throw Error(PQ_ERR_CORRUPT, "corrupt or unsupported page encoding met on the device (code " + std::to_string(h_counters[1]) + ")");
      if (block && d_block.p && copy_bytes <= kKeepDeviceResult) { block->dev = d_block.p; d_block.p = nullptr; dev_blocks_.push_back(block); }
      metrics.rows_selected = total;
      const uint32_t out_batches = n_rows ? uint32_t((n_rows + batch_rows - 1) / batch_rows) : 1u;
      for (uint32_t b = 0; b < out_batches; b++) {
        const unsigned long long r0 = uint64_t(b) * batch_rows;
        const uint32_t nb = n_rows ? uint32_t(std::min<unsigned long long>(batch_rows, n_rows - r0)) : 0u;
        OutBatch ob;
        ob.rows = nb;
        for (uint32_t c = 0; c < npc; c++) {
          OutColumn oc;
          oc.name = pcs[c].name;
          oc.type = pcs[c].type;
          if (nb) {
            const ProjCol& pc = pj.cols[c];
            oc.ext = block;
            oc.ext_all = true;
            oc.null_count = reinterpret_cast<const uint32_t*>(block->p + nulls_off)[c * nbatches + b];
            oc.ext_validity_off = pc.valid_off + uint64_t(b) * wpb * 4;
            if (pc.kind == DK_STR) { oc.ext_offsets_off = pc.val_off + r0 * 4; oc.ext_off = pc.data_off; }
            else if (pc.kind == DK_BOOL) oc.ext_off = pc.val_off + uint64_t(b) * wpb * 4;
            else oc.ext_off = pc.val_off + r0 * 8;
          } else if (oc.type == PQ_T_UTF8) oc.offsets.assign(1, 0);
          ob.cols.push_back(std::move(oc));
        }
        batches_.push_back(std::move(ob));
      }
      float ms = 0;
      cudaEventElapsedTime(&ms, t_all.a, t_all.b);
      metrics.device_ms = ms;
      if (!items.empty() && nrg) { cudaEventElapsedTime(&ms, t_scan.a, t_scan.b); metrics.scan_kernel_ms = ms; }
      metrics.kernel_launches = launches;
      return;
    }
    if (want_rows && !items.empty()) {
      unsigned long long hint = shape->last_total.load();
      bool done = false;
      if (hint != ~0ull) {
        // optimistic pass: room for the previous answer plus a margin
        unsigned long long cap = std::min(lim, hint + hint / 8 + 1024);
        if (cap) {
          d_ids.alloc(cap, stream);
          uint32_t grid = std::min<uint32_t>(uint32_t(items.size()), uint32_t(ctx.sm_count() * 8));
          k_compact_row_ids<<<grid, 256, 0, stream>>>(d_bitmap.p, shape->d_items, d_item_counts.p, d_item_base.p, uint32_t(items.size()), d_ids.p, cap);
          launches++;
          ids_block = std::make_shared<PinnedBlock>();
          ids_block->p = ctx.pinned_acquire(cap * 8);
          ids_block->bytes = cap * 8;
          PQB_CUDA(cudaMemcpyAsync(ids_block->p, d_ids.p, cap * 8, cudaMemcpyDeviceToHost, stream));
        }
        PQB_CUDA(cudaStreamSynchronize(stream));
        const unsigned long long keep = std::min(total, lim);
        if (keep <= cap) { done = true; n_ids = keep; metrics.d2h_bytes += cap * 8; }
        else ids_block.reset();
      } else {
        PQB_CUDA(cudaStreamSynchronize(stream));
      }
      mark("scan done, selected-row total on host");
      if (!done) {
        const unsigned long long keep = std::min(total, lim);
        if (keep) {
          DevBuf<unsigned long long> d_ids2;
          d_ids2.alloc(keep, stream);
          uint32_t grid = std::min<uint32_t>(uint32_t(items.size()), uint32_t(ctx.sm_count() * 8));
          k_compact_row_ids<<<grid, 256, 0, stream>>>(d_bitmap.p, shape->d_items, d_item_counts.p, d_item_base.p, uint32_t(items.size()), d_ids2.p, keep);
          launches++;
          ids_block = std::make_shared<PinnedBlock>();
          ids_block->p = ctx.pinned_acquire(keep * 8);
          ids_block->bytes = keep * 8;
          n_ids = keep;
          PQB_CUDA(cudaMemcpyAsync(ids_block->p, d_ids2.p, keep * 8, cudaMemcpyDeviceToHost, stream));
          PQB_CUDA(cudaStreamSynchronize(stream));
          metrics.d2h_bytes += keep * 8;
        }
      }
      shape->last_total.store(total);
    }
    PQB_CUDA(cudaEventRecord(t_all.b, stream));
    PQB_CUDA(cudaStreamSynchronize(stream));
    mark("results on host");
    if (h_counters[1]) throw Error(PQ_ERR_CORRUPT, "corrupt or unsupported page encoding met on the device (code " + std::to_string(h_counters[1]) + ")");
    metrics.rows_selected = total;
    if (has_aggs) {  // SELECT COUNT(*) [, COUNT(*)...] WHERE ...
      if (allreduce) {
        comm_allreduce_u64(d_total.p, 1, 0, stream);
        PQB_CUDA(cudaMemcpyAsync(&total, d_total.p, 8, cudaMemcpyDeviceToHost, stream));
        PQB_CUDA(cudaStreamSynchronize(stream));
      }
      OutBatch ob;
      ob.rows = 1;
      for (uint32_t a = 0; a < d.n_aggs; a++) {
        OutColumn oc;
        oc.name = "count(*)";
        oc.type = PQ_T_I64;
        oc.values.resize(8);
        std::memcpy(oc.values.data(), &total, 8);
        ob.cols.push_back(std::move(oc));
      }
      metrics.groups = 1;
      batches_.push_back(std::move(ob));
    } else if (want_rows) {
      // selected row ordinals, ascending
      for (size_t r0 = 0; r0 < n_ids || (r0 == 0 && n_ids == 0); r0 += batch_rows) {
        size_t nb = std::min<size_t>(batch_rows, n_ids - r0);
        OutBatch ob;
        ob.rows = int64_t(nb);
        OutColumn oc;
        oc.name = "__row_id";
        oc.type = PQ_T_I64;
        if (nb) { oc.ext = ids_block; oc.ext_off = r0 * 8; }
        ob.cols.push_back(std::move(oc));
        batches_.push_back(std::move(ob));
        if (n_ids == 0) break;
      }
    }
  }
  float ms = 0;
  cudaEventElapsedTime(&ms, t_all.a, t_all.b);
  metrics.device_ms = ms;
  if (!items.empty() && nrg) { cudaEventElapsedTime(&ms, t_scan.a, t_scan.b); metrics.scan_kernel_ms = ms; }
  metrics.kernel_launches = launches;
}

void Query::schema(ArrowSchema* out) const {
  if (!batches_.empty()) { export_batch(batches_[0], nullptr, out); return; }
  OutBatch none;
  export_batch(none, nullptr, out);
}

// JSON egress (json_egress.cuh): all batches of the result, formatted on the device.
void Query::json(uint32_t flags, const char** out, uint64_t* len) {
  Context& ctx = Context::get();
  cudaStream_t stream = cudaStreamPerThread;
  const bool lines = (flags & PQ_JSON_LINES) != 0;
  unsigned long long n = 0;
  for (const OutBatch& b : batches_) n += uint64_t(b.rows);
  json_block_.reset();
  auto finish_empty = [&]() {
    json_block_ = std::make_shared<PinnedBlock>();
    json_block_->p = ctx.pinned_acquire(16);
    json_block_->bytes = lines ? 0 : 2;
    if (!lines) { json_block_->p[0] = '['; json_block_->p[1] = ']'; }
    *out = reinterpret_cast<const char*>(json_block_->p);
    *len = json_block_->bytes;
  };
  if (n == 0 || batches_.empty() || batches_[0].cols.empty()) { finish_empty(); return; }
  const OutBatch* first = nullptr;
  for (const OutBatch& b : batches_) if (b.rows) { first = &b; break; }
  const size_t ncols = first->cols.size();
  if (ncols > size_t(kJsonMaxCols)) throw Error(PQ_ERR_UNSUPPORTED, "JSON egress: more than 64 result columns");
  JsonArgs ja{};
  ja.ncols = uint32_t(ncols);
  ja.n_rows = n;
  ja.lines = lines ? 1u : 0u;
  ja.batch_rows = batch_rows_;
  ja.words_per_batch = (batch_rows_ + 31) / 32;
  size_t nonempty = 0;
  for (const OutBatch& b : batches_) nonempty += b.rows ? 1 : 0;
  std::vector<uint8_t> keys;
  std::vector<DevBuf<uint8_t>> temps(ncols * 3);
  for (size_t c = 0; c < ncols; c++) {
    const OutColumn& oc = first->cols[c];
    JsonCol& jc = ja.cols[c];
    jc.type = oc.type == PQ_T_F64 ? JT_F64 : oc.type == PQ_T_BOOL ? JT_BOOL : oc.type == PQ_T_UTF8 ? JT_UTF8 : oc.type == PQ_T_TS_MS ? JT_TS_MS : JT_I64;
    // "name": with the name escaped like any string
    jc.key_off = uint32_t(keys.size());
    keys.push_back('"');
    { std::vector<char> e(oc.name.size() * 6 + 1);
      const uint32_t k = jf_escape(reinterpret_cast<const uint8_t*>(oc.name.data()), uint32_t(oc.name.size()), e.data());
      keys.insert(keys.end(), e.begin(), e.begin() + k); }
    keys.push_back('"'); keys.push_back(':');
    jc.key_len = uint32_t(keys.size()) - jc.key_off;
    bool any_nulls = false;
    for (const OutBatch& b : batches_) if (b.rows) any_nulls = any_nulls || b.cols[c].null_count != 0;
    if (oc.ext_all) {
      // device-assembled result: one regular layout over all batches (values and offsets contiguous, bit-packed buffers per batch)
      const uint8_t* base = oc.ext->dev ? oc.ext->dev : oc.ext->p;   // the kept device block, or the mapped page-locked copy
      jc.values = base + oc.ext_off;
      jc.validity = any_nulls ? reinterpret_cast<const uint32_t*>(base + oc.ext_validity_off) : nullptr;
      jc.offsets = oc.type == PQ_T_UTF8 ? reinterpret_cast<const int32_t*>(base + oc.ext_offsets_off) : nullptr;
    } else if (oc.ext) {
      if (oc.null_count || oc.type == PQ_T_UTF8 || oc.type == PQ_T_BOOL) throw Error(PQ_ERR_UNSUPPORTED, "JSON egress: result layout not supported");
      jc.values = oc.ext->p + oc.ext_off;   // 8-byte values of all batches, contiguous (row ids)
    } else {
      // a small host-built batch (a global aggregate over zero rows, COUNT(*) only): its buffers go up as they are
      if (nonempty != 1) throw Error(PQ_ERR_UNSUPPORTED, "JSON egress: result layout not supported");
      ja.batch_rows = 0x7fffffffu;
      ja.words_per_batch = 0;
      std::vector<uint8_t> v = oc.values;
      v.resize(std::max<size_t>((v.size() + 7) & ~size_t(7), 8), 0);   // 8-byte values / whole words of bit-packed booleans
      temps[3 * c].upload(v, stream);
      jc.values = temps[3 * c].p;
      if (oc.null_count) {
        std::vector<uint8_t> vv = oc.validity;
        vv.resize((vv.size() + 7) & ~size_t(7), 0);   // the kernel reads whole 32-bit words
        temps[3 * c + 1].upload(vv, stream);
        jc.validity = reinterpret_cast<const uint32_t*>(temps[3 * c + 1].p);
      }
      if (oc.type == PQ_T_UTF8) {
        std::vector<uint8_t> o(oc.offsets.size() * 4);
        std::memcpy(o.data(), oc.offsets.data(), o.size());
        temps[3 * c + 2].upload(o, stream);
        jc.offsets = reinterpret_cast<const int32_t*>(temps[3 * c + 2].p);
      }
    }
  }
  DevBuf<uint8_t> d_keys; d_keys.upload(keys, stream);
  ja.keys = d_keys.p;
  DevBuf<uint32_t> d_lens; d_lens.alloc(n, stream);
  DevBuf<long long> d_offs; d_offs.alloc(n + 1, stream);
  const uint32_t grid = uint32_t((n + 255) / 256);
  k_json_sizes<<<grid, 256, 0, stream>>>(ja, d_lens.p);
  k_json_scan<<<1, 1024, 0, stream>>>(d_lens.p, n, d_offs.p, lines ? 0 : 1);
  long long total = 0;
  PQB_CUDA(cudaMemcpyAsync(&total, d_offs.p + n, 8, cudaMemcpyDeviceToHost, stream));
  PQB_CUDA(cudaStreamSynchronize(stream));
  DevBuf<char> d_out; d_out.alloc(size_t(total) + 16, stream);
  k_json_write<<<grid, 256, 0, stream>>>(ja, d_offs.p, d_out.p);
  PQB_CUDA(cudaGetLastError());
  json_block_ = std::make_shared<PinnedBlock>();
  json_block_->p = ctx.pinned_acquire(size_t(total) + 16);
  json_block_->bytes = size_t(total);
  PQB_CUDA(cudaMemcpyAsync(json_block_->p, d_out.p, size_t(total), cudaMemcpyDeviceToHost, stream));
  PQB_CUDA(cudaStreamSynchronize(stream));
  if (!lines) { json_block_->p[0] = '['; json_block_->p[total - 1] = ']'; }   // the last row's ',' closes the array
  metrics.d2h_bytes += uint64_t(total);
  metrics.kernel_launches += 3;
  *out = reinterpret_cast<const char*>(json_block_->p);
  *len = uint64_t(total);
}

int Query::next(int partition, ArrowArray* out, ArrowSchema* schema) {
  (void)partition;
  if (next_batch_ >= batches_.size()) return PQ_END_OF_STREAM;
  export_batch(batches_[next_batch_++], out, schema);
  return PQ_OK;
}

}  // namespace pqb
