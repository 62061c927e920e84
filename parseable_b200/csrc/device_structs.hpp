// POD structures shared by the host planner and the sm_100a kernels.
// Vocabulary follows the reference's domain: row groups, column chunks, pages,
// dictionaries (SURVEY.md §8 row a10), not ML terms.
#pragma once
#include <cstdint>

namespace pqb {

constexpr int kMaxCols = 12;      // columns one query may reference
constexpr int kMaxLeaves = 16;    // leaf predicates
constexpr int kMaxPredOps = 40;   // postfix program length
constexpr int kMaxKeys = 4;       // GROUP BY columns
constexpr int kMaxAggs = 8;       // aggregates
constexpr int kSlabRows = 2048;   // rows decoded per CTA iteration
constexpr int kSlabWords = kSlabRows / 32;
constexpr int kMaxDirEntries = 64;  // run-directory entries per stream per slab
constexpr int kDirEntryMaxValues = 512;
constexpr int kMaxDeltaEntries = 80;  // DELTA_BINARY_PACKED miniblock directory entries per slab
constexpr int kDeltaWindowBytes = 8192 + 64;
constexpr int kPredStack = 8;
constexpr int kFastDirEntries = 16;   // slab index: run-directory entry budget per slab (a page's slabs share the page's budget)
constexpr int kRecBatch = 16;         // slab records a CTA keeps in shared memory at a time

// page value encodings as the kernels see them
enum DevEnc : uint8_t { DE_DICT = 0, DE_PLAIN = 1, DE_DELTA = 2, DE_RLE_BOOL = 3,
                        DE_DELTA_BYTES = 4, DE_DELTA_LEN_BYTES = 5 /* both only while a table opens: rewritten to DE_PLAIN */ };
// DE_DICT and DE_RLE_BOOL carry an RLE / bit-packed hybrid value stream (staged + walked)
#define PQB_ENC_HAS_STREAM(e) ((e) == ::pqb::DE_DICT || (e) == ::pqb::DE_RLE_BOOL)
// ... and DE_DELTA pages are staged too (their own walker: block / miniblock headers)
#define PQB_ENC_HAS_WINDOW(e) (PQB_ENC_HAS_STREAM(e) || (e) == ::pqb::DE_DELTA)
// physical value kinds
enum DevKind : uint8_t { DK_I64 = 0, DK_F64 = 1, DK_STR = 2, DK_BOOL = 3, DK_I32 = 4, DK_F32 = 5 };

struct DevPage {               // one data page
  uint64_t off;                // arena byte offset of the page payload (after its header)
  uint32_t len;                // payload bytes
  uint32_t num_rows;           // values incl. nulls == rows (flat schema)
  uint32_t first_row;          // within the row group
  uint32_t def_off, def_len;   // RLE def-level bytes inside the payload (def_len==0: no nulls possible)
  uint32_t val_off;            // values section inside the payload
  uint8_t enc;                 // DevEnc
  uint8_t bit_width;           // DE_DICT: index bit width
  uint16_t chunk_slot;         // table column of this page
  uint32_t chunk;              // index into chunks[]
  uint32_t slab0;              // first record of this page in the table's slab index
  uint32_t flags;              // host copy only: bit 0 = every slab of the page is in the slab index
};

// DELTA_BYTE_ARRAY / DELTA_LENGTH_BYTE_ARRAY pages are rewritten as PLAIN BYTE_ARRAY pages at table open (flat_store.cuh)
struct DbaJob {
  uint32_t page;
  uint32_t with_prefix;   // 1 DELTA_BYTE_ARRAY, 0 DELTA_LENGTH_BYTE_ARRAY (no prefix stream)
  uint64_t len_tmp;       // scratch: prefix lengths [rows] then suffix lengths [rows] (u32), byte offset in the scratch buffer
  uint64_t dst;           // k_dba_materialise: byte offset of the new page payload in the materialised buffer
};
struct DbaInfo { uint64_t bytes; uint32_t nvals; uint32_t data_pos; uint32_t ok; uint32_t _pad; };

struct DevChunk {              // one column chunk (row group x referenced column)
  uint64_t dict_off;           // arena offset of the PLAIN dictionary payload
  uint32_t dict_len;
  uint32_t dict_n;             // dictionary entries (0: no dictionary page)
  uint32_t first_page;         // into pages[]
  uint32_t n_pages;
  uint32_t lut_base;           // base into the COLUMN's per-entry side tables (str offsets / leaf LUTs / gid LUTs):
                               // entries of this column in the row groups before this one (table level, query independent)
  uint32_t present;            // 0: column missing from this file -> all NULL
  uint64_t dict8_off;          // flat-store offset of the 8-byte aligned copy of a numeric dictionary (~0: none)
};

// Flat store (flat_store.cuh): the scan-ready copy of one data page.
enum FlatKind : uint8_t { FK_NONE = 0, FK_INDEX = 1, FK_PLAIN8 = 2, FK_BITS = 3, FK_BYTES = 4,
                          FK_IDS = 5 };   // FK_IDS (per query): u32 group id per row of a GROUP BY column's page without a dictionary
struct FlatPageRec {           // parallel to pages[]
  uint64_t off;                // byte offset in the flat buffer, 16-byte aligned: one slot per ROW (NULL rows hold 0)
  uint64_t voff;               // validity bitmap (1 bit per row, LSB first like Arrow), or ~0: the page holds no NULLs
  uint32_t rows;
  uint8_t bw;                  // FK_INDEX: bits per dictionary index; FK_BITS: 1
  uint8_t fkind;               // FlatKind: FK_INDEX dictionary indices, FK_PLAIN8 8-byte values, FK_BITS boolean values,
                               // FK_BYTES PLAIN byte arrays: one u32 per row = where the row's bytes start, relative to `base`
  uint16_t _pad;
  uint64_t base;               // FK_BYTES: arena offset of the page's values section (a value's 4-byte length sits right before its bytes)
};

struct DevItem {               // unit of CTA work: rows between two page boundaries common to all columns
  uint32_t rg;                 // dense row-group slot
  uint32_t row0;               // first row inside the row group
  uint32_t nrows;
  uint32_t bitmap_word0;       // first word of this item's region in the selection bitmap
  uint64_t global_row0;        // ordinal of row0 in the scanned table (row-id output)
  uint32_t page[kMaxCols];     // page index (into pages[]) holding row0, per column slot
  uint32_t poff[kMaxCols];     // flat items: row0 minus the page's first row (a piece may start inside a page)
  uint32_t fast;               // bit 0: every referenced column has exactly one, slab-indexed page over this item (k_scan);
                               // bit 1: ... exactly one page with a flat-store copy (k_flat_*)
  uint32_t absent;             // flat items: bit s = column slot s is missing from this file (reads as all NULL)
};
constexpr uint32_t kItemSlabIndexed = 1u, kItemFlat = 2u;

// One slab (kSlabRows rows from the page start) of one page in the table's slab index
// (k_slab_index, built when the table is opened): what the per-slab control of k_scan would derive
// by walking the run headers, computed for every page at once.
struct DevSlabRec {
  uint64_t win_off;            // arena offset the value window is staged from (16-byte aligned)
  uint64_t val_base;           // arena offset of the page's values section
  uint32_t vals_done;          // values of the page consumed before this slab
  uint16_t nent;               // run-directory entries (two sentinels follow)
  uint8_t enc;                 // DevEnc
  uint8_t bw;                  // index bit width
  uint32_t ent0;               // first run-directory entry of this slab in the index (entries are 16 bytes)
  uint32_t _pad;
};

struct DevColumn {
  uint8_t kind;                // DevKind
  uint8_t max_def;             // 0: REQUIRED
  uint8_t need_idx;            // stage dictionary indices in the row phase
  uint8_t staged;              // flat kernels: 1 = predicate / key / aggregate input (TMA-staged per slab); 0 = only projected
  uint32_t max_bw;             // widest dictionary index over all pages read
  uint32_t has_delta, has_plain, has_dict;
};

enum DevLeafKind : uint8_t { LK_CMP = 1, LK_IS_NULL = 2, LK_IS_NOT_NULL = 3, LK_LIKE = 4 };

struct DevLeaf {
  uint8_t kind;                // DevLeafKind
  uint8_t cmp;                 // PqCmp
  uint8_t col;                 // column slot
  uint8_t lit_kind;            // DevKind of the literal after coercion
  uint32_t flags;              // like flags
  int64_t lit_i64;             // I64/TS/BOOL literal or f64 bits
  uint32_t str_off, str_len;   // UTF8 literal / LIKE pattern in the literal pool
  uint32_t lut_off;            // this leaf's per-dictionary-entry LUT (bytes) starts at lut_off; entry = chunk.lut_base+idx
  uint32_t _pad;
};

enum DevPredKind : uint8_t { PK_LEAF = 1, PK_AND = 2, PK_OR = 3, PK_NOT = 4, PK_CONST = 5 };
struct DevPredOp { uint8_t kind; uint8_t arg; /* leaf id, or const: 0 F, 1 T, 2 NULL */ };

enum DevAggFn : uint8_t { AG_COUNT_STAR = 0, AG_COUNT = 1, AG_SUM = 2, AG_MIN = 3, AG_MAX = 4, AG_AVG = 5 };
struct DevAgg {
  uint8_t fn;
  uint8_t col;       // column slot
  uint8_t kind;      // DevKind of the input (I64 / F64 / BOOL)
  uint8_t acc_slot;  // which 8-byte accumulator array
  uint8_t nn_slot;   // which non-null counter array (one per aggregated column)
  uint8_t update_nn; // 1: this aggregate bumps nn[nn_slot] (first aggregate over its column)
  uint8_t _pad[2];
};

enum DevKeyKind : uint8_t { KK_DICT_LUT = 0, KK_BOOL = 1, KK_BIN = 2 };   // KK_BIN: DATE_BIN of an Int64 / Timestamp column
struct DevKey {
  uint8_t col;
  uint8_t kind;       // DevKeyKind
  uint16_t _pad;
  uint32_t card;      // global distinct values; NULL takes id == card
  uint32_t stride;    // mixed-radix stride of this key in the dense group slot
  uint32_t _pad2;
  const uint32_t* gid;  // gid LUT of the key column (u32 per dictionary entry, entry = chunk.lut_base + idx)
  int64_t bin_base;     // KK_BIN: start of bin 0 (the lowest bin any scanned row group can hold, from footer statistics)
  int64_t bin_width;    // KK_BIN: stride; group id = floor((value - bin_base) / bin_width)
  uint64_t wstride;     // the same stride in 64 bits (hashed group-by: the mixed radix may be wider than the dense table)
};

enum ScanMode : uint32_t { SM_FILTER = 0, SM_AGG = 1 };

struct DevPlan {
  uint32_t mode;               // ScanMode
  uint32_t ncols;
  uint32_t nleaves;
  uint32_t npred;
  uint32_t nkeys;
  uint32_t naggs;
  uint32_t n_acc;              // 8-byte accumulator arrays
  uint32_t n_nn;               // non-null counter arrays
  uint32_t nslots;             // dense group slots
  uint32_t smem_acc;           // 1: accumulate in shared memory, flush per CTA
  uint32_t write_bitmap;       // filter mode: store the selection bitmap
  uint32_t n_items;
  DevColumn cols[kMaxCols];
  DevLeaf leaves[kMaxLeaves];
  DevPredOp pred[kMaxPredOps];
  DevKey keys[kMaxKeys];
  DevAgg aggs[kMaxAggs];
  // per accumulator array, how cells start and merge: 0 integer add (0), 1 f64 add (0.0),
  // 2 signed min (INT64_MAX), 3 signed max (INT64_MIN); f64 MIN/MAX run on order keys
  uint8_t acc_init[kMaxAggs * 2];
  // leaves a dictionary LUT answers, per column (host precomputed): how many, and the first two
  uint8_t col_nlut[kMaxCols];
  int8_t col_l0[kMaxCols];
  int8_t col_l1[kMaxCols];
  uint32_t row_major;          // 1: no-NULL slabs use the register-only row-major pass
  uint32_t fast_and;           // 1: the predicate is leaf AND leaf AND ... (1-4 CMP/LIKE leaves): specialised pass
  uint32_t conj;               // 1: the predicate is a pure conjunction of leaves (flat kernels: survivors-only evaluation)
  uint32_t hot_slots;          // flat aggregate kernel: group slots < hot_slots accumulate in shared memory
  uint32_t lane_slots;         // flat aggregate kernel: the first lane_slots (hottest) group slots own one shared-memory cell per lane
  uint32_t flat_krows;         // flat aggregate kernel: rows per consumer thread per slab
  uint32_t direct8;            // flat aggregate kernel: 8-byte values are read in place from the flat store, not staged
  uint32_t dbg;                // measurement switches: bit 0 / 1 = k_flat_filter / k_flat_agg consumers hand every stage back untouched (PQB_FILTER_NOWORK, PQB_AGG_NOWORK: the supply-side limit)
  uint32_t flat_slab_rows;     // rows per slab of the flat kernels
  uint32_t no_flat;            // 1: the flat kernels do not run (NULL literal in the predicate, PQB_FLAT_SCAN=0): k_scan takes every item
  uint32_t replicas;           // accumulator table copies in global memory; CTA b adds into copy b % replicas (merged by k_acc_reduce)
  uint32_t smem_share;         // of every 8 consumer warps of k_flat_agg, how many keep hot slots in shared memory (the rest use L2)
  uint32_t f64_global;         // 1: f64 SUM / AVG cells always go to L2 (no native shared-memory f64 atomic)
  uint32_t f64_smem;           // 1: f64 SUM / AVG of every hot slot in shared memory (CAS loop); 0: only the per-lane cells, the
                               // other hot slots send them to L2 (native reduction)
  uint32_t hashed;             // 1: the key space is wider than the dense table: group cells are found through DevScanArgs.hkeys
  uint32_t hmask;              // hashed: table capacity - 1 (nslots == capacity)
  // flat aggregate kernel, shared-memory hot table: planes rows, acc[0 .. n_acc), nn[0 .. n_nn) as in the global table, but
  // not all 8 bytes wide.  The rows and nn planes and the narrow MIN / MAX planes hold 4-byte cells; hot_off is each plane's
  // byte offset inside the hot table (8-byte planes first, so every cell is aligned to its width)
  uint32_t hot_off[1 + 2 * kMaxAggs];
  uint32_t hot_cell_bytes;     // bytes of one hot cell over all planes
  uint32_t acc_narrow;         // bit a: acc[a] is an Int64 MIN / MAX whose hot cells hold u32 offsets from acc_base[a]
                               // (MIN: v - base, empty 0xffffffff; MAX: v - base + 1, empty 0).  A value outside
                               // [base, base + 2^32 - 2] updates the global 8-byte cell instead
  int64_t acc_base[kMaxAggs];
};

// Accumulator table layout (device, 8-byte cells, struct of arrays over nslots):
//   rows[nslots]                       selected rows per group  (COUNT(*))
//   acc[a][nslots]  a < n_acc          SUM / MIN / MAX cells (i64, f64 bits, or order-preserving f64 keys)
//   nn[k][nslots]   k < n_nn           non-null inputs per aggregated column

struct DevScanArgs {
  const uint8_t* arena;        // encoded column chunks, HBM resident
  const DevPage* pages;
  const DevChunk* chunks;      // [rg_slot * ncols + col]
  const DevItem* items;
  const uint8_t* luts;         // leaf LUT bytes (0 false, 1 true) per dictionary entry
  const uint8_t* lit_pool;
  const uint8_t* rg_live;      // per row group: 0 = pruned by statistics for this query (nullptr: all live)
  const uint8_t* flat;         // flat store (flat_store.cuh)
  const FlatPageRec* fpages;   // parallel to pages[]
  uint32_t* bitmap;            // selection bitmap, per-item word regions
  uint32_t* item_counts;       // selected rows per item
  unsigned long long* acc;     // accumulator table (global)
  unsigned long long* hkeys;   // hashed group-by: wide group id per accumulator slot (~0: empty)
  unsigned long long* counters;  // [0] rows selected, [1] error flag, [2] work-queue head
  // the table's slab index (fast items)
  const DevSlabRec* slab_recs;       // [page.slab0 + k]
  const struct DirEntry* slab_dirs;  // [rec.ent0 + e]
};

// one page the second pass of the slab index re-packs flat (k_flatten_pages)
struct FlatJob { uint32_t page; uint32_t _pad; uint64_t side_off; };

// run-directory entry produced by the stream walker
struct DirEntry {     // 16 bytes: bulk-copyable (TMA) from the prebuilt slab directory
  uint32_t start;    // first value (slab relative)
  uint16_t count;
  uint8_t kind;      // 0 RLE, 1 bit-packed
  uint8_t chunk0;    // running count of 32-value chunks before this entry (balances warps)
  uint32_t payload;  // RLE: value; bit-packed: bit offset of the first value inside the window
  uint32_t _pad;
};
constexpr int kDirWords = 4;  // DirEntry as 32-bit words: {start, count | kind << 16 | chunk0 << 24, payload, -}

}  // namespace pqb
