// scan_kernels.cuh -- device-side types shared between the kernels (scan_kernels.cu) and the host
// orchestration (capi.cu).  See DESIGN.md for the HBM layout and the roofline of each kernel.
#pragma once

#include <cuda_runtime.h>

#include <cstdint>

#include "part_dir.hpp"

namespace bydb {

constexpr int kWarpsPerCta = 8;          // 256 threads; every warp is an independent block worker
#ifndef BYDB_STAGE_BYTES
#define BYDB_STAGE_BYTES 2048            // experiment knobs (make variant EXTRA="-DBYDB_STAGE_BYTES=4096 -DBYDB_STAGES=3")
#endif
#ifndef BYDB_STAGES
#define BYDB_STAGES 2
#endif
#ifndef BYDB_SPARSE
#define BYDB_SPARSE 0                    // 1: masked / ranged delta pages take delta_page_sparse (measured slower, see DESIGN.md 4.2; make variant EXTRA="-DBYDB_SPARSE=1 -DBYDB_STAGES=3")
#endif
#ifndef BYDB_MASKED_SWAR
#define BYDB_MASKED_SWAR 1               // 0: masked / ranged SUM pages keep the serial decoder (A/B timing)
#endif
#ifndef BYDB_FAST_CTAS
#define BYDB_FAST_CTAS 3                 // resident CTAs per SM the fast lane is compiled for (register cap 65536 / (256 x n))
#endif
constexpr int kStageBytes = BYDB_STAGE_BYTES;  // one TMA bulk copy (cp.async.bulk) per stage
constexpr int kStages = BYDB_STAGES;           // per-warp ring: decode stage k while stage k+1 lands
constexpr int kChunkBytes = 512;         // 32 lanes x 16 B per decode iteration
constexpr int kMaskWords = 264;          // row bitmask: 8448 rows (memPart blocks hold <= 8193 rows)
constexpr int kMaxFcols = 8;             // distinct aggregated fields per query
constexpr int kMaxPreds = 8;             // conjunctive row predicates per query
constexpr int kMaxLit = 64;              // inline literal bytes of a string predicate
constexpr int kMaxParts = 64;            // parts per query

// device error codes written to ScanParams::err[0] (first error wins); err[1] = global block index
enum DevErr : uint32_t {
    kErrNone = 0,
    kErrPlainPage = 1,      // numeric fallback page (EncodeTypePlain, column.go:147-153): needs zstd on device
    kErrZstdDict = 2,       // dictionary whose value block is zstd-compressed (>=128 B, bytes.go:291-304)
    kErrBigBlock = 3,       // predicate on a block with more rows than the smem row mask holds
    kErrCorrupt = 4,        // varint stream does not decode to `count` values / bad header
    kErrTypeMix = 5,        // one field name with int64 and float64 pages in the same query
    kErrBadEnc = 6,         // unknown encode type byte
    kErrTagPlain = 7,       // high-cardinality (>256 values) string tag page: plain bytes block
    kErrOverlap = 8,        // same series in several parts with overlapping time spans: needs version dedup
    kErrPredType = 9,       // predicate literal type does not match the stored tag column type
    kErrTmaTimeout = 10,    // a bulk copy never completed (internal error)
    kErrPeerTimeout = 11,   // multi-GPU reduce: a peer rank never delivered its partial table / never freed the slot
    kErrKeyCap = 12,        // per-row group key: more distinct values than the caller's max_values
    kErrKeyLong = 13,       // per-row group key: a value longer than kMaxLit bytes
};
constexpr int kOpEqOrNil = 7;  // internal predicate operator of the group-key passes: the cell is nil or equals the literal

struct DevPartRef {
    const DevBlock *blocks;
    const DevCol *cols;
    const uint8_t *const *files;  // device array of file base pointers (indexed by DevCol::file_id)
    uint32_t n_blocks;
    uint32_t block_base;          // global index of blocks[0] in this query
};

struct DevPred {
    int64_t lit_i64;
    uint32_t lit_len;
    uint16_t name_id;
    uint8_t op;
    uint8_t value_type;
    uint8_t lit[kMaxLit];
};

// per (block, field) partial aggregate; `i` views are used for int64 fields, `f` for float64 fields
struct BlockPartial {
    union { double f; int64_t i; } sum, mn, mx;
    int64_t cnt;
};
static_assert(sizeof(BlockPartial) == 32, "BlockPartial layout");

struct ScanParams {
    DevPartRef parts[kMaxParts];
    uint32_t n_parts;
    uint32_t total_blocks;
    const uint64_t *q_sids;       // ascending
    uint32_t n_series;
    uint32_t n_fcols;
    uint32_t n_preds;
    uint32_t pad0;
    int64_t tmin, tmax;
    uint16_t fcol_name[kMaxFcols];
    uint8_t fcol_need[kMaxFcols]; // bit0: sum wanted (SUM/MEAN), bit1: min/max wanted; 0 = COUNT only
    DevPred preds[kMaxPreds];
    uint32_t *worklist;           // [total_blocks] global block indices selected by plan_blocks
    uint32_t *work_count;
    uint32_t *work_next;
    uint32_t *rest_list;          // [total_blocks] express lane only (else NULL): blocks it left to the regular fast lane
    uint32_t *rest_count;
    uint32_t *rest_next;
    uint32_t *slow_list;          // [total_blocks] blocks the fast lane deferred to the general decoder
    uint32_t *slow_count;
    uint32_t *slow_next;
    int32_t *block_qsid;          // [total_blocks] query-series index or -1
    uint32_t *first_block;        // [n_parts * n_series] first block of the series in the part (0xffffffff = none); may be NULL
    BlockPartial *P;              // [total_blocks * n_fcols]
    uint32_t *Prows;              // [total_blocks] rows that passed range + predicates
    uint32_t *Pfirst;             // [total_blocks] first surviving row of the block (group-key passes only, else NULL)
    int32_t *col_type;            // [n_fcols] 0 unknown / BYDB_VT_INT64 / BYDB_VT_FLOAT64
    uint32_t *err;                // [2]
    unsigned long long *stats;    // [0] rows_scanned [1] rows_matched [2] page_bytes [3] blocks
    // ---- version dedup across overlapping parts (query.go:995-1004); all NULL when no parts overlap
    int32_t *dd_index;            // [total_blocks] compact index of a block that needs dedup, or -1
    unsigned long long *dd_row_off; // [total_blocks] offset of the block's rows in dd_ts / dd_ver
    uint32_t *dd_list;            // [n_dd_blocks] global block indices
    unsigned long long *dd_counts; // [0] flagged blocks, [1] flagged rows
    int64_t *dd_ts, *dd_ver;      // decoded timestamps / versions of the flagged blocks
    uint32_t *dd_shadow;          // [n_dd_blocks * kMaskWords] 1 = row survives the dedup
    uint32_t n_dd_blocks;
    uint32_t pad1;
};

struct ReduceParams {
    DevPartRef parts[kMaxParts];
    uint32_t n_parts;
    uint32_t n_series;
    uint32_t n_fcols;
    int32_t n_groups;
    const uint64_t *q_sids;
    const int32_t *order;         // [n_series] query-series indices sorted by (group, series)
    const int32_t *group_start;   // [n_groups + 1] into order
    const int32_t *block_qsid;
    const uint32_t *first_block;  // see ScanParams
    const BlockPartial *P;
    const uint32_t *Prows;
    const int32_t *col_type;
    BlockPartial *S;              // [n_series * n_fcols] per-series partials
    int64_t *Srows;               // [n_series]
    uint32_t *err;
    uint32_t dedup_done;          // 1 = overlapping parts were resolved by the dedup kernels
    uint32_t pad2;
    // group-key passes only (else NULL): where the series first shows the pass's key value -- (ts_min of the earliest block
    // with a surviving row, that row's index); INT64_MAX = the series never shows it
    const uint32_t *Pfirst;
    int64_t *Kts;                 // [n_series]
    uint32_t *Krow;               // [n_series]
    // partial table (see bydb_gpu.h): written by group_reduce
    double *sum_f64, *max_f64, *negmin_f64;
    int64_t *sum_i64, *cnt, *rows, *max_i64, *notmin_i64, *coltype;
};

struct FinalizeParams {
    int32_t n_groups;
    uint32_t n_fcols;
    uint32_t n_aggs;
    uint32_t row_path_types;      // 1 = COUNT is typed like its field (the row path's N-typed countFunc) instead of int64
    int32_t agg_fcol[32];
    int32_t agg_func[32];
    const double *sum_f64, *max_f64, *negmin_f64;
    const int64_t *sum_i64, *cnt, *rows, *max_i64, *notmin_i64, *coltype;
    int64_t *out_i64;             // [n_groups * n_aggs]
    double *out_f64;              // [n_groups * n_aggs]
    uint8_t *out_is_float;        // [n_aggs]
    uint32_t *err_out;            // DevErr carried in the table's coltype words (0 = none); may be NULL
};

// output row selection on the device: stable compaction of the groups that appeared, or Top-N
constexpr int kMaxDeviceTopN = 2048;
struct SelectParams {
    int32_t n_groups;
    uint32_t n_fcols, n_aggs;
    int32_t top_n, top_agg, top_desc, top_fcol, top_is_count;
    const int64_t *rows, *cnt;
    const int64_t *val_i64;       // finalized values [n_groups * n_aggs]
    const double *val_f64;
    const uint8_t *is_float;      // [n_aggs]
    uint64_t *keys;               // scratch [n_groups]
    uint8_t *kstate;              // scratch [n_groups]
    int32_t *sel_group;           // outputs, capacity = top_n > 0 ? min(top_n, n_groups) : n_groups
    int64_t *sel_rows;
    int64_t *sel_i64;
    double *sel_f64;
    uint32_t *sel_count;
};
void launch_select_rows(const SelectParams &p, cudaStream_t s);

// ---- per-row group key (a stored dictionary tag): see "Group key" in scan_kernels.cu
constexpr uint32_t kKeySlots = 1024;   // open-addressing table of the distinct key values (at most 256 are accepted)
constexpr uint32_t kMaxKeyValues = 256;
struct KeyParams {
    DevPartRef parts[kMaxParts];
    uint32_t n_parts, total_blocks;
    const uint64_t *q_sids;
    uint32_t n_series;
    uint32_t cap;                 // distinct values the caller accepts
    int64_t tmin, tmax;
    uint16_t key_name;
    uint16_t pad[3];
    unsigned long long *slots;    // [kKeySlots] 0 = empty, else bit63 | len << 48 | device address of the bytes
    uint32_t *count;              // distinct values found
    uint32_t *err;                // [2]
    uint8_t *vals;                // [cap * kMaxLit] packed by key_pack
    uint32_t *lens;               // [cap]
};
void launch_key_values(const KeyParams &p, int grid, cudaStream_t s);
struct KeyOrderParams {
    int32_t n_groups;             // G: groups of series
    uint32_t n_values;            // V
    uint32_t n_series;
    uint32_t pad;
    const int32_t *order, *group_start;
    const int64_t *Kts;           // [V * n_series]
    const uint32_t *Krow;         // [V * n_series]
    int32_t *slot;                // [n_series * V] preset to -1: composite group whose first row is (series, rank)
    int32_t *first_series;        // [V * G] -1 = the composite group never appeared
    int32_t *perm;                // [V * G] composite groups in insertion order, then the ones that never appeared
    uint32_t *n_present;
};
void launch_key_order(const KeyOrderParams &p, cudaStream_t s);
struct TablePtrs {
    double *sum_f64, *max_f64, *negmin_f64;
    int64_t *sum_i64, *cnt, *rows, *max_i64, *notmin_i64, *coltype;
};
// dst[j] = src[perm[j]] for every group row of a partial table; coltype = the passes' column types merged
void launch_permute_table(const TablePtrs &dst, const TablePtrs &src, const int32_t *perm, uint32_t n_groups, uint32_t n_fcols,
                          const int64_t *pass_coltype, uint32_t n_passes, cudaStream_t s);

// ---- keyed collective (bydb_scan_reduce_keyed): see "Keyed collective" in scan_kernels.cu
// every rank: where each composite group (v, g) first shows, as (series id, Kts, Krow); absent = (UINT64_MAX, INT64_MAX, UINT32_MAX)
struct KeyFirstParams {
    int32_t n_groups;
    uint32_t n_values;
    const uint64_t *q_sids;       // [n_series] ascending
    const int32_t *order, *group_start;
    const int64_t *Kts;           // [V * n_series]
    const uint32_t *Krow;
    uint32_t n_series;
    uint32_t pad;
    uint32_t *n_values_out;       // receives n_values (the rank's slot header)
    uint64_t *first_sid;          // [V * G]
    int64_t *first_ts;
    uint32_t *first_row;
};
void launch_key_first(const KeyFirstParams &p, cudaStream_t s);
// the root: the ranks' key dictionaries -> one global dictionary (ids in order of first occurrence over (rank, local id))
struct KeyUnionParams {
    uint32_t n_ranks, cap;        // every slot holds up to cap values
    const uint8_t *slots;         // rank r's slot at slots + r * slot_bytes
    uint64_t slot_bytes;
    uint64_t off_nv, off_lens, off_vals;  // inside a slot: u32 V_r, u32 lens[cap], bytes[cap * kMaxLit]
    uint32_t *hash;               // [hash_slots] zeroed: entry index + 1 of the first (rank, value) with those bytes
    uint32_t hash_slots;          // power of two >= 2 * n_ranks * cap
    int32_t *rep;                 // [n_ranks * cap] scratch
    int32_t *remap;               // [n_ranks * cap] preset to -1: global id of (r, v)
    int32_t *inv;                 // [n_ranks * cap] preset to -1: local id on rank r of global value g (index r * cap + g)
    uint32_t *ctl;                // [0] distinct values over all ranks  [1] kErrKeyCap when that exceeds cap
    uint32_t *g_lens;             // [cap] the global dictionary
    uint8_t *g_vals;              // [cap * kMaxLit]
};
void launch_key_union(const KeyUnionParams &p, cudaStream_t s);
// the root: the ranks' composite tables folded into one Vg x G table (rank order), first appearances merged
struct KeyCombineParams {
    uint32_t n_ranks, cap, n_values, n_fcols;  // n_values = Vg
    int32_t n_groups;
    uint32_t pad;
    uint64_t slot_bytes;          // stride between the ranks' slots
    TablePtrs src;                // composite table in rank 0's slot (cap * n_groups groups); rank r's is src + r * slot_bytes
    const int64_t *src_ct;        // [cap * n_fcols] pass column types in rank 0's slot
    const uint64_t *src_fsid;     // [cap * n_groups] first appearances in rank 0's slot
    const int64_t *src_fts;
    const uint32_t *src_frow;
    const int32_t *inv;           // KeyUnionParams::inv
    TablePtrs dst;                // Vg * n_groups groups
    int64_t *dst_ct;              // [Vg * n_fcols] column types of the global values, merged over the ranks
    uint64_t *fsid;               // [Vg * n_groups]
    int64_t *fts;
    uint32_t *frow;
};
void launch_key_combine(const KeyCombineParams &p, cudaStream_t s);
// perm = 0..n-1 sorted by first appearance (sid, ts, row), absent groups last; temp == NULL: *temp_bytes receives the size
int launch_key_rank(const uint64_t *fsid, const int64_t *fts, const uint32_t *frow, int32_t *perm, uint32_t n, void *temp, size_t *temp_bytes,
                    cudaStream_t s);
constexpr int kFusedFinalizeGroups = 8192;  // up to here one CTA finalises and selects in a single launch
struct FinalizeParams;
uint32_t launch_finalize_select(const FinalizeParams &fp, const SelectParams &p, cudaStream_t s);  // -> kernels launched
// combines n partial tables (each `words` 8-byte words, laid out back to back) into the first one, rank order
void launch_combine_tables(uint64_t *tables, uint32_t n_tables, uint64_t words, uint64_t sum_f64_lo, uint64_t sum_f64_hi, uint64_t max_f64_lo,
                           uint64_t max_f64_hi, uint64_t sum_i64_lo, uint64_t sum_i64_hi, uint64_t max_i64_lo, uint64_t max_i64_hi, cudaStream_t s,
                           uint64_t stride_words = 0);
// peer-mailbox reduce (bydb_comm_*): bounded wait for n epoch flags, release-store of one
void launch_comm_wait(const unsigned long long *flags, uint32_t n, unsigned long long epoch, uint32_t *err, uint32_t err_code, cudaStream_t s);
void launch_comm_signal(unsigned long long *flag, unsigned long long epoch, cudaStream_t s);
// graph-replayable forms: the epoch comes from a device block refreshed by a memcpy node of the graph
struct CommArgs {
    unsigned long long epoch, prev_use;
};
void launch_comm_wait_args(const unsigned long long *flags, uint32_t n, const CommArgs *a, int which, uint32_t *err, uint32_t err_code, cudaStream_t s);
void launch_comm_signal_args(unsigned long long *flag, unsigned long long *status, const CommArgs *a, cudaStream_t s);
void launch_comm_done_args(unsigned long long *done, const CommArgs *a, cudaStream_t s);

// ---- fallback-page normalisation at part admission (unpack_kernels.cu)
constexpr uint8_t kEncRawCells = 0x40;   // numeric page rewritten as [0x40][has_nulls][6 pad][n x u64 LE][n x u8 valid]
constexpr uint8_t kBlockRawLong = 2;     // compressBlock rewritten as [2][u32 LE len][bytes] (an inflated zstd frame)
constexpr uint32_t kUnpackNumeric = 1, kUnpackString = 2;
struct UnpackJob {
    uint64_t out_off;   // into the unpack arena
    uint32_t col;       // index into the part's DevCol table
    uint32_t rows;
    uint32_t out_cap;
    uint32_t kind;
};
struct UnpackParams {
    const DevBlock *blocks;
    DevCol *cols;                   // rewritten in place for the pages that were unpacked
    const uint8_t *const *files;
    uint32_t n_blocks;
    uint32_t arena_file_id;         // slot of the unpack arena in the part's file table
    UnpackJob *jobs;
    unsigned long long max_jobs, n_jobs;
    unsigned long long *counters;   // [0] jobs found [1] arena bytes [2] cursor [3] pages left as they are [4] pages unpacked
    uint8_t *arena;
    uint8_t *scratch;               // n_warps * unpack_scratch_stride()
};
size_t unpack_scratch_stride();
void launch_classify_pages(const UnpackParams &p, cudaStream_t s);
void launch_unpack_pages(const UnpackParams &p, int n_warps, cudaStream_t s);

// ---- write side: numeric field pages encoded on the device (encode_kernels.cu)
struct EncodeParams {
    const void *values;           // int64 / double, the blocks back to back
    const uint64_t *block_off;    // [n_blocks + 1] value offsets
    uint32_t n_blocks;
    uint32_t is_float;
    int64_t *scratch;             // [n_values] decimal integers of a float64 column
    int16_t *exps;                // [n_values]
    uint8_t *slots;               // worst-case page slots
    const uint64_t *slot_off;     // [n_blocks + 1]
    uint32_t *page_len;           // [n_blocks] 0 = the block goes to the CPU writer
    uint8_t *status;              // [n_blocks] 1 = not encoded here
};
void launch_encode_pages(const EncodeParams &p, int grid, cudaStream_t s);
void launch_gather_pages(const EncodeParams &p, const uint64_t *out_off, uint8_t *out, int grid, cudaStream_t s);
void preload_encode_kernels();   // encode_kernels.cu

size_t scan_smem_bytes();
void launch_plan_blocks(const ScanParams &p, cudaStream_t s);
void launch_scan_blocks(const ScanParams &p, int grid_fast, int grid_slow, cudaStream_t s);
void launch_series_reduce(const ReduceParams &p, cudaStream_t s);
void launch_group_reduce(const ReduceParams &p, cudaStream_t s, bool small_groups = false);  // small_groups: no group has more than 32 series
void launch_finalize(const FinalizeParams &p, cudaStream_t s);
void launch_detect_overlap(const ScanParams &p, cudaStream_t s);
void launch_dedup(const ScanParams &p, int grid, cudaStream_t s);
int upload_pow10_table();
void scan_max_ctas_per_sm(int *fast, int *slow);
void preload_kernels();          // scan_kernels.cu: forces the (lazily loaded) code of every kernel onto the current device
void preload_unpack_kernels();   // unpack_kernels.cu
void preload_index_kernels();    // index_kernels.cu

}  // namespace bydb
