/*
 * bydb_gpu.h -- C ABI of libbydbgpu.so: the B200-native measure scan -> filter -> aggregate path.
 *
 * This is the drop-in boundary a cgo binding in BanyanDB would bind (see INTEGRATION.md).  It
 * replaces, for one query, the reference's HOT LOOPS 1-3 (SURVEY.md section 3.1):
 *
 *   bydb_part_register  <- banyand/measure/part.go:312-375 (mustOpenFilePart) +
 *                          part_iter.go:184-208 (readPrimaryBlock -> blockMetadata cache)
 *   bydb_part_release   <- banyand/measure/part.go:282-299 (partWrapper.decRef -> close)
 *   bydb_scan_agg       <- banyand/measure/query.go:594-639 (searchBlocks) +
 *                          query_batch.go:64-238 (PullBatch / loadCursorsForBatch / mergeBatch) +
 *                          block.go:793-870 (blockCursor.loadData) +
 *                          pkg/query/vectorized/measure/aggregation.go:193-334 (BatchAggregation) +
 *                          pkg/query/vectorized/measure/top.go:145-214 (BatchTop)
 *   bydb_scan_partials / bydb_reduce_finalize
 *                       <- pkg/query/logical/measure/measure_plan_aggregation.go:67-124
 *                          (emitPartial map phase / reduceAccumulator.Combine)
 *
 * Rules: C linkage, plain pointers and sizes; no pointer passed in is retained after the call
 * returns (cgo rule); every function is thread-safe; functions return 0 or a negative errno-style
 * code and never abort; bydb_last_error() returns a thread-local message.  There is NO CPU fallback
 * behind this ABI: pages the device path cannot decode make the call fail with BYDB_ENOTSUP so the
 * caller can route the query to its own CPU path outside this library.
 */
#ifndef BYDB_GPU_H
#define BYDB_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BYDB_OK 0
#define BYDB_ENOENT (-2)    /* unknown part handle / missing file            */
#define BYDB_EIO (-5)       /* CUDA runtime failure                          */
#define BYDB_ENOMEM (-12)   /* HBM budget exceeded / allocation failure      */
#define BYDB_EINVAL (-22)   /* malformed argument or corrupt part            */
#define BYDB_ENOTSUP (-95)  /* encoding not handled on the device path       */

/* value types, pkg/pb/v1/value.go:39-47 */
#define BYDB_VT_STR 1
#define BYDB_VT_INT64 2
#define BYDB_VT_FLOAT64 3
#define BYDB_VT_BINARY 4

/* aggregation functions, api/proto/banyandb/model/v1/common.proto:75-80 */
#define BYDB_AGG_MEAN 1
#define BYDB_AGG_MAX 2
#define BYDB_AGG_MIN 3
#define BYDB_AGG_COUNT 4
#define BYDB_AGG_SUM 5

/* row-predicate operators on a stored tag column */
#define BYDB_OP_EQ 1
#define BYDB_OP_NE 2
#define BYDB_OP_LT 3
#define BYDB_OP_LE 4
#define BYDB_OP_GT 5
#define BYDB_OP_GE 6

typedef struct bydb_ctx bydb_ctx; /* owns one device, its streams and the HBM part cache */
typedef uint64_t bydb_part_h;

typedef struct {
    int32_t device;            /* CUDA device ordinal                                    */
    int32_t warps_per_sm;      /* scan workers per SM; 0 = default (16)                  */
    uint64_t hbm_budget_bytes; /* cap on resident part bytes; 0 = no cap                 */
    uint32_t flags;            /* BYDB_CFG_*                                             */
    uint32_t reserved;
} bydb_cfg;
#define BYDB_CFG_HOST_INDEX 1u /* bydb_part_register: parse the block index (meta.bin / primary.bin / *.tfm) on the host instead of
                                  with the device kernels (the default; both build the same directory -- the host parser is what
                                  the cold host-buffer paths use, where one frame's latency matters more than throughput) */

/* One file image of a part (banyand/measure/part.go:40-55).  name is one of "meta.bin",
 * "primary.bin", "timestamps.bin", "fv.bin", "<family>.tf", "<family>.tfm". */
typedef struct {
    const char *name;
    const uint8_t *data;
    uint64_t len;
} bydb_file;

typedef struct {
    uint32_t n_files;
    const bydb_file *files;
} bydb_part_files;

typedef struct {
    const char *family;   /* tag family name                                   */
    const char *tag;      /* tag name                                          */
    int32_t op;           /* BYDB_OP_*                                         */
    int32_t value_type;   /* BYDB_VT_STR / BYDB_VT_BINARY / BYDB_VT_INT64      */
    const uint8_t *lit;   /* literal bytes for STR/BINARY                      */
    uint64_t lit_len;
    int64_t lit_i64;      /* literal for INT64                                 */
} bydb_pred;

typedef struct {
    const char *field; /* field name (model.MeasureAgg input)       */
    int32_t func;      /* BYDB_AGG_*                                */
    int32_t reserved;
} bydb_agg;

/* bydb_query.flags */
#define BYDB_Q_HOST_ZERO_COPY 1u /* bydb_scan_agg_host only: the file images are in pinned, device-mapped host memory,
                                    16-byte aligned, with >= 64 readable bytes after each buffer; the kernels then read
                                    only the pages the query touches, in place over PCIe (no staging copy) */

#define BYDB_Q_ROW_PATH_TYPES 2u /* result typing of the reference's ROW path (a14 / a15): every aggregate, COUNT included, is typed
                                    like its field -- countFunc[N] is N-typed (pkg/query/aggregation/function.go:78-93,
                                    measure_plan_aggregation.go:152-175), so the count over a float64 field comes back as a float64.
                                    Default (flag clear) is the vectorized path's typing: COUNT is int64 (aggregation.go:425-430) */

/* One query = selected series (+ their dense group ids) x parts x predicates x aggregations.
 * Mirrors model.MeasureQueryOptions (pkg/query/model/model.go:75-88) after series resolution:
 * series_ids is what searchSeriesList returned (ascending, query.go:601), series_group is the
 * GroupBy key of each series densified by the caller in first-appearance order (entity / indexed
 * tags live in the series index, not in the part: SURVEY.md F3). */
typedef struct {
    uint32_t n_parts;
    const bydb_part_h *parts;
    uint64_t n_series;
    const uint64_t *series_ids;   /* ascending, unique                                   */
    const int32_t *series_group;  /* [n_series] dense group id; NULL = one group (scalar) */
    int32_t n_groups;             /* ignored when series_group is NULL                    */
    int32_t reserved0;
    int64_t tmin, tmax;           /* inclusive (pkg/timestamp/range.go:143)               */
    uint32_t n_preds;
    const bydb_pred *preds;       /* conjunction                                          */
    uint32_t n_aggs;
    const bydb_agg *aggs;
    int32_t top_n;                /* 0 = no Top                                           */
    int32_t top_agg;              /* index into aggs                                      */
    int32_t top_desc;             /* 1 = largest first                                    */
    uint32_t flags;               /* BYDB_Q_*                                             */
} bydb_query;

typedef struct {
    uint64_t rows_scanned;    /* rows of every selected block (before time trim)            */
    uint64_t rows_matched;    /* rows folded into an aggregate                               */
    uint64_t blocks_scanned;
    uint64_t page_bytes;      /* encoded page bytes the scan kernel consumed                 */
    uint64_t h2d_bytes;       /* host->device bytes moved by this call                       */
    uint64_t d2h_bytes;       /* device->host bytes moved by this call                       */
    double scan_kernel_ms;    /* CUDA-event time of the scan kernel on the call's stream     */
    double device_ms;         /* CUDA-event time of all kernels of the call                  */
    uint32_t kernel_launches; /* kernels launched by this call                               */
    uint32_t blocks_slow_lane; /* blocks the fast lane handed to the general decoder          */
    uint32_t slow_lane_reasons; /* OR of: 1 irregular timestamps, 2 int64 tag page, 4<<c field c needs the general decoder */
    uint32_t reserved;
} bydb_stats;

/* Dense result table; arrays are owned by the library until bydb_result_free.
 * Rows are groups in group-id order (groups that never appeared are omitted), or rank order when
 * top_n > 0.  Column a has type is_float[a]: COUNT is always int64, everything else follows the
 * field type (pkg/query/vectorized/measure/aggregation.go:425-430). */
typedef struct {
    int32_t n_rows;
    int32_t n_aggs;
    const int32_t *group_id;  /* [n_rows]            */
    const int64_t *rows;      /* [n_rows]            */
    const uint8_t *is_float;  /* [n_aggs]            */
    const int64_t *val_i64;   /* [n_rows * n_aggs]   */
    const double *val_f64;    /* [n_rows * n_aggs]   */
    bydb_stats stats;
    void *owner;              /* private             */
} bydb_result;

int bydb_init(const bydb_cfg *cfg, bydb_ctx **out);
void bydb_shutdown(bydb_ctx *ctx);

/* Upload an immutable part into HBM and build its block directory.  Idempotent per part_id. */
int bydb_part_register(bydb_ctx *ctx, uint64_t part_id, const bydb_part_files *files, bydb_part_h *out);
int bydb_part_release(bydb_ctx *ctx, bydb_part_h part);
/* resident bytes / block / row counts of a registered part */
int bydb_part_info(bydb_ctx *ctx, bydb_part_h part, uint64_t *hbm_bytes, uint64_t *n_blocks, uint64_t *n_rows);
/* Fallback pages of a registered part -- EncodeTypePlain numeric pages (null cells, floats that are not short
 * decimals; banyand/measure/column.go:147-153,203-208) and zstd-compressed string blocks (pkg/encoding/bytes.go:
 * 291-304): `unpacked` were rewritten into scan-friendly pages in HBM when the part was registered, `left` could
 * not be (a query that touches one of those returns BYDB_ENOTSUP). */
int bydb_part_fallback_pages(bydb_ctx *ctx, bydb_part_h part, uint64_t *unpacked, uint64_t *left);
/* Diagnostics: copies the part's DEVICE block directory (the DevBlock[64 B] / DevCol[16 B] records the scan kernels read,
 * csrc/part_dir.hpp) into caller buffers; either pointer may be NULL to only query the counts.  Tests compare the directory the
 * device index kernels build with the host parser's. */
int bydb_part_directory(bydb_ctx *ctx, bydb_part_h part, void *blocks_out, uint64_t blocks_cap_bytes, void *cols_out, uint64_t cols_cap_bytes,
                        uint64_t *n_blocks, uint64_t *n_cols);

/* Scan -> filter -> aggregate over parts already resident in HBM. */
int bydb_scan_agg(bydb_ctx *ctx, const bydb_query *q, bydb_result *out);

/* Group-by on a STORED tag: the key changes from row to row inside a series (a12; the vectorized path's BatchAggregation with
 * a non-entity key column, pkg/query/vectorized/measure/aggregation.go:193-254).  A row belongs to the group
 * (series_group of its series, value of the key tag in that row); groups come back in insertion order -- the scan order is
 * series by series (ascending series id), by time inside a series -- or in rank order when top_n > 0 (ties: the group
 * inserted first, top.go:62-76).  A nil cell and "" are the same key (groupby.go:226-254 encodes a string / bytes key as
 * length + raw bytes).  The key must be a string / binary tag stored with the dictionary encoding (<= 256 distinct values
 * per block, pkg/encoding/dictionary.go); a block that fell back to the plain bytes block makes the call return
 * BYDB_ENOTSUP, more than max_values distinct values over the selected blocks BYDB_ENOMEM (the reference's aggregation
 * memory budget), a value longer than 64 bytes BYDB_ENOTSUP.  Device side: one pass collects the distinct values from the
 * dictionary pages, then ONE SCAN PASS PER VALUE (the key as an extra predicate) fills that value's slice of a composite
 * partial table; stats count every pass.  Across GPUs: bydb_scan_reduce_keyed below.  Not available through the prepared /
 * partial-table / host-image entry points, and not over parts that overlap in time. */
typedef struct {
    const char *family;    /* tag family of the key tag                                      */
    const char *tag;       /* tag name                                                       */
    uint32_t max_values;   /* distinct key values accepted over the whole query; 0 = 64, at most 256 */
    uint32_t reserved;
} bydb_group_key;

typedef struct {
    bydb_result base;          /* rows as in bydb_result; base.group_id[r] = series_group of row r       */
    const int32_t *key_id;     /* [base.n_rows] key value of row r: index into the table below           */
    int32_t n_keys;            /* distinct key values found in the selected blocks (some may have no row) */
    int32_t reserved;
    const uint32_t *key_off;   /* [n_keys + 1] value k is key_bytes[key_off[k] .. key_off[k+1])          */
    const uint8_t *key_bytes;
    void *owner;               /* private                                                                 */
} bydb_keyed_result;

int bydb_scan_agg_keyed(bydb_ctx *ctx, const bydb_query *q, const bydb_group_key *key, bydb_keyed_result *out);
void bydb_keyed_result_free(bydb_ctx *ctx, bydb_keyed_result *r);

/* Write side (SURVEY 8 f4): numeric field pages encoded ON THE DEVICE, byte for byte what banyand/measure/column.go:113-234
 * (encodeInt64Column / encodeFloat64Column -> pkg/encoding/int_list.go:27-53, float.go:30-124) writes into fv.bin for a block:
 * [encode type][decimal exponent, float64 only][first value][zig-zag varint body].  The building block of a device-side merger
 * (decoded blocks in, pages out).  A float64 block that needs the reference's general shortest-digits search, holds NaN / Inf or
 * overflows on the common exponent is not encoded here: needs_cpu[b] = 1 and its page is empty -- the CPU writer (which owns the
 * EncodeTypePlain fallback page) takes it.  Columns with null cells are not accepted (they always take the fallback page). */
typedef struct {
    int32_t value_type;          /* BYDB_VT_INT64 / BYDB_VT_FLOAT64                                  */
    uint32_t n_blocks;
    const uint32_t *block_rows;  /* [n_blocks] rows of each block (>= 1)                              */
    const void *values;          /* HOST memory: int64_t / double values, the blocks back to back     */
} bydb_encode_input;

typedef struct {
    uint32_t n_blocks;
    uint32_t reserved;
    const uint64_t *page_off;    /* [n_blocks + 1] page b = bytes[page_off[b] .. page_off[b+1])       */
    const uint8_t *bytes;
    const uint8_t *needs_cpu;    /* [n_blocks]                                                        */
    uint64_t n_cpu_blocks;
    double device_ms;            /* CUDA-event time of the two kernels (encode + gather)              */
    void *owner;                 /* private                                                           */
} bydb_encoded_pages;

int bydb_encode_pages(bydb_ctx *ctx, const bydb_encode_input *in, bydb_encoded_pages *out);
void bydb_encoded_pages_free(bydb_ctx *ctx, bydb_encoded_pages *r);

/* Same, but the parts come as HOST file images: they are uploaded, scanned and dropped inside the
 * call (the end-to-end path of a cold query).  q->parts / q->n_parts are ignored. */
int bydb_scan_agg_host(bydb_ctx *ctx, uint32_t n_parts, const bydb_part_files *parts, const bydb_query *q, bydb_result *out);

void bydb_result_free(bydb_ctx *ctx, bydb_result *r);

/* Prepared queries.  A query that is executed many times (dashboard refresh, alert rule) is copied and planned once;
 * from its third execution on, the whole step -- staging copy, block selection, scan, reduce, finalisation, row
 * selection, read-back -- is replayed as ONE captured CUDA graph: one launch and one synchronisation per call instead of
 * ~20 runtime calls.  Every execution still scans the parts (nothing is cached but the launch sequence).  Results and
 * errors are those of bydb_scan_agg; stats.scan_kernel_ms is 0 on replays (per-kernel events do not exist inside a
 * graph), stats.device_ms is the whole graph.  Queries whose parts overlap in time (version dedup needs a host
 * decision) transparently keep the ordinary path.  One execution at a time per prepared query; different prepared
 * queries run concurrently.  The parts named by the query must stay registered while it exists. */
typedef struct bydb_prepared bydb_prepared;
int bydb_query_prepare(bydb_ctx *ctx, const bydb_query *q, bydb_prepared **out);
int bydb_scan_agg_prepared(bydb_ctx *ctx, bydb_prepared *pq, bydb_result *out);
void bydb_query_release(bydb_ctx *ctx, bydb_prepared *pq);

/* ---- multi-GPU map/reduce: per-rank partial tables, one collective, one finalize ----
 * Layout of a partial table for (n_groups G, n_fields F = distinct aggregated fields):
 *   double  sum_f64[G*F]; double max_f64[G*F]; double negmin_f64[G*F];
 *   int64   sum_i64[G*F]; int64 cnt[G*F]; int64 rows[G]; int64 max_i64[G*F]; int64 negmin_i64[G*F];
 * so that ONE all-reduce(SUM) over [sum_f64] + [sum_i64,cnt,rows] and one all-reduce(MAX) over the
 * max/negmin halves combine ranks (min is carried as max of the negation; int64 negation of
 * INT64_MIN is handled by carrying ~x instead of -x).  bydb_partials_layout reports the byte
 * offsets so the caller can issue the collectives on sub-ranges. */
typedef struct {
    uint64_t total_bytes;
    uint64_t off_sum_f64, off_max_f64;   /* [sum_f64] , [max_f64 | negmin_f64]                 */
    uint64_t off_sum_i64, off_max_i64;   /* [sum_i64 | cnt | rows] , [max_i64 | notmin_i64]    */
    uint64_t n_sum_f64, n_max_f64, n_sum_i64, n_max_i64; /* element counts of the four ranges */
} bydb_partials_layout_t;

int bydb_partials_layout(const bydb_query *q, bydb_partials_layout_t *out);
/* Run the scan and leave the partial table in caller-provided DEVICE memory (e.g. a torch tensor),
 * enqueued on `stream` (a cudaStream_t passed as void*; NULL = the CUDA legacy default stream, for this call
 * and for bydb_partials_combine / bydb_reduce_finalize alike, so consecutive calls are always ordered).
 * stats != NULL: the call waits for the scan, fills *stats and reports device-side failures itself.
 * stats == NULL: ASYNCHRONOUS -- the call returns once the work is enqueued, so the collective that ships the
 * table can be enqueued right behind it with no host round trip; a device-side failure (corrupt page, ...) then
 * travels inside the table and is returned by bydb_reduce_finalize on whichever rank finalises. */
int bydb_scan_partials(bydb_ctx *ctx, const bydb_query *q, void *d_partials, uint64_t bytes, void *stream, bydb_stats *stats);
/* Combine n_tables partial tables laid out back to back in DEVICE memory (e.g. the output of ONE all-gather of the
 * per-rank tables) into the first one, in rank order: sums add, max ranges take the maximum.  Deterministic. */
int bydb_partials_combine(bydb_ctx *ctx, const bydb_query *q, void *d_tables, uint32_t n_tables, uint64_t bytes_each, void *stream);
/* Finalize a (reduced) partial table: MEAN finalisation, output typing, Top-N; copies the result to host. */
int bydb_reduce_finalize(bydb_ctx *ctx, const bydb_query *q, const void *d_partials, uint64_t bytes, void *stream, bydb_result *out);

/* Map-phase rows in the reference's wire shape (a18 / f3): what a data node answers when the liaison asks for partials
 * (InternalQueryRequest.agg_return_partial -> mapAccumulator.Result with emitPartial, measure_plan_aggregation.go:67-84;
 * aggregation.PartialToFieldValues, pkg/query/aggregation/aggregation.go:128-145).  One row per group that appeared; aggregate a
 * carries Partial.Value -- SUM: the sum, COUNT: the count, MAX / MIN: the extreme (the N-typed sentinel when no value was
 * folded, aggregation.go:169-191), MEAN: the SUM -- and, for MEAN only, Partial.Count, which the Go side ships as the extra
 * field "__agg_count".  Everything is typed like the FIELD (the row path is N-typed: the count over a float64 field is a
 * float64; function.go:20-236).  The liaison's reduceAccumulator.Combine consumes exactly these pairs. */
typedef struct {
    int32_t n_rows;
    int32_t n_aggs;
    const int32_t *group_id;  /* [n_rows]                                             */
    const uint8_t *is_float;  /* [n_aggs] N of aggregate a = its field's type         */
    const int64_t *val_i64;   /* [n_rows * n_aggs] Partial.Value when !is_float[a]    */
    const double *val_f64;    /* [n_rows * n_aggs] Partial.Value when  is_float[a]    */
    const int64_t *cnt_i64;   /* [n_rows * n_aggs] Partial.Count (MEAN only, else 0)  */
    const double *cnt_f64;
    void *owner;              /* private                                              */
} bydb_partial_rows;
int bydb_partials_rows(bydb_ctx *ctx, const bydb_query *q, const void *d_partials, uint64_t bytes, void *stream, bydb_partial_rows *out);
void bydb_partial_rows_free(bydb_ctx *ctx, bydb_partial_rows *r);

/* ---- multi-GPU reduce behind the C ABI: one process (or thread) per GPU, no torch, no NCCL ----
 * Replaces the liaison gather + reduceAccumulator.Combine (pkg/query/logical/measure/measure_plan_aggregation.go:96-124,
 * measure_plan_distributed.go:254-328) inside one node: every rank owns a MAILBOX in its GPU's memory; in a collective
 * bydb_scan_reduce each rank's reduce kernel writes its partial table straight into its slot of the ROOT's mailbox (peer
 * memory: the stores travel over NVLink / NVSwitch) and raises an arrival flag there; the root waits for the flags on the
 * device, combines the slots in rank order (deterministic float sums) and finalises.  No data-path library collective.
 *
 *   1. every rank:  bydb_comm_export(ctx, max_table_bytes, max_ranks, &h)     -- allocates the mailbox, h is 128 opaque bytes
 *   2. the caller exchanges the handles by any channel it has (gRPC between data nodes, a pipe, torch all_gather in tests)
 *   3. every rank:  bydb_comm_connect(ctx, rank, nranks, handles)             -- opens the peers' mailboxes (CUDA IPC between
 *                   processes, plain peer access between contexts of one process)
 *   4. every rank, in the same order:  bydb_scan_reduce(ctx, &q, root, &out)  -- q names THIS rank's parts and series; group
 *                   layout, aggregations and Top-N must be the same on all ranks.  The root gets the result; the others get
 *                   n_rows = 0 and their own scan statistics.  A rank that fails to arrive makes the root return BYDB_EIO
 *                   after a bounded wait; a device-side scan error of any rank travels in its table and fails the root's call.
 * max_table_bytes: the largest bydb_partials_layout().total_bytes of the queries to come. */
typedef struct { uint8_t bytes[128]; } bydb_comm_handle;
int bydb_comm_export(bydb_ctx *ctx, uint64_t max_table_bytes, int32_t max_ranks, bydb_comm_handle *out);
int bydb_comm_connect(bydb_ctx *ctx, int32_t rank, int32_t nranks, const bydb_comm_handle *all);
int bydb_scan_reduce(bydb_ctx *ctx, const bydb_query *q, int32_t root, bydb_result *out);
/* The same collective for a prepared query (bydb_query_prepare): from its second execution on, per root, the rank's whole step is
 * replayed as ONE captured CUDA graph -- the epoch of the call travels in a small device block that a memcpy node of the graph
 * refreshes.  Ranks may mix bydb_scan_reduce and bydb_scan_reduce_prepared within one collective. */
int bydb_scan_reduce_prepared(bydb_ctx *ctx, bydb_prepared *pq, int32_t root, bydb_result *out);
/* The same collective with every rank's parts given as HOST file images (cold distributed query, end to end): admitted for
 * the duration of the call (with BYDB_Q_HOST_ZERO_COPY only the block directory is uploaded and the scan pulls the pages it
 * touches over PCIe), scanned into the root's mailbox, dropped.  q->parts / q->n_parts are ignored. */
int bydb_scan_reduce_host(bydb_ctx *ctx, uint32_t n_parts, const bydb_part_files *parts, const bydb_query *q, int32_t root, bydb_result *out);

/* Group-by on a stored tag as a collective (bydb_scan_agg_keyed across the connected ranks): the root gets exactly what ONE
 * context scanning every rank's parts and series would return from bydb_scan_agg_keyed -- the same rows in the same order
 * (insertion order, or Top-N rank order with ties to the group inserted first), the same key bytes and series group per row,
 * int64 results, counts, min and max bit-identical; float sums add the ranks in rank order (within 1e-12 relative of the
 * single-context sum).  Key ids index the root's key table, which numbers the values in order of first occurrence over
 * (rank, that rank's own value order).  Every rank passes the same series-group count, aggregations, Top-N, key and
 * max_values; q names THIS rank's parts and series.  A series may live on several ranks only in pieces that do not overlap in
 * time (the duplicate rule of bydb_scan_reduce).  The other ranks get n_rows = 0, n_keys = 0 and their own scan statistics.
 * Each rank finds its own distinct values, runs one scan pass per value into its slot of the root's mailbox and leaves there its
 * dictionary and where each composite group first showed; the root unites the dictionaries, folds the slices in rank order and
 * restores the insertion order on the device.  Epochs, slot parities and waits are bydb_scan_reduce's: keyed and plain
 * collectives may alternate on the same mailboxes, and a failure on any rank leaves them usable.  Errors: a rank's own failure
 * (BYDB_ENOTSUP for a plain-encoded key block or a value over 64 bytes, BYDB_EINVAL for a key tag that is not a string / binary
 * dictionary tag or a slot too small for the table, BYDB_ENOMEM for more than max_values values on that rank, BYDB_ENOTSUP for
 * parts of that rank that overlap in time) is returned by that rank and by the root; more than max_values distinct values over
 * all ranks is BYDB_ENOMEM on the root.
 * bydb_keyed_reduce_layout (host only) gives the slot size such a query needs: pass the largest over the queries to come (and
 * over bydb_partials_layout().total_bytes of the plain collectives) as max_table_bytes of bydb_comm_export. */
int bydb_keyed_reduce_layout(const bydb_query *q, const bydb_group_key *key, uint64_t *slot_bytes);
int bydb_scan_reduce_keyed(bydb_ctx *ctx, const bydb_query *q, const bydb_group_key *key, int32_t root, bydb_keyed_result *out);

const char *bydb_last_error(void);
const char *bydb_version(void);

#ifdef __cplusplus
}
#endif
#endif
