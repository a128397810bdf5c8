/*
 * flockgpu.h -- C ABI of the B200-native executor for Flock's per-batch hot path.
 *
 * Every entry point below is what the reference-side FFI binding would bind (the Rust shim under
 * rust/flock-gpu-exec/ and INTEGRATION.md show that binding).  The reference has no FFI today: the
 * path sits behind the DataFusion `ExecutionPlan` trait object (flock/src/runtime/plan.rs:139-146),
 * driven by `collect`/`collect_partitioned` (flock/src/runtime/context.rs:172-216).  Each group of
 * functions cites the reference interface it replaces.
 *
 * Conventions
 *   - every function returns 0 on success and a negative FLOCKGPU_ERR_* code on failure; the message
 *     is available through flockgpu_last_error() (thread-local).  Nothing unwinds or aborts: the
 *     reference is built with panic='abort' (Cargo.toml [profile.release]), so an unwound panic
 *     would kill the Lambda instance.
 *   - record batches cross the boundary through the Arrow C Data Interface (struct ArrowSchema /
 *     struct ArrowArray, arrow/c/abi.h).  Inputs are BORROWED for the duration of the call (the
 *     caller keeps `release`); outputs are new arrays owned by this library until the consumer calls
 *     their `release` callback.  Inputs are never mutated (flock/src/datasource/nexmark/queries/
 *     q5.rs:127-131 asserts that).
 *   - a flockgpu_table is an immutable, reference-counted, device-resident relation: the columns of
 *     one or more RecordBatches laid out contiguously in HBM.  Operators map tables to tables without
 *     touching the host.
 *   - a flockgpu_ctx owns one CUDA stream; calls on one ctx are serialised by an internal mutex, so a
 *     ctx may be shared between threads (DataFusion calls `execute(partition)` concurrently,
 *     context.rs:178).  Use one ctx per thread for concurrency.
 */
#ifndef FLOCKGPU_H
#define FLOCKGPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- Arrow C Data Interface (verbatim ABI from the Arrow specification) ---------------------- */
#ifndef ARROW_C_DATA_INTERFACE
#define ARROW_C_DATA_INTERFACE
#define ARROW_FLAG_DICTIONARY_ORDERED 1
#define ARROW_FLAG_NULLABLE 2
#define ARROW_FLAG_MAP_KEYS_SORTED 4
struct ArrowSchema {
  const char* format;
  const char* name;
  const char* metadata;
  int64_t flags;
  int64_t n_children;
  struct ArrowSchema** children;
  struct ArrowSchema* dictionary;
  void (*release)(struct ArrowSchema*);
  void* private_data;
};
struct ArrowArray {
  int64_t length;
  int64_t null_count;
  int64_t offset;
  int64_t n_buffers;
  int64_t n_children;
  const void** buffers;
  struct ArrowArray** children;
  struct ArrowArray* dictionary;
  void (*release)(struct ArrowArray*);
  void* private_data;
};
#endif

/* ---- error codes ------------------------------------------------------------------------------ */
#define FLOCKGPU_OK 0
#define FLOCKGPU_ERR_INVALID (-1)     /* bad argument / malformed plan or expression            */
#define FLOCKGPU_ERR_UNSUPPORTED (-2) /* valid, but outside what the GPU path implements        */
#define FLOCKGPU_ERR_CUDA (-3)        /* CUDA runtime error (message carries file:line)         */
#define FLOCKGPU_ERR_NCCL (-4)        /* NCCL error                                             */
#define FLOCKGPU_ERR_EXECUTION (-5)   /* run-time data error (e.g. divide by zero), maps to     */
                                      /* FlockError::Execution (flock/src/error.rs:28-76)       */
#define FLOCKGPU_ERR_NO_DEVICE (-6)   /* no CUDA device: there is NO CPU fallback               */

typedef struct flockgpu_ctx flockgpu_ctx;
typedef struct flockgpu_table flockgpu_table;

/* ---- context ---------------------------------------------------------------------------------- */
/* Opens device `device` (cudaSetDevice) and creates the stream, memory pool and scratch state.    */
int flockgpu_open(int device, flockgpu_ctx** out);
int flockgpu_close(flockgpu_ctx* ctx);
/* Message of the last error raised on the calling thread ("" if none). Never NULL.                */
const char* flockgpu_last_error(void);
/* Library build description, e.g. "flockgpu 0.1 sm_100a".                                          */
const char* flockgpu_version(void);
/* Blocks until every operation queued on the ctx stream has completed.                            */
int flockgpu_synchronize(flockgpu_ctx* ctx);
/* CUDA-event timers on the ctx stream (bench.py times kernels with these: torch.cuda.Event only
 * sees torch's own stream).  `slot` in [0, 16).                                                    */
int flockgpu_timer_start(flockgpu_ctx* ctx, int slot);
int flockgpu_timer_stop(flockgpu_ctx* ctx, int slot);              /* records the stop event       */
int flockgpu_timer_elapsed_ms(flockgpu_ctx* ctx, int slot, float* ms); /* syncs on the stop event  */
/* Number of kernels this library has launched on the ctx since it was opened.                     */
int64_t flockgpu_kernel_launches(flockgpu_ctx* ctx);
/* Bytes that have crossed the host link for this ctx since it was opened: direction 0 = host -> device (copies issued
 * by table import / feed_data_sources plus what kernels read in place from page-locked batches under "feed_zero_copy"),
 * 1 = device -> host (table export).  bench.py's e2e leg reports the difference across its timed region.             */
int64_t flockgpu_bytes_moved(flockgpu_ctx* ctx, int32_t direction);
/* Context options.  "feed_zero_copy" (0/1, default 0): flock_context_feed_data_sources leaves fixed-width columns
 * whose buffers are page-locked (flockgpu_host_alloc / cudaHostRegister) and uniformly batched (every batch but the
 * last has the same power-of-two row count >= 4096) in HOST memory; the vectorised filter then reads them in place
 * over PCIe and other operators copy them to HBM on first use.  With the option on, fed batches must stay alive and
 * unmodified until flock_context_clean_data_sources -- exactly what the reference does anyway: MemoryExec owns the fed
 * RecordBatches until clean_data_sources (flock/src/runtime/context.rs:227-254).
 * "compact_mode" (0 automatic | 1 always decoupled look-back): which grid-wide prefix protocol the compaction /
 * scan kernels use; results are identical, the parity tests run both.
 * "exchange_window_mb" (default 4096): size of the receive window the multi-GPU exchange stores rows into over NVLink
 * peer memory; read by flockgpu_comm_init, so set it first.
 * Feeding PAGEABLE batches (what arrow-rs allocates): "feed_stage_threads" (default 8, 0 = plain cudaMemcpyAsync): host
 * threads that copy the batches into a page-locked ring ahead of the DMA; "feed_stream_stores" (default 1): those copies
 * use non-temporal stores; "feed_register" (default 0): page-lock the caller's buffers in place (cudaHostRegister) for
 * the span feed .. clean instead of staging them.  "host_trace_dump": print the host-side spans collected under
 * FLOCKGPU_HOST_TRACE=1.                                                                                              */
int flockgpu_set_option(flockgpu_ctx* ctx, const char* name, int64_t value);
/* Per-kernel device timing: between _begin and _end every kernel this library launches on the ctx is
 * bracketed by its own pair of CUDA events on the ctx stream.  _end waits for the stream and writes a JSON
 * object {"<kernel>": {"launches": n, "ms": total}, ...} into out_json (bench.py's roofline numerator).  */
int flockgpu_profile_begin(flockgpu_ctx* ctx);
int flockgpu_profile_end(flockgpu_ctx* ctx, char* out_json, int32_t capacity);
/* Pinned host memory (page-locked) for staging Arrow buffers: bench.py's e2e leg and the Rust shim
 * allocate record-batch buffers here so that host<->device copies are true DMA and the zero-copy feed can read them
 * in place.  Blocks are 256-byte aligned and carved out of 64 MB page-locked slabs in allocation order (buffers
 * allocated one after the other are contiguous: few large GPU mappings instead of one per buffer); a slab's space
 * returns when all of its blocks have been freed -- the lifetime pattern of record batches.            */
int flockgpu_host_alloc(flockgpu_ctx* ctx, int64_t bytes, void** out);
int flockgpu_host_free(flockgpu_ctx* ctx, void* ptr);
/* Overwrites a scratch buffer larger than L2 (126 MB) so that the next timed launch starts cold.   */
int flockgpu_flush_l2(flockgpu_ctx* ctx);

/* ---- tables: the MemoryExec leaf (datafusion MemoryExec::set_partitions, fed by
 *      ExecutionContext::feed_data_sources, flock/src/runtime/context.rs:257-325) ---------------- */
/* Host -> HBM.  `schema` is a struct schema ("+s"); `batches[i]` are struct arrays of that schema.
 * `projection` (may be NULL = all columns) selects and orders the columns that are copied -- the
 * MemoryExec `projection` of the reference plan (flock/src/tests/data/plan/join.json: "projection": [0, 1]).
 * Supported column types: Int32 "i", UInt32 "I", Int64 "l", UInt64 "L", Float64 "g",
 * Timestamp "ts?:..", Utf8 "u".  Arrays with nulls are rejected with FLOCKGPU_ERR_UNSUPPORTED
 * (every NEXMark field is non-nullable, event.rs:130-149, :220-245, :336-352).                     */
int flockgpu_table_import(flockgpu_ctx* ctx, const struct ArrowSchema* schema,
                          const struct ArrowArray* const* batches, int32_t n_batches,
                          const int32_t* projection, int32_t n_projection, flockgpu_table** out);
/* HBM -> host.  Fills `out_schema` / `out_array` (a struct array) with rows [row_begin, row_begin +
 * row_count) of the table; row_count < 0 means "to the end".  Blocks until the copy has finished.  */
int flockgpu_table_export(flockgpu_ctx* ctx, const flockgpu_table* table, int64_t row_begin,
                          int64_t row_count, struct ArrowSchema* out_schema,
                          struct ArrowArray* out_array);
/* ---- payload frames: Arrow IPC record-batch messages <-> tables (flock/src/runtime/payload.rs:161-192
 *      Payload::to_record_batch = flight_data_to_arrow_batch per DataFrame; flock/src/transmute.rs:178-247 to_payload /
 *      to_bytes = flight_data_from_arrow_batch; the arena hands the frames over, runtime/arena/mod.rs:114-169) ------- */
/* Host -> HBM from `n_frames` DataFrame { header, body } pairs (Encoding::None): header = the flatbuffer Message of a
 * RecordBatch (FlightData.data_header), body = its buffers (FlightData.data_body).  Nothing is decoded: the body
 * buffers are the column buffers, only their extents are read from the header.  `schema` / `projection` as in
 * flockgpu_table_import; frames with nulls, dictionaries or compressed bodies are rejected (FLOCKGPU_ERR_UNSUPPORTED). */
int flockgpu_table_import_ipc(flockgpu_ctx* ctx, const struct ArrowSchema* schema, const uint8_t* const* headers, const int64_t* header_lens,
                              const uint8_t* const* bodies, const int64_t* body_lens, int32_t n_frames, const int32_t* projection,
                              int32_t n_projection, flockgpu_table** out);
/* HBM -> one DataFrame for rows [row_begin, row_begin + row_count) (row_count < 0: to the end): *out_header receives a
 * flatbuffer Message { RecordBatch } (MetadataVersion V5, 8-byte aligned buffers, what arrow-rs writes), *out_body the
 * buffers.  Both blocks belong to the caller and are released with flockgpu_ipc_free.                                */
int flockgpu_table_export_ipc(flockgpu_ctx* ctx, const flockgpu_table* table, int64_t row_begin, int64_t row_count, uint8_t** out_header,
                              int64_t* out_header_len, uint8_t** out_body, int64_t* out_body_len);
void flockgpu_ipc_free(uint8_t* block);
/* ---- NDJSON events -> table: event_bytes_to_batch (flock/src/transmute.rs:255-266; call sites flock/src/datasource/
 *      nexmark/nexmark.rs:181-203), the schema-driven arrow json::Reader over the generator's serde_json lines ---------
 * One flat JSON object per line; fields are matched BY NAME in any order, unknown fields (nested values included) are
 * skipped; Int32/UInt32/Int64/UInt64/Timestamp columns take JSON integers in range, Float64 numbers of at most 15
 * significant digits and |exponent| <= 22 (exact with one IEEE operation), Utf8 JSON strings (unescaped, \uXXXX and
 * surrogate pairs to UTF-8).  A malformed line, a missing field or a null fails the call with FLOCKGPU_ERR_EXECUTION
 * naming the first bad line.  `data` is borrowed for the call.                                                          */
int flockgpu_table_import_ndjson(flockgpu_ctx* ctx, const struct ArrowSchema* schema, const uint8_t* data, int64_t n_bytes,
                                 flockgpu_table** out);
/* Schema only (no data movement).                                                                  */
int flockgpu_table_schema(flockgpu_ctx* ctx, const flockgpu_table* table,
                          struct ArrowSchema* out_schema);
int flockgpu_table_retain(flockgpu_table* table);
int flockgpu_table_release(flockgpu_table* table);
int64_t flockgpu_table_num_rows(const flockgpu_table* table);
int32_t flockgpu_table_num_columns(const flockgpu_table* table);
/* Bytes of HBM the table's buffers occupy (data + offsets).                                        */
int64_t flockgpu_table_nbytes(const flockgpu_table* table);
/* Concatenates tables of identical schema (CoalesceBatchesExec / concat, transmute.rs:55-72).      */
int flockgpu_table_concat(flockgpu_ctx* ctx, flockgpu_table* const* tables, int32_t n,
                          flockgpu_table** out);

/* ---- window assembly on the device (flock-function/src/aws/window/hopping.rs:54-74, tumbling.rs; the Arena that
 *      collects a window's pieces: flock/src/runtime/arena/mod.rs:60-85) ------------------------------------------------
 * A window is `window_size` consecutive epochs (the reference's epochs are seconds); every hop drops the oldest
 * `hop_size` epochs and waits for as many new ones (hop_size = window_size: tumbling).  Epoch relations stay resident
 * in HBM between invocations: a hop uploads the new epochs only, and the relation a plan scans is concatenated on
 * the device.                                                                                                          */
typedef struct flockgpu_window flockgpu_window;
int flockgpu_window_open(flockgpu_ctx* ctx, int32_t window_size, int32_t hop_size, flockgpu_window** out);
int flockgpu_window_close(flockgpu_window* w);
/* The relation of the next epoch (retained; the caller may release its handle).                                        */
int flockgpu_window_push(flockgpu_window* w, flockgpu_table* epoch);
/* *out = 1 when `window_size` epochs are buffered.                                                                      */
int flockgpu_window_ready(const flockgpu_window* w, int32_t* out);
/* The next window as one relation (epochs in order); *first_epoch (may be NULL) = number of its first epoch; the
 * window then moves forward by `hop_size` epochs.                                                                       */
int flockgpu_window_next(flockgpu_window* w, flockgpu_table** out, int64_t* first_epoch);

/* ---- expressions: the PhysicalExpr trees of FilterExec / ProjectionExec ------------------------
 * A program is the postfix (RPN) encoding of a DataFusion physical expression
 * (column / literal / cast_expr / try_cast_expr / binary_expr / not, as serialised in
 * flock/src/tests/data/plan/aggregate.json "predicate").                                           */
enum flockgpu_dtype {
  FLOCKGPU_BOOL = 0,
  FLOCKGPU_INT32 = 1,
  FLOCKGPU_INT64 = 2,
  FLOCKGPU_UINT64 = 3,
  FLOCKGPU_FLOAT64 = 4,
  FLOCKGPU_TIMESTAMP = 5, /* int64 storage; unit/timezone carried by the Arrow format string */
  FLOCKGPU_UTF8 = 6,
  FLOCKGPU_UINT32 = 7
};
enum flockgpu_op {
  FLOCKGPU_OP_COLUMN = 1,   /* push column `col` of the input table                              */
  FLOCKGPU_OP_LIT_I64 = 2,  /* push Int64 literal `i64` (ScalarValue::Int64; also Int32 etc.)    */
  FLOCKGPU_OP_LIT_F64 = 3,  /* push Float64 literal `f64`                                        */
  FLOCKGPU_OP_LIT_UTF8 = 4, /* push Utf8 literal (`str`, `str_len`)                              */
  FLOCKGPU_OP_CAST = 5,     /* pop x, push CAST(x AS dtype)                                      */
  FLOCKGPU_OP_ADD = 10, FLOCKGPU_OP_SUB = 11, FLOCKGPU_OP_MUL = 12, FLOCKGPU_OP_DIV = 13,
  FLOCKGPU_OP_MOD = 14,     /* truncated remainder, sign of the dividend (Rust `%`)              */
  FLOCKGPU_OP_EQ = 20, FLOCKGPU_OP_NE = 21, FLOCKGPU_OP_LT = 22, FLOCKGPU_OP_LE = 23,
  FLOCKGPU_OP_GT = 24, FLOCKGPU_OP_GE = 25,
  FLOCKGPU_OP_AND = 30, FLOCKGPU_OP_OR = 31, FLOCKGPU_OP_NOT = 32
};
typedef struct flockgpu_expr_token {
  int32_t op;      /* enum flockgpu_op                                      */
  int32_t dtype;   /* enum flockgpu_dtype: CAST target / literal type       */
  int32_t col;     /* FLOCKGPU_OP_COLUMN: input column index                */
  int32_t str_len; /* FLOCKGPU_OP_LIT_UTF8                                  */
  int64_t i64;
  double f64;
  const char* str;
} flockgpu_expr_token;
typedef struct flockgpu_expr {
  const flockgpu_expr_token* tokens;
  int32_t n_tokens;
} flockgpu_expr;

/* ---- FilterExec + CoalesceBatchesExec + ProjectionExec, fused (planner.rs:90-92, :120-124) -----
 * out = SELECT projection[0..n) FROM in WHERE predicate.  `predicate` may be NULL (pure
 * projection); `projections` may be NULL with n_projections = 0 (all input columns pass through).
 * Surviving rows keep their input order (arrow `filter_record_batch`).  Pass-through columns of a
 * pure projection are zero-copy (they share the input's HBM buffers, like `Arc` clones in
 * ProjectionExec).  `out_names[i]` names output column i (NULL: keep / derive).                    */
int flockgpu_filter_project(flockgpu_ctx* ctx, const flockgpu_table* in,
                            const flockgpu_expr* predicate, const flockgpu_expr* projections,
                            const char* const* out_names, int32_t n_projections,
                            flockgpu_table** out);

/* ---- HashAggregateExec (modes as in stage.rs:535-543, :597-600) ------------------------------- */
enum flockgpu_agg_mode {
  FLOCKGPU_AGG_PARTIAL = 0,           /* rows -> (keys, state columns "<name>[count]" ...)        */
  FLOCKGPU_AGG_FINAL = 1,             /* states -> values (single partition)                       */
  FLOCKGPU_AGG_FINAL_PARTITIONED = 2, /* states -> values (input hash-partitioned on the keys)     */
  FLOCKGPU_AGG_SINGLE = 3             /* rows -> values: Partial + Final fused on one GPU          */
};
enum flockgpu_agg_func {
  FLOCKGPU_AGG_COUNT = 0, FLOCKGPU_AGG_SUM = 1, FLOCKGPU_AGG_MIN = 2, FLOCKGPU_AGG_MAX = 3,
  FLOCKGPU_AGG_AVG = 4
};
typedef struct flockgpu_agg_spec {
  int32_t func; /* enum flockgpu_agg_func                                                         */
  int32_t col;  /* PARTIAL/SINGLE: input column (-1 for COUNT(*) i.e. COUNT(UInt8(1)));           */
                /* FINAL*: index of the FIRST state column of this aggregate in the input          */
  const char* name; /* output name, e.g. "COUNT(UInt8(1))"; state columns append "[count]" ...     */
} flockgpu_agg_spec;
/* Group columns come first in the output, then one column per aggregate (two state columns
 * "[count]","[sum]" for AVG in PARTIAL mode).  n_group_cols = 0 is the global aggregate (one row,
 * even over empty input: COUNT = 0, others NULL -- the only place a NULL can appear).  An empty
 * aggregate list is the DISTINCT-style group-by of NEXMark q8.  Group order in the output is
 * unspecified (the reference compares sorted, flock/src/launcher/aws/mod.rs:675).                  */
int flockgpu_hash_aggregate(flockgpu_ctx* ctx, const flockgpu_table* in, int32_t mode,
                            const int32_t* group_cols, int32_t n_group_cols,
                            const flockgpu_agg_spec* aggs, int32_t n_aggs, flockgpu_table** out);

/* ---- HashJoinExec { mode: Partitioned, join_type: Inner | Left | Right | Full | Semi | Anti } (planner.rs:169, :239)
 * Inner: out = left ++ right columns for every pair with equal keys (NULL != NULL; duplicates give the
 * full cross product).  `left` is the textual left of the SQL join, as in the reference.  Key column
 * types must match pairwise (Int32/Int64/UInt64/Timestamp/Utf8).
 * The other DataFusion 6 join types (flockgpu_hash_join_typed):
 *   Left   left ++ right: every pair, plus each left row without a match, its right columns NULL
 *   Right  left ++ right: every pair, plus each right row without a match, its left columns NULL
 *   Full   Left and Right together: pairs, unmatched left rows, unmatched right rows
 *   Semi   left columns only: each left row with at least one match, once, in left input order
 *   Anti   left columns only: each left row without a match, in left input order
 * A row whose key is NULL matches nothing but is still a row of its side (kept by Left / Right / Full,
 * returned by Anti).  The padded side's columns are nullable in the output; a padded value is NULL
 * (fixed width 0, Utf8 empty).  Row order of Inner / Left / Right / Full is unspecified.           */
enum flockgpu_join_type {
  FLOCKGPU_JOIN_INNER = 0, FLOCKGPU_JOIN_LEFT = 1, FLOCKGPU_JOIN_RIGHT = 2, FLOCKGPU_JOIN_FULL = 3,
  FLOCKGPU_JOIN_SEMI = 4, FLOCKGPU_JOIN_ANTI = 5
};
/* Inner join; the same as flockgpu_hash_join_typed(..., FLOCKGPU_JOIN_INNER, out). */
int flockgpu_hash_join(flockgpu_ctx* ctx, const flockgpu_table* left, const flockgpu_table* right,
                       const int32_t* left_keys, const int32_t* right_keys, int32_t n_keys,
                       flockgpu_table** out);
/* Any join type; an unknown `join_type` is FLOCKGPU_ERR_INVALID. */
int flockgpu_hash_join_typed(flockgpu_ctx* ctx, const flockgpu_table* left, const flockgpu_table* right,
                             const int32_t* left_keys, const int32_t* right_keys, int32_t n_keys,
                             int32_t join_type, flockgpu_table** out);

/* ---- SortExec / WindowAggExec(ROW_NUMBER) / GlobalLimitExec: what NEXMark q6 adds (benchmarks/src/nexmark/query/
 *      q6.sql, q6_plan.fmt; serialised sort_exec / global_limit_exec: flock/src/tests/data/plan/join.json) ------------- */
/* Rows ordered by cols[0] (descending[0] != 0: DESC), then cols[1] ...; rows that tie on every sort column are ordered
 * by the remaining columns, ascending, in column order (the reference leaves ties undefined; this is the oracle's
 * choice, and it makes the result independent of the input order).  Fixed-width, non-null columns only.               */
int flockgpu_sort(flockgpu_ctx* ctx, const flockgpu_table* in, const int32_t* cols, const int32_t* descending, int32_t n_keys,
                  flockgpu_table** out);
/* ROW_NUMBER() OVER (PARTITION BY partition_cols ORDER BY <the order `in` is sorted in>): `in` must be sorted so that
 * the rows of a window partition are contiguous (the SortExec DataFusion plans below every WindowAggExec).  The UInt64
 * window column `name` comes FIRST in the output, then the input columns (WindowAggExec's schema).                       */
int flockgpu_row_number(flockgpu_ctx* ctx, const flockgpu_table* in, const int32_t* partition_cols, int32_t n_cols, const char* name,
                        flockgpu_table** out);
/* The first `limit` rows.                                                                                                */
int flockgpu_limit(flockgpu_ctx* ctx, const flockgpu_table* in, int64_t limit, flockgpu_table** out);

/* ---- RepartitionExec: Hash([keys], n) (planner.rs:153, :160; call shape
 *      playground/src/distributed_plan/shuffle_writer.rs:105-146) -------------------------------- */
/* Splits `in` into n_parts tables by hash(keys) -- rows keep their input order inside a partition.
 * The hash is Murmur3-fmix based, not ahash: partition membership is not observable in results
 * (SURVEY.md Appendix C.6); what matters is that equal keys meet in one partition and that both
 * join sides use the same function.                                                                */
int flockgpu_hash_partition(flockgpu_ctx* ctx, const flockgpu_table* in, const int32_t* key_cols,
                            int32_t n_keys, int32_t n_parts, flockgpu_table** out_parts);

/* ---- multi-GPU exchange: the hash shuffle between stages (flock-function/src/aws/actor.rs:
 *      425-543 = N x M Lambda invokes) as ONE all-to-all over NVLink ----------------------------- */
#define FLOCKGPU_UNIQUE_ID_BYTES 128
/* Rank 0 creates the id and distributes the bytes out of band (bench.py: torch.distributed).       */
int flockgpu_comm_unique_id(uint8_t out_id[FLOCKGPU_UNIQUE_ID_BYTES]);
int flockgpu_comm_init(flockgpu_ctx* ctx, const uint8_t id[FLOCKGPU_UNIQUE_ID_BYTES], int32_t rank,
                       int32_t world_size);
int flockgpu_comm_rank(flockgpu_ctx* ctx, int32_t* rank, int32_t* world_size);
/* parts[r] goes to rank r; `out` = concatenation (in rank order) of what every rank sent to us.    */
int flockgpu_all_to_all(flockgpu_ctx* ctx, flockgpu_table* const* parts, int32_t n_parts,
                        flockgpu_table** out);
/* RepartitionExec(Hash(keys, world_size)) fused with the exchange: the partition kernel stores every row straight
 * into the receiving rank's window over NVLink peer memory (CUDA IPC; no NCCL call on the data path).  The result
 * holds, in source-rank order, the rows every rank routed here; inside one source the input order is kept.           */
int flockgpu_hash_exchange(flockgpu_ctx* ctx, const flockgpu_table* in, const int32_t* key_cols,
                           int32_t n_keys, flockgpu_table** out);

/* ---- ExecutionContext: the caller-facing surface (flock/src/runtime/context.rs) ----------------
 * `flock_context` mirrors flock::runtime::context::ExecutionContext { plan, name, next, .. }:
 * it owns one or more physical plans deserialised from the reference's own serde-JSON plan format
 * (the string `marshal` puts into the Lambda environment, context.rs:366-381, Encoding::None) and
 * executes them on the GPU.                                                                        */
typedef struct flock_context flock_context;
/* plans_json: either one plan object {"execution_plan": ...}, an array of them, or an
 * ExecutionContext object {"plan": {"execution_plans": [...]}, "name": ...}.                        */
int flock_context_unmarshal(flockgpu_ctx* ctx, const char* plans_json, flock_context** out);
int flock_context_free(flock_context* ec);
int32_t flock_context_num_plans(const flock_context* ec);
/* ExecutionContext::feed_data_sources (context.rs:257-325): sources[i] is one relation given as
 * n_batches[i] record batches of schemas[i]; leaves are matched by field-name sub/superset
 * (compare_schema, context.rs:402-416), unmatched leaves get empty input.                          */
int flock_context_feed_data_sources(flock_context* ec, const struct ArrowSchema* const* schemas,
                                    const struct ArrowArray* const* const* batches,
                                    const int32_t* n_batches, int32_t n_sources);
/* Same, with relations already resident in HBM (bench.py's device-resident leg).                   */
int flock_context_feed_tables(flock_context* ec, flockgpu_table* const* tables, int32_t n_sources);
/* ExecutionContext::execute (context.rs:172-191): runs plan `plan_index`, result stays in HBM.     */
int flock_context_execute(flock_context* ec, int32_t plan_index, flockgpu_table** out);
/* ExecutionContext::execute_partitioned (context.rs:197-216): one table per output partition.
 * `out_parts` has room for `max_parts` entries; *n_parts receives the count.                       */
int flock_context_execute_partitioned(flock_context* ec, int32_t plan_index,
                                      flockgpu_table** out_parts, int32_t max_parts,
                                      int32_t* n_parts);
/* ExecutionContext::clean_data_sources (context.rs:227-254).                                       */
int flock_context_clean_data_sources(flock_context* ec);
/* ExecutionContext::is_shuffling (context.rs:328-337).                                             */
int flock_context_is_shuffling(const flock_context* ec, int32_t* out);
/* Indented plan rendering after the GPU rewrite, like `displayable(plan).indent()`; the returned
 * string is owned by the context and valid until the next call.                                    */
const char* flock_context_plan_str(flock_context* ec, int32_t plan_index);

/* ---- self tests of the expression compiler (NOT an execution path) ------------------------------
 * Run one predicate / value expression over a HOST record batch with the kernels' own term/chain
 * interpreter compiled for the host, so that CPU-only CI can check how DataFusion expressions are
 * lowered.  No operator or plan node ever calls these.                                             */
int flockgpu_selftest_eval_predicate(const struct ArrowSchema* schema, const struct ArrowArray* batch,
                                     const flockgpu_expr* predicate, uint8_t* out_mask,
                                     int32_t* out_fast_kind);
int flockgpu_selftest_eval_value(const struct ArrowSchema* schema, const struct ArrowArray* batch,
                                 const flockgpu_expr* expr, void* out, int32_t* out_dtype,
                                 int32_t* out_passthrough);
/* CPU-only: the arithmetic of the vectorised filter predicate CAST(x AS Int64) [% modulus] cmp rhs (modulus 0 = no `%`),
 * with the constants and the per-row test the GPU kernel uses (flock_b200/csrc/pred_i32.h).  out_keep[i] in {0, 1}. */
int flockgpu_selftest_pred_i32(int64_t modulus, int32_t cmp, int64_t rhs, const int32_t* x, int64_t n, uint8_t* out_keep, int32_t* out_mode);

#ifdef __cplusplus
}
#endif
#endif /* FLOCKGPU_H */
