// internal.h -- host-side C++ types shared by every translation unit of libflockgpu.
//
// Nothing here is part of the ABI (include/flockgpu.h is).  Data model:
//   Ctx      one CUDA device + stream + stream-ordered memory pool + scratch state
//   Buffer   a reference-counted HBM allocation (freed stream-ordered when the last owner drops it)
//   Column   one Arrow column resident in HBM: fixed-width values, or Utf8 = int32 offsets + bytes
//   Table    an immutable relation = columns of equal length (the device form of Vec<RecordBatch>)
#pragma once

#include <cuda_runtime.h>

#include <atomic>
#include <condition_variable>
#include <cstdint>
#include <functional>
#include <thread>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/flockgpu.h"

namespace fg {

// ------------------------------------------------------------------------------------------------
// errors: thrown inside the library, converted to return codes at the extern "C" boundary
// ------------------------------------------------------------------------------------------------
struct Error {
  int code;
  std::string msg;
};
[[noreturn]] void fail(int code, const char* fmt, ...) __attribute__((format(printf, 2, 3)));
void set_last_error(const std::string& msg);

#define FG_CUDA(expr)                                                                          \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess)                                                                     \
      ::fg::fail(FLOCKGPU_ERR_CUDA, "%s:%d: %s -> %s", __FILE__, __LINE__, #expr,              \
                 cudaGetErrorString(_e));                                                      \
  } while (0)

#define FG_CHECK(cond, code, ...)                 \
  do {                                            \
    if (!(cond)) ::fg::fail((code), __VA_ARGS__); \
  } while (0)

// Runs `body` and maps fg::Error / std::exception to an ABI return code.
template <typename F>
int guarded(F&& body) noexcept {
  try {
    body();
    return FLOCKGPU_OK;
  } catch (const Error& e) {
    set_last_error(e.msg);
    return e.code;
  } catch (const std::exception& e) {
    set_last_error(std::string("internal error: ") + e.what());
    return FLOCKGPU_ERR_INVALID;
  } catch (...) {
    set_last_error("internal error: unknown exception");
    return FLOCKGPU_ERR_INVALID;
  }
}

// ------------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------------
struct Comm;  // comm.cc

// Scratch of the single-pass compaction / scan kernels (compact.cuh).  Never reset between launches: tickets are a
// monotonic counter whose base the host tracks, status words carry the launch epoch.
struct ScanScratch {
  unsigned long long* ep_state = nullptr;    // [ep_capacity * stride] {epoch:20, flag:2, value:42}
  unsigned long long* ep_counts = nullptr;   // [ep_capacity] dense epoch-tagged per-tile counts (single-wave mode)
  unsigned* ep_counters = nullptr;           // [0] tickets issued, [1] tiles arrived
  int64_t ep_capacity = 0;
  unsigned tickets_issued = 0, arrived = 0, epoch = 0;
};

// Host threads that stage pageable batch buffers into page-locked memory (core.cu: import_batches).  Kept alive
// between feeds: creating eight threads costs more than copying their share of a 10 M-row relation.
struct StagePool {
  std::vector<std::thread> threads;
  std::mutex mu;
  std::condition_variable wake, idle;
  const std::function<void()>* job = nullptr;
  uint64_t generation = 0;
  int active = 0, running = 0;
  bool stop = false;
  void start(int n, const std::function<void()>* fn);  // the first n workers run *fn once
  void wait();                                         // until all of them have returned
  ~StagePool();
};

struct CtxCore {
  int device = 0;
  cudaStream_t stream = nullptr;
  // H2D fan-out (import_batches): one 256 KB copy per record batch and column leaves ~4 us of dead time between
  // dependent copies on ONE stream (28 GB/s measured); dealt over several streams they overlap and fill the link.
  static constexpr int kCopyStreams = 4;
  cudaStream_t copy_streams[kCopyStreams] = {};
  cudaEvent_t copy_fork = nullptr, copy_join[kCopyStreams] = {};
  cudaMemPool_t pool = nullptr;
  // Freed device blocks by rounded size.  cudaMallocAsync on the stream-ordered pool was measured at 0.5 us most of the
  // time and 1-100 ms every so often (profiles/r2_q5_host_trace_run6.txt: 454 ms in 353 calls), which no 0.1 ms query
  // survives; every kernel of a context runs on ONE stream, so a block released by its last owner can be handed to
  // the next operator at once -- stream order does the rest.  Blocks go back to CUDA when the context closes (or
  // when a fresh allocation fails).
  StagePool stage_pool;
  std::mutex block_mu;
  std::unordered_map<size_t, std::vector<void*>> free_blocks;
  size_t cached_bytes = 0;
  void* take_block(size_t rounded);
  void give_block(void* p, size_t rounded);
  void drop_cached_blocks();
  int sm_count = 148;
  std::recursive_mutex mu;

  // small pinned buffer for device->host scalar read-backs and device scalars
  // d_scalars[0, kScalars): counters / totals written by kernels; read_scalars() mirrors a range into h_scalars at the
  // same indices.  h_scalars[kScalars, kScalars + kPendingSlots): the pinned row-count slots of PendingRows.
  static constexpr int kScalars = 512;
  unsigned long long* h_scalars = nullptr;  // pinned, kScalars + kPendingSlots x u64
  unsigned long long* d_scalars = nullptr;  // device, kScalars x u64

  ScanScratch scan;
  void* l2_flush = nullptr;
  size_t l2_flush_bytes = 0;

  cudaEvent_t timer_start[16] = {};
  cudaEvent_t timer_stop[16] = {};
  std::atomic<int64_t> launches{0};
  // bytes that crossed the host link on behalf of this context (flockgpu_bytes_moved): copies issued by import /
  // export plus what kernels read in place from page-locked batches (zero-copy feed)
  std::atomic<int64_t> h2d_bytes{0}, d2h_bytes{0};

  // pinned host blocks handed out by flockgpu_host_alloc and by table export
  std::mutex pin_mu;
  std::unordered_map<void*, size_t> pinned;
  // flockgpu_host_alloc sub-allocates from page-locked SLABS: record batches allocated one after the other end up
  // contiguous in one large registration (few, large GPU mappings) instead of thousands of 256 KB registrations --
  // the in-place PCIe read of such batches measured 40.6 GB/s over 153 separate allocations against 51.1 GB/s over
  // one 40 MB allocation (profiles/r1_microbench_pcie_run17.txt).
  struct PinSlab {
    char* base = nullptr;
    size_t size = 0, used = 0;
    int64_t live = 0;
  };
  static constexpr size_t kPinSlabBytes = size_t(64) << 20;
  std::vector<PinSlab> pin_slabs;
  std::unordered_map<void*, size_t> pin_owner;  // allocation -> slab index

  std::shared_ptr<Comm> comm;  // comm.cc (shared_ptr: Comm is incomplete here)

  // row counts still in flight (see PendingRows): pinned slots h_scalars[kScalars + i]
  static constexpr int kPendingSlots = 256;
  std::weak_ptr<struct PendingRows> pending_owner[kPendingSlots];
  int pending_next = 0;

  // per-kernel CUDA-event profile (flockgpu_profile_begin / _end; bench.py's roofline numerator)
  bool profiling = false;
  struct ProfiledLaunch {
    const char* kernel;
    cudaEvent_t start, stop;
  };
  std::vector<ProfiledLaunch> profile;

  // feed_data_sources keeps page-locked, uniformly batched fixed-width columns in host memory (flockgpu_set_option)
  bool feed_zero_copy = false;
  // with feed_zero_copy: page-lock ordinary (pageable) batch buffers in place at feed time (cudaHostRegister) and
  // release them when the fed relation is dropped -- for callers whose Arrow allocator cannot be hooked
  bool feed_register = false;
  // pageable sources of a copy feed are staged into a page-locked block by this many host threads, each issuing the
  // DMA of a batch as soon as it has copied it (0: hand the pageable pointer to cudaMemcpyAsync)
  int feed_stream_stores = 1;  // non-temporal stores into the staging ring (host/stream_copy.cpp); 0: memcpy
  int feed_stage_threads = 8;  // run 27: 3.08 ms per 80 MB feed at 8 threads, 3.40 at 4, 4.4-5.7 at 16-32 (profiles/r2_feed_threads_run27.txt)
  // grid-wide prefix protocol of the compaction kernels: 0 = automatic (single wave when every tile is resident,
  // decoupled look-back otherwise), 1 = always decoupled look-back (flockgpu_set_option "compact_mode"; the parity
  // tests run both)
  int compact_mode = 0;
  // size of this rank's NVLink receive window (exchange.cu), fixed when the communicator is attached
  int64_t exchange_window_mb = 4096;

  // recycled CUDA events (creating one costs about a microsecond; a q2 step is one ~10 us kernel)
  std::vector<cudaEvent_t> sync_events;    // cudaEventDisableTiming
  std::vector<cudaEvent_t> timing_events;
  cudaEvent_t get_event(bool timing);
  void put_event(cudaEvent_t e, bool timing) { (timing ? timing_events : sync_events).push_back(e); }

  ~CtxCore();
};
using CtxPtr = std::shared_ptr<CtxCore>;

// Host-side wall time per named span, accumulated process-wide when FLOCKGPU_HOST_TRACE is set and printed to stderr
// by flockgpu_close (where does a 0.3 ms step spend its host time: allocation, waits, launches?).
struct HostSpan {
  const char* name;
  long long t0;
  explicit HostSpan(const char* n);
  ~HostSpan();
};
void host_trace_dump(bool reset);

// RAII: when profiling is on, brackets ONE kernel launch with events on the context stream.
struct LaunchTimer {
  CtxCore* ctx;
  cudaEvent_t stop = nullptr;
  LaunchTimer(const CtxPtr& c, const char* kernel);
  ~LaunchTimer();
};

// A survivor count that a kernel is still producing.  The operator enqueues an async copy of the device
// counter into a pinned slot and returns at once; the first consumer that needs the number waits.
struct PendingRows {
  CtxPtr ctx;
  int slot = 0;
  int64_t h2d_bytes_per_row = 0;  // zero-copy feed: bytes a survivor's pass-through values cost on the host link
  cudaEvent_t ev = nullptr;
  bool done = false;
  int64_t value = 0;
  int64_t wait();
  unsigned long long* host_slot() const;  // pinned (device-accessible) slot the count lands in
  ~PendingRows();
};
// reserve a pinned host slot (the compaction kernel stores the count there itself: CompactScratch::host_count),
// launch, then commit (records the event wait() blocks on)
std::shared_ptr<PendingRows> reserve_row_count(const CtxPtr& ctx);
void commit_row_count(const std::shared_ptr<PendingRows>& p);

struct Buffer {
  CtxPtr ctx;
  void* ptr = nullptr;
  size_t bytes = 0;
  size_t block_bytes = 0;  // size class of an owned block (CtxCore::take_block)
  // A VIEW (a slice of another allocation: one partition of a partition-ordered relation, a column inside a
  // peer-exchange window) keeps its owner alive through `parent` and frees nothing itself.
  std::shared_ptr<const void> parent;
  Buffer(CtxPtr c, size_t n);
  Buffer(CtxPtr c, void* p, size_t n, std::shared_ptr<const void> owner) : ctx(std::move(c)), ptr(p), bytes(n), parent(std::move(owner)) {}
  ~Buffer();
  Buffer(const Buffer&) = delete;
  Buffer& operator=(const Buffer&) = delete;
  template <typename T>
  T* as() const {
    return static_cast<T*>(ptr);
  }
};
using BufferPtr = std::shared_ptr<Buffer>;
BufferPtr alloc(const CtxPtr& ctx, size_t bytes);  // bytes == 0 still yields a valid (tiny) buffer
// `bytes` bytes of `b` starting at byte `off`; the caller keeps `off` 16-byte aligned when vector loads will read it
inline BufferPtr view_of(const BufferPtr& b, size_t off, size_t bytes) {
  return std::make_shared<Buffer>(b->ctx, static_cast<char*>(b->ptr) + off, bytes, std::static_pointer_cast<const void>(b));
}

// Grid-prefix tuning (FLOCKGPU_LB_STRIDE / FLOCKGPU_LB_SLEEP override): 64-bit words between the look-back words of
// consecutive tiles (32 = one 256-byte L2 chunk each), back-off of a polling thread in ns.
int scan_stride();
int scan_poll_sleep_ns();
// CTAs of `kernel` (block size `threads`, `smem` dynamic shared bytes) that fit on the context's device at once.  The
// occupancy query costs microseconds per call and most kernels here run ~10 us, so the answer is cached per
// (device, kernel, smem): processes that drive unlike GPUs get the right value for each.
int resident_ctas(const CtxPtr& ctx, const void* kernel, int threads, size_t smem = 0);
// Host copy into memory a device reads next (host/stream_copy.cpp).
void stage_copy(void* dst, const void* src, size_t n, int streaming);
// Copies `n` u64 scalars from d_scalars[first..] to the host and waits.
void read_scalars(const CtxPtr& ctx, int first, int n, unsigned long long* out);

// ------------------------------------------------------------------------------------------------
// columns and tables
// ------------------------------------------------------------------------------------------------
int dtype_width(int dtype);                 // bytes per value; 0 for Utf8
const char* dtype_name(int dtype);
int dtype_from_format(const char* format);  // -1 if unsupported
std::string default_format(int dtype);

// A fixed-width column that still lives in page-locked HOST memory, one chunk per fed record batch.  The filter
// kernel reads such a column straight over PCIe (UVA), so a q2 invocation moves each input byte once and never
// stages the relation in HBM; every other operator materialises it first (Table::dense()).
// Host ranges this library page-locked on behalf of a fed relation (feed_register); released with the last column.
struct HostRegistration {
  std::vector<std::pair<void*, size_t>> ranges;
  ~HostRegistration();
};

struct HostChunks {
  std::shared_ptr<HostRegistration> registration;  // keeps cudaHostRegister'ed sources locked while the column lives
  BufferPtr table;                // device array of chunk base pointers (device-accessible host addresses)
  std::vector<const void*> ptrs;  // the same pointers on the host
  std::vector<int64_t> rows;      // rows per chunk
  int shift = 16;                 // rows per chunk = 1 << shift for every chunk but the last
};

struct Column {
  int dtype = FLOCKGPU_INT32;
  std::string name;
  std::string format;  // Arrow C format string ("i", "tsm:", "u", ...)
  bool nullable = false;
  int64_t length = 0;
  BufferPtr data;      // fixed width: values; Utf8: value bytes (NULL while `chunks` is set)
  std::shared_ptr<HostChunks> chunks;  // host-resident form (zero-copy feed); see HostChunks
  BufferPtr offsets;   // Utf8 only: int32[length + 1]; offsets[0] may be > 0
  int64_t values_bytes = 0;  // Utf8: number of value bytes addressed by offsets
  // The one-row result of a global aggregate over empty input is NULL as a whole (SURVEY App. C.7).
  bool all_null = false;
  // Row-wise NULLs: one byte per row, 1 = valid; no buffer = no NULL in the column.  (Arrow's bit-packed bitmap is
  // expanded at import and packed again at export: every kernel that moves rows moves these bytes like one more
  // 1-byte column.)
  BufferPtr validity;
  const uint8_t* valid() const { return validity ? validity->as<uint8_t>() : nullptr; }

  const void* values() const { return data ? data->ptr : nullptr; }
  const int32_t* offs() const { return offsets ? offsets->as<int32_t>() : nullptr; }
  int width() const { return dtype_width(dtype); }
};

struct Table;
using TablePtr = std::shared_ptr<const Table>;

// A relation whose rows have not been written out yet: a group-by result that still lives in its direct-address
// table (hash_agg.cu).  Table::resolve() materialises it; the operators that can work on the table form directly
// (NEXMark q5: MAX over the counts, then "count = max") ask for that instead and never pay for the 78 MB of
// (auction, count) rows that the plan would otherwise write and read twice.
struct DeferredTable {
  virtual ~DeferredTable() = default;
  virtual void materialise(const Table& self) = 0;  // fills self.cols / self.num_rows
  // Fast paths: each returns nullptr when it does not apply (the caller then resolves and takes the generic path).
  // `out = SELECT self.src_cols AS names`:
  virtual TablePtr project(const Table& self, const std::vector<int>& src_cols, const std::vector<std::string>& names) { return nullptr; }
  // one-row relation MAX(self.col) (mode: FLOCKGPU_AGG_PARTIAL state or a final value -- the same number):
  virtual TablePtr global_max(const Table& self, int col, const std::string& out_name) { return nullptr; }
  // self JOIN one_row ON self.key_col = one_row.one_key, output columns self ++ one_row (or the reverse):
  virtual TablePtr select_equal(const Table& self, int key_col, const TablePtr& one_row, int one_key, bool self_is_left) { return nullptr; }
};

struct Table {
  CtxPtr ctx;
  // `cols[i].length` and `num_rows` are -1 while `pending` is set (a filter's survivor count that has not
  // been read back yet); resolve() waits for it and fills them in.  Every operator resolves its inputs.
  mutable std::vector<Column> cols;
  mutable int64_t num_rows = 0;
  mutable std::shared_ptr<PendingRows> pending;
  mutable std::shared_ptr<DeferredTable> deferred;  // see DeferredTable; cols carry names / types only until resolved
  std::string metadata;  // raw Arrow schema metadata block (may be empty)
  // Set on the output of a multi-GPU hash exchange: the NAMES of the columns whose values routed the rows (the
  // routing function of partition.cu over exactly these columns, `partition_world` ranks).  Operators that keep those
  // columns under the same names hand the property on; a later RepartitionExec(Hash) over the same routing columns
  // finds its input already in place and moves nothing (q8 plans Hash([p_id, name]) and then Hash([p_id])).
  std::vector<std::string> partitioned_on;
  int partition_world = 0;
  int64_t nbytes() const;
  void resolve() const {
    if (deferred) {
      std::shared_ptr<DeferredTable> d = deferred;
      d->materialise(*this);
      deferred.reset();
    }
    if (!pending) return;
    num_rows = pending->wait();
    for (Column& c : cols) c.length = num_rows;
    pending.reset();
  }
  // resolve() + copy host-resident columns into HBM (every operator except the vectorised filter needs this)
  void dense() const;
  bool has_host_columns() const {
    for (const Column& c : cols)
      if (c.chunks) return true;
    return false;
  }
};

}  // namespace fg

// ABI handles ------------------------------------------------------------------------------------
struct flockgpu_ctx {
  fg::CtxPtr core;
};
struct flockgpu_table {
  fg::TablePtr table;
  std::atomic<int> refs{1};
};

namespace fg {
flockgpu_table* wrap_table(TablePtr t);
inline const Table& deref(const flockgpu_table* t) {
  if (!t || !t->table) fail(FLOCKGPU_ERR_INVALID, "null table handle");
  t->table->resolve();
  return *t->table;
}
inline CtxPtr core_of(flockgpu_ctx* c) {
  if (!c || !c->core) fail(FLOCKGPU_ERR_INVALID, "null context handle");
  return c->core;
}

// Operators that do not implement NULL semantics for some input refuse it (FLOCKGPU_ERR_UNSUPPORTED): the Rust shim then
// keeps the CPU plan for that data.  Never a silent wrong answer.
inline void require_no_nulls(const Column& c, const char* what) {
  if (c.validity) fail(FLOCKGPU_ERR_UNSUPPORTED, "%s: column \"%s\" contains NULLs, which this operator does not handle on the GPU path", what, c.name.c_str());
}

// ---- operators (implemented in the .cu files; called by the ABI layer and by the plan layer) ----
struct ExprTok {
  int op, dtype, col;
  int64_t i64;
  double f64;
  std::string str;
};
using Expr = std::vector<ExprTok>;  // postfix

TablePtr import_batches(const CtxPtr& ctx, const ArrowSchema* schema, const ArrowArray* const* batches,
                        int n_batches, const int* projection, int n_projection, bool zero_copy = false);
void export_table(const CtxPtr& ctx, const Table& t, int64_t row_begin, int64_t row_count,
                  ArrowSchema* out_schema, ArrowArray* out_array);
void export_schema(const Table& t, ArrowSchema* out_schema);
TablePtr concat_tables(const CtxPtr& ctx, const std::vector<TablePtr>& tables);
TablePtr empty_like(const CtxPtr& ctx, const Table& t);

TablePtr filter_project(const CtxPtr& ctx, const TablePtr& in, const Expr* predicate,
                        const std::vector<Expr>& projections, const std::vector<std::string>& names);

struct AggSpec {
  int func;
  int col;
  std::string name;
};
TablePtr hash_aggregate(const CtxPtr& ctx, const TablePtr& in, int mode, const std::vector<int>& group_cols,
                        const std::vector<AggSpec>& aggs);
// Estimate from the first 64 Ki rows: fraction of rows that repeat an earlier group key (hash_agg.cu).
double distinct_sample_duplicates(const CtxPtr& ctx, const TablePtr& in, const std::vector<int>& group_cols);
TablePtr hash_join(const CtxPtr& ctx, const TablePtr& left, const TablePtr& right,
                   const std::vector<int>& left_keys, const std::vector<int>& right_keys,
                   int join_type = FLOCKGPU_JOIN_INNER);
std::vector<TablePtr> hash_partition(const CtxPtr& ctx, const TablePtr& in, const std::vector<int>& keys,
                                     int n_parts);
// The columns of `keys` that actually route a row: the fixed-width ones when there are any (hashing `p_id` routes
// (p_id, name) groups just as well as hashing the name bytes too, and lets a later Hash([p_id]) stay in place).
std::vector<int> routing_columns(const Table& in, const std::vector<int>& keys);
// RepartitionExec(Hash(keys, world)) + the inter-GPU shuffle in one step (exchange.cu): rows travel straight from the
// partition kernel into the receivers' windows over NVLink peer memory; `dest` >= 0 sends every row to that rank
// instead (CoalescePartitionsExec).  Falls back to hash_partition + the NCCL all-to-all when peer windows are
// unavailable.
TablePtr hash_exchange(const CtxPtr& ctx, const TablePtr& in, const std::vector<int>& keys, int dest = -1);
// SortExec / WindowAggExec(ROW_NUMBER) / GlobalLimitExec (sort.cu)
struct SortKey {
  int col;
  bool descending;
  bool nulls_first;  // no effect: columns with NULLs are not sortable on the GPU path
};
TablePtr sort_table(const CtxPtr& ctx, const TablePtr& in, const std::vector<SortKey>& keys);
TablePtr row_number(const CtxPtr& ctx, const TablePtr& in, const std::vector<int>& partition_cols, const std::string& name);
TablePtr limit_rows(const CtxPtr& ctx, const TablePtr& in, int64_t limit);
// Row gather: out.col[c][i] = in.col[c][idx[i]] for every column (fixed width and Utf8).
TablePtr gather_rows(const CtxPtr& ctx, const Table& in, const std::vector<int>& cols, const uint32_t* d_idx,
                     int64_t n_idx);
// Gathers single columns (used by filter for Utf8 pass-through and by join).
Column gather_column(const CtxPtr& ctx, const Column& in, const uint32_t* d_idx, int64_t n_idx);
// `pad`: d_idx may hold the pad sentinel ~0u (the unmatched rows of an outer join): such a row is NULL -- value 0,
// Utf8 length 0, validity 0 -- and every output column carries validity bytes.
std::vector<Column> gather_columns(const CtxPtr& ctx, const std::vector<const Column*>& in, const uint32_t* d_idx, int64_t n, bool pad = false);
// `n` rows of NULL in the columns of `t` (validity 0, values 0, Utf8 empty), marked nullable: the padded side of an
// outer join whose other side found no partner at all.
std::vector<Column> null_columns(const CtxPtr& ctx, const Table& t, int64_t n);

TablePtr all_to_all(const CtxPtr& ctx, const std::vector<TablePtr>& parts);
void comm_unique_id(uint8_t* out);
void comm_init(const CtxPtr& ctx, const uint8_t* id, int rank, int world);
int comm_world(const CtxPtr& ctx);  // 1 when no communicator is attached
int comm_rank(const CtxPtr& ctx);   // 0 when no communicator is attached

inline void count_launch(const CtxPtr& ctx, int n = 1) { ctx->launches.fetch_add(n, std::memory_order_relaxed); }

}  // namespace fg
