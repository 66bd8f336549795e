// libb200exec host side: the GPU ExecutionEngine / QueryStageExecutor.
//
// Mirrors (reference file:line):
//   DefaultExecutionEngine::create_query_stage_exec     ballista/executor/src/execution_engine.rs:106-169
//   DefaultQueryStageExec::execute_query_stage          ballista/executor/src/execution_engine.rs:235-254
//   ShuffleWriterExec::execute_shuffle_write            ballista/core/src/execution_plans/shuffle_writer.rs:203-402
//   SortShuffleWriterExec::execute_shuffle_write        ballista/core/src/execution_plans/sort_shuffle/writer.rs:199-373
//   ShuffleReaderExec::execute                          ballista/core/src/execution_plans/shuffle_reader.rs:248-318
//   collect_plan_metrics                                ballista/core/src/utils.rs:328-339
// The operator tree below the writer (FilterExec/ProjectionExec/AggregateExec/HashJoinExec/SortExec,
// DataFusion 53.1 [EXT]) is executed by the CUDA kernels in csrc/device.  There is no CPU path:
// every operator either runs on the GPU or fails with B200_ERR_UNSUPPORTED.
#include <sched.h>
#include <sys/stat.h>

#include <algorithm>
#include <atomic>
#include <cctype>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <map>
#include <mutex>
#include <functional>
#include <set>

#include "../common/arrow_host.hpp"
#include "../common/tpch_gen.hpp"
#include "../device/kernels.h"
#include "host_pool.hpp"
#include "lower.hpp"
#include "nccl_dyn.hpp"
#include "../common/plan_proto.hpp"
#include "../common/plan_dump.hpp"
#include "parquet_meta.hpp"
#include "arrow_ipc.hpp"

using namespace b200;

namespace {

thread_local std::string g_err;

struct Piece {
  int64_t file_id;
  DevBatchPtr batch;
  int64_t r0, r1;
  int32_t src_rank = 0;               // which executor's map task produced it (exchange)
  std::vector<int64_t> str_bytes;     // per Utf8 column of the batch: character bytes of rows [r0, r1); empty = unknown
};
struct ShuffleKey {
  std::string job;
  int64_t stage;
  int64_t part;
  bool operator<(const ShuffleKey& o) const {
    if (job != o.job) return job < o.job;
    if (stage != o.stage) return stage < o.stage;
    return part < o.part;
  }
};

struct OpMetrics {
  std::string name;
  uint64_t output_rows = 0, input_rows = 0, elapsed_ns = 0, bytes_read = 0, bytes_written = 0, launches = 0;
};

}  // namespace

struct b200_engine {
  int device = 0;
  int rank = 0, world = 1;
  int sm_count = 148;
  cudaStream_t own_stream = nullptr;
  cudaStream_t stream = nullptr;
  std::mutex mu;
  std::map<std::string, std::map<int, DevBatchPtr>> tables;
  std::map<ShuffleKey, std::vector<Piece>> shuffle;
  std::map<ShuffleKey, DevBatchPtr> packed_cache;  // b200_partition_device_buffers: exchange-layout copies handed out by pointer
  std::atomic<uint64_t> launches{0};
  std::atomic<uint64_t> n_fused{0}, n_fused_static{0}, n_vm{0}, n_groupby{0}, n_groupby_pf{0}, n_fastfilter{0};  // pipelines per kernel family (b200_engine_counter)
  int64_t batch_size = 8192;
  std::map<std::string, std::string> config;
  std::map<std::string, int> agg_hint;       // plan fingerprint -> sink that worked (0 reg, >0 log2 cap)
  uint64_t pf_bucket_slots = (uint64_t)1 << 19;  // partition-first aggregation: table slots per bucket (power of two; 0 = off)
  int64_t pf_min_rows = (int64_t)1 << 22;
  std::map<std::string, uint64_t> agg_groups;  // plan fingerprint -> most groups any task of that shape produced (sizes the table)
  std::map<std::string, uint64_t> agg_spec;    // plan fingerprint + input partition -> groups of its last run, when the hinted sink held them at once
  void* pinned_stage = nullptr;              // small pinned buffer for status read-backs
  // ingest narrowing (import_batch): host pool + two pinned staging slots with their device mirrors
  std::unique_ptr<HostPool> pool;
  std::mutex ingest_mu;                      // one narrowing pipeline at a time (pool and staging slots are shared)
  struct NarrowSlot {
    void* pinned = nullptr;
    void* dev = nullptr;
    cudaEvent_t done = nullptr;
    bool used = false;
    size_t bytes = 0;
  } nslot[4];
  int64_t ingest_chunk_rows = (int64_t)1 << 22;
  int ingest_slots = 3;
  // per-kernel device timing (b200.metrics.kernel_timing = on): CUDA event pairs on the launching stream, resolved
  // when the statistics are read (b200_engine_kernel_stats)
  bool kernel_timing = false;
  struct KernelSample { std::string name; cudaEvent_t e0, e1; uint64_t bytes; };
  std::vector<KernelSample> ksamples;
  struct KernelStat { double ms = 0; uint64_t launches = 0, bytes = 0; };
  std::map<std::string, KernelStat> kstats;
  ncclComm_t comm = nullptr;                 // exchange communicator (b200_engine_comm_init); nullptr = single executor
  std::mutex comm_mu;                        // one collective at a time
  uint64_t exch_sent_bytes = 0, exch_recv_bytes = 0;
  // fused shuffle (b200_stage_execute_exchange): one window of HBM per executor, mapped into every peer process through
  // CUDA IPC at b200_engine_comm_init, so the partition scatter kernel stores each row straight into the HBM of the executor
  // that owns its output partition (NVLink / NVSwitch peer stores) -- no staging copy, no separate transfer
  size_t win_config_bytes = 0;               // b200.exchange.window_bytes
  uint8_t* win_local = nullptr;
  size_t win_bytes = 0, win_used = 0;
  std::vector<uint8_t*> win_peer;            // [rank] -> this process's mapping of that rank's window (own rank: win_local)
  uint64_t fused_exchanges = 0;
  std::mutex export_mu;                      // small-result export arena (pinned), one export at a time
  uint8_t* export_arena = nullptr;
  std::atomic<uint64_t> narrowed_bytes_saved{0};         // PCIe bytes not sent thanks to narrowing (b200_engine_counter)
  std::atomic<uint64_t> stream_syncs{0};                 // host waits on the stream inside tasks and exports (b200_engine_counter)
  // parsed stage plans, keyed by stage id + plan text (job id taken out when the caller names the job): the same stage of
  // the next job is not parsed again.  The trees are shared read-only by every b200_stage prepared from them.
  struct CachedPlan { std::shared_ptr<const PlanNode> plan; uint64_t used; };
  std::map<std::string, CachedPlan> plan_cache;
  uint64_t plan_cache_tick = 0;
};
static const size_t PLAN_CACHE_ENTRIES = 32;

struct b200_stage {
  b200_engine* eng = nullptr;
  std::string job_id;
  int64_t stage_id = 0;
  std::shared_ptr<const PlanNode> plan;  // shared with the engine's plan cache: read-only; its job_id is not this stage's
  std::string fingerprint;
  std::vector<OpMetrics> metrics;  // pre-order
  std::map<const PlanNode*, int> metric_index;
};

#define NCCL_CHECK(expr)                                                                                              \
  do {                                                                                                                \
    ncclResult_t _r = (expr);                                                                                         \
    if (_r != 0) throw EngineError(B200_ERR_CUDA, std::string("NCCL error: ") + NcclApi::get().GetErrorString(_r) + " at " + __FILE__ + ":" + std::to_string(__LINE__)); \
  } while (0)

static void release_window(b200_engine* e);
static void setup_window(b200_engine* e);

namespace {

// ------------------------------------------------------------------------------------------------
// Small helpers
// ------------------------------------------------------------------------------------------------
// Per-thread read-back arena: scalars the host needs from the device (row counts, status words, string
// byte totals) are queued as asynchronous copies into one pinned buffer and become readable after the next
// Exec::sync().  Checks that only have to hold before the task RETURNS (arithmetic-overflow flags of kernels
// whose output size is already known) are deferred to that same synchronisation instead of costing their own.
struct TaskCtx {
  uint8_t* arena = nullptr;
  size_t pos = 0;
  bool drained = true;
  std::vector<std::function<void()>> checks;
};
static const size_t TASK_ARENA_BYTES = (size_t)1 << 16;
inline TaskCtx& task_ctx() {
  static thread_local TaskCtx t;
  if (!t.arena && cudaHostAlloc((void**)&t.arena, TASK_ARENA_BYTES, cudaHostAllocDefault) != cudaSuccess) t.arena = nullptr;
  return t;
}

// Thrown by a deferred check when a task that ran on a remembered aggregate group count finds the count (or the sink) was
// wrong: b200_stage_execute discards the task's outputs and runs it again without guessing.
struct SpeculationMiss {};

struct Exec {
  b200_engine* e;
  b200_stage* s;
  const volatile int32_t* cancel;
  bool speculate = false;  // aggregates may run on the group count of their last run (run_aggregate); only b200_stage_execute retries
  cudaStream_t st() const { return e->stream; }
  void check_cancel() const {
    if (cancel && *cancel) throw EngineError(B200_ERR_CANCELLED, "task cancelled");
  }
  void count(uint64_t n = 1) const { e->launches.fetch_add(n, std::memory_order_relaxed); }
  OpMetrics* m(const PlanNode* n) const {
    if (!s) return nullptr;
    auto it = s->metric_index.find(n);
    return it == s->metric_index.end() ? nullptr : &s->metrics[(size_t)it->second];
  }
  // queue a device->host copy of `bytes` bytes; the returned pointer is readable after sync()
  const void* fetch_bytes(const void* dptr, size_t bytes) const {
    TaskCtx& t = task_ctx();
    if (!t.arena) throw EngineError(B200_ERR_OOM, "pinned read-back arena unavailable");
    if (t.drained) {
      t.pos = 0;
      t.drained = false;
    }
    const size_t at = (t.pos + 15) & ~(size_t)15;
    if (at + bytes > TASK_ARENA_BYTES) {  // rare: flush what is queued, then start over
      sync();
      return fetch_bytes(dptr, bytes);
    }
    CUDA_CHECK(cudaMemcpyAsync(t.arena + at, dptr, bytes, cudaMemcpyDeviceToHost, st()));
    t.pos = at + bytes;
    return t.arena + at;
  }
  // pinned host scratch for an asynchronous host->device upload; valid until the next sync()
  void* stage_bytes(size_t bytes) const {
    TaskCtx& t = task_ctx();
    if (!t.arena) throw EngineError(B200_ERR_OOM, "pinned staging arena unavailable");
    if (t.drained) {
      t.pos = 0;
      t.drained = false;
    }
    size_t at = (t.pos + 15) & ~(size_t)15;
    if (at + bytes > TASK_ARENA_BYTES) {
      sync();
      t.pos = 0;
      t.drained = false;
      at = 0;
      if (bytes > TASK_ARENA_BYTES) throw EngineError(B200_ERR_INVALID, "staging request larger than the arena");
    }
    t.pos = at + bytes;
    return t.arena + at;
  }
  template <class T>
  const T* fetch(const void* dptr) const {
    return (const T*)fetch_bytes(dptr, sizeof(T));
  }
  void defer(std::function<void()> fn) const { task_ctx().checks.push_back(std::move(fn)); }
  // wait for everything enqueued so far, then run the deferred checks (they may throw)
  void sync() const {
    TaskCtx& t = task_ctx();
    e->stream_syncs++;
    cudaError_t se = cudaStreamSynchronize(st());
    t.drained = true;
    std::vector<std::function<void()>> cs;
    cs.swap(t.checks);
    CUDA_CHECK(se);
    for (auto& c : cs) c();
    check_cancel();
  }
  // wait for everything enqueued so far; deferred checks stay queued for the next sync()
  void wait() const {
    e->stream_syncs++;
    CUDA_CHECK(cudaStreamSynchronize(st()));
  }
  // drop deferred checks without running them (error unwinding)
  static void abandon() {
    TaskCtx& t = task_ctx();
    t.checks.clear();
    t.drained = true;
  }
  template <class T>
  T get(const void* dptr) const {
    const T* p = fetch<T>(dptr);
    sync();
    return *p;
  }
};

// Brackets one kernel (or one short sequence) with CUDA events when kernel timing is on; `bytes` = algorithmic bytes
// (SURVEY.md 8(d) formulas) so that achieved GB/s per kernel family can be reported next to the HBM roofline.
struct KernelTimer {
  b200_engine* e;
  cudaStream_t st;
  b200_engine::KernelSample ks;
  bool on;
  KernelTimer(const Exec& x, const char* name, uint64_t bytes) : e(x.e), st(x.st()), on(x.e->kernel_timing) {
    if (!on) return;
    ks.name = name;
    ks.bytes = bytes;
    if (cudaEventCreate(&ks.e0) != cudaSuccess || cudaEventCreate(&ks.e1) != cudaSuccess) {
      on = false;
      return;
    }
    cudaEventRecord(ks.e0, st);
  }
  ~KernelTimer() {
    if (!on) return;
    cudaEventRecord(ks.e1, st);
    std::lock_guard<std::mutex> g(e->mu);
    e->ksamples.push_back(ks);
  }
};

// B200_TIMING=1: host wall time of the phases of a task (diagnostic; stderr)
struct ScopeTimer {
  const char* name;
  std::chrono::steady_clock::time_point t0;
  bool on;
  explicit ScopeTimer(const char* n) : name(n) {
    static const bool enabled = getenv("B200_TIMING") != nullptr;
    on = enabled;
    if (on) t0 = std::chrono::steady_clock::now();
  }
  ~ScopeTimer() {
    if (on) fprintf(stderr, "[b200-time] %s host_ms=%.3f\n", name, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
  }
};

uint64_t next_pow2(uint64_t v) {
  uint64_t p = 1;
  while (p < v) p <<= 1;
  return p;
}

DevColumn make_out_column(const std::string& name, const DataType& t, Phys phys, int64_t cap, bool with_valid, cudaStream_t st) {
  DevColumn c;
  c.name = name;
  c.type = t;
  c.phys = phys;
  c.n = cap;
  DevPtr d = dev_alloc((size_t)std::max<int64_t>(cap, 1) * phys_width(phys), st);
  c.data = (const uint8_t*)d->ptr;
  c.keep.push_back(d);
  if (with_valid) {
    DevPtr v = dev_alloc((size_t)std::max<int64_t>(cap, 1), st);
    c.valid = (const uint8_t*)v->ptr;
    c.keep.push_back(v);
  }
  c.nullable = with_valid;
  return c;
}

// A batch of small copy / string-conversion jobs executed by ONE kernel (shuffle.cu pack_jobs_kernel): the tail of
// a query moves a handful of rows through a dozen columns and is bound by launch count, not bytes.
struct PackList {
  std::vector<PackJob> jobs;
  void copy(const void* src, void* dst, uint64_t bytes) {
    if (!bytes) return;
    PackJob j;
    memset(&j, 0, sizeof j);
    j.kind = PK_COPY;
    j.src = src;
    j.dst = dst;
    j.bytes = bytes;
    jobs.push_back(j);
  }
  // string column slice (views or Arrow offsets positioned at the first row) -> offsets (rows + 1, from 0) + chars
  void bitmap(const uint8_t* bytes, int64_t rows, void* bitmap_out, void* zero_count_out) {
    PackJob j;
    memset(&j, 0, sizeof j);
    j.kind = PK_BITMAP;
    j.src = bytes;
    j.dst = bitmap_out;
    j.dst2 = zero_count_out;
    j.rows = rows;
    jobs.push_back(j);
  }
  // Arrow Utf8 slice -> views written at `views_out` (rows x 16 bytes)
  void utf8_views(const DevColumn& c, void* views_out) {
    PackJob j;
    memset(&j, 0, sizeof j);
    j.kind = PK_UTF8_VIEWS;
    j.src = c.data;
    j.chars = c.chars;
    j.dst = views_out;
    j.rows = c.n;
    jobs.push_back(j);
  }
  void strings(const DevColumn& c, void* offsets_out, void* chars_out, uint64_t chars_cap = ~0ull) {
    PackJob j;
    memset(&j, 0, sizeof j);
    j.bytes = chars_cap;
    j.kind = c.phys == PH_STRVIEW ? PK_STR_VIEWS : PK_STR_UTF8;
    j.src = c.data;
    j.valid = c.valid;
    j.chars = c.chars;
    j.dst = offsets_out;
    j.dst2 = chars_out;
    j.rows = c.n;
    jobs.push_back(j);
  }
  void run(const Exec& x, std::vector<DevPtr>* keep = nullptr) {
    if (jobs.empty()) return;
    const size_t bytes = jobs.size() * sizeof(PackJob);
    DevPtr d = dev_alloc(bytes, x.st());
    if (bytes <= TASK_ARENA_BYTES / 4) {
      void* h = x.stage_bytes(bytes);
      memcpy(h, jobs.data(), bytes);
      CUDA_CHECK(cudaMemcpyAsync(d->ptr, h, bytes, cudaMemcpyHostToDevice, x.st()));
    } else {
      CUDA_CHECK(cudaMemcpyAsync(d->ptr, jobs.data(), bytes, cudaMemcpyHostToDevice, x.st()));  // pageable: staged by the driver before returning
    }
    launch_pack_jobs((const PackJob*)d->ptr, (int)jobs.size(), x.st());
    x.count();
    if (keep) keep->push_back(d);
    jobs.clear();
  }
};

// strings as views (needed for gather / scatter / sort / join); zero-copy for non-strings
DevColumn as_views(const Exec& x, const DevColumn& c) {
  if (c.phys != PH_UTF8) return c;
  DevColumn o = c;
  DevPtr v = dev_alloc((size_t)std::max<int64_t>(c.n, 1) * 16, x.st());
  launch_utf8_to_views((const int32_t*)c.data, c.chars, (unsigned long long*)v->ptr, c.n, x.st());
  x.count();
  o.phys = PH_STRVIEW;
  o.data = (const uint8_t*)v->ptr;
  o.chars = nullptr;
  o.keep.push_back(v);
  return o;
}

// views -> Arrow Utf8 (offsets + chars), contiguous
DevColumn as_utf8(const Exec& x, const DevColumn& c, int64_t known_total = -1) {
  if (c.phys != PH_STRVIEW) return c;
  const int64_t n = c.n;
  if (known_total >= 0 && n <= 4096) {
    // small column whose character count the host already knows: offsets + chars in ONE launch, no read-back
    DevPtr offsets = dev_alloc((size_t)(n + 1) * 4, x.st());
    DevPtr chars = dev_alloc((size_t)known_total + 16, x.st());
    PackList pl;
    pl.strings(c, offsets->ptr, chars->ptr);
    pl.run(x);
    DevColumn o;
    o.name = c.name;
    o.type = c.type;
    o.nullable = c.nullable;
    o.phys = PH_UTF8;
    o.n = n;
    o.data = (const uint8_t*)offsets->ptr;
    o.chars = (const uint8_t*)chars->ptr;
    o.chars_bytes = known_total;
    o.valid = c.valid;
    o.keep.push_back(offsets);
    o.keep.push_back(chars);
    if (c.valid)
      for (auto& k : c.keep) o.keep.push_back(k);
    return o;
  }
  DevPtr lens = dev_alloc((size_t)(n + 1) * 4, x.st());
  DevPtr offs64 = dev_alloc((size_t)(n + 2) * 8, x.st());
  DevPtr scratch = dev_alloc((size_t)(n / 1024 + 4) * 8, x.st());
  launch_view_lengths((const unsigned long long*)c.data, c.valid, (uint32_t*)lens->ptr, n, x.st());
  launch_scan_u32_to_u64((const uint32_t*)lens->ptr, (uint64_t*)offs64->ptr, n, (uint64_t*)scratch->ptr, x.st());
  x.count(4);
  uint64_t total = known_total >= 0 ? (uint64_t)known_total : x.get<uint64_t>((const uint64_t*)offs64->ptr + n);
  if (total > 0x7FFFFFFFull) throw EngineError(B200_ERR_UNSUPPORTED, "string column exceeds 2 GiB (LargeUtf8 not supported)");
  DevPtr offsets = dev_alloc((size_t)(n + 1) * 4, x.st());
  DevPtr chars = dev_alloc((size_t)total + 16, x.st());
  launch_views_to_utf8((const unsigned long long*)c.data, c.valid, (const uint64_t*)offs64->ptr, (int32_t*)offsets->ptr, (uint8_t*)chars->ptr, n, x.st());
  x.count();
  DevColumn o;
  o.name = c.name;
  o.type = c.type;
  o.nullable = c.nullable;
  o.phys = PH_UTF8;
  o.n = n;
  o.data = (const uint8_t*)offsets->ptr;
  o.chars = (const uint8_t*)chars->ptr;
  o.chars_bytes = (int64_t)total;
  o.valid = c.valid;
  o.keep.push_back(offsets);
  o.keep.push_back(chars);
  if (c.valid)
    for (auto& k : c.keep) o.keep.push_back(k);  // validity lives in the old allocations
  return o;
}

// Registered tables: every Utf8 column whose strings are all at most 3 bytes long (TPC-H flags, status, ...) gets a
// companion of 4-byte key images (len << 24 | bytes).  An aggregate that groups by such a column then streams 4 bytes per
// row through the same TMA ring as its other operands instead of gathering characters behind the offsets.
void prepack_short_strings(const Exec& x, DevBatch& b) {
  struct Cand { size_t col; DevPtr img, flag; const unsigned int* h; };
  std::vector<Cand> cands;
  for (size_t ci = 0; ci < b.cols.size(); ci++) {
    DevColumn& c = b.cols[ci];
    if (c.phys != PH_UTF8 || c.valid || c.pk32 || c.n == 0) continue;
    if (c.chars_bytes < 0 || c.chars_bytes > 3 * c.n) continue;  // some string must be longer
    Cand cd;
    cd.col = ci;
    cd.img = dev_alloc((size_t)c.n * 4 + 64, x.st());
    cd.flag = dev_alloc(16, x.st());
    CUDA_CHECK(cudaMemsetAsync(cd.flag->ptr, 0, 16, x.st()));
    launch_prepack3((const int32_t*)c.data, c.chars, c.n, (uint32_t*)cd.img->ptr, (unsigned int*)cd.flag->ptr, x.st());
    x.count();
    cd.h = x.fetch<unsigned int>(cd.flag->ptr);
    cands.push_back(cd);
  }
  if (cands.empty()) return;
  x.sync();
  for (auto& cd : cands) {
    if (*cd.h) continue;
    DevColumn& c = b.cols[cd.col];
    c.pk32 = (const uint32_t*)cd.img->ptr;
    c.keep.push_back(cd.img);
  }
}

DevBatchPtr gather_batch(const Exec& x, const DevBatch& in, const int64_t* idx, int64_t n_out, bool may_be_null) {
  auto out = std::make_shared<DevBatch>();
  out->n = n_out;
  GatherCols gc;
  gc.n = 0;
  auto flush = [&]() {
    if (gc.n) {
      uint64_t b = 8;
      for (int k = 0; k < gc.n; k++) b += 2ull * (uint64_t)gc.c[k].width;
      KernelTimer kt(x, "gather", (uint64_t)n_out * b);
      launch_gather_multi(gc, idx, n_out, x.st());
      x.count();
      gc.n = 0;
    }
  };
  for (auto& c0 : in.cols) {
    DevColumn c = as_views(x, c0);
    bool with_valid = c.valid != nullptr || may_be_null;
    DevColumn o = make_out_column(c.name, c.type, c.phys, n_out, with_valid, x.st());
    o.n = n_out;
    GatherCol& g = gc.c[gc.n++];
    g.in = c.data;
    g.valid_in = c.valid;
    g.out = (void*)o.data;
    g.valid_out = (uint8_t*)o.valid;
    g.width = c.width();
    if (gc.n == GATHER_MAX_COLS) flush();
    for (auto& k : c.keep) o.keep.push_back(k);
    out->cols.push_back(o);
  }
  flush();
  return out;
}

// ------------------------------------------------------------------------------------------------
// Arrow import (host -> HBM)
// ------------------------------------------------------------------------------------------------
// Decimal128 ingest with the sign-extension bytes squeezed out on the host (see host_pool.hpp).
// `src` = n 16-byte values in host memory, `dst` = n 16-byte slots in HBM.  Chunks are narrowed by the
// host pool into one of two pinned staging slots while the previous chunk is still on the bus; a chunk
// whose values do not fit int32 is retried as int64 and finally copied as is.  Bit-exact by construction.
static const int64_t NARROW_CHUNK_ROWS_DEFAULT = (int64_t)1 << 22;  // 64 MiB of source per chunk (b200.ingest.chunk_rows)
static const int64_t NARROW_BLOCK_ROWS = (int64_t)1 << 16;          // one pool task
static const int NARROW_SLOTS = 4;                                  // staging buffers in flight (b200.ingest.slots: 2..4)

void ingest_decimal_narrowed(b200_engine* e, const uint8_t* src, uint8_t* dst, int64_t n, cudaStream_t st) {
  std::lock_guard<std::mutex> ingest_guard(e->ingest_mu);
  if (!e->pool) {
    // default pool size: 1.5 x the CPUs this process may use (cgroup quota if there is one; the loops
    // are memory-latency bound, a few more threads than cores help, many more get throttled) --
    // measured on the B200 box (16-CPU quota): 12/16/24/32 threads -> 59.8/58.1/48.7/57.9 ms for SF10 lineitem
    int cpus = (int)std::thread::hardware_concurrency();
    if (cpus <= 0) cpus = 8;
    if (FILE* f = fopen("/sys/fs/cgroup/cpu.max", "r")) {
      long long quota = 0, period = 0;
      if (fscanf(f, "%lld %lld", &quota, &period) == 2 && quota > 0 && period > 0) cpus = std::min<int>(cpus, (int)std::max<long long>(1, quota / period));
      fclose(f);
    }
    int want = std::max(2, cpus + cpus / 2);
    {
      std::lock_guard<std::mutex> g(e->mu);
      auto it = e->config.find("b200.ingest.threads");
      if (it != e->config.end() && atoi(it->second.c_str()) > 0) want = atoi(it->second.c_str());
    }
    e->pool.reset(new HostPool(std::min(want, 256)));
  }
  const int64_t NARROW_CHUNK_ROWS = std::max<int64_t>(NARROW_BLOCK_ROWS, e->ingest_chunk_rows);
  const int n_slots = std::min(NARROW_SLOTS, std::max(2, e->ingest_slots));
  for (int si = 0; si < n_slots; si++) {
    auto& sl = e->nslot[si];
    const size_t need = (size_t)NARROW_CHUNK_ROWS * 8;
    if (sl.pinned && sl.bytes < need) {
      CUDA_CHECK(cudaStreamSynchronize(st));
      cudaFreeHost(sl.pinned);
      cudaFree(sl.dev);
      sl.pinned = sl.dev = nullptr;
      sl.used = false;
    }
    if (!sl.pinned) {
      CUDA_CHECK(cudaHostAlloc(&sl.pinned, need, cudaHostAllocDefault));
      CUDA_CHECK(cudaMalloc(&sl.dev, need));
      if (!sl.done) CUDA_CHECK(cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming));
      sl.bytes = need;
    }
  }
  int which = 0;
  for (int64_t r0 = 0; r0 < n; r0 += NARROW_CHUNK_ROWS, which = (which + 1) % n_slots) {
    const int64_t rows = std::min(NARROW_CHUNK_ROWS, n - r0);
    b200_engine::NarrowSlot& sl = e->nslot[which];
    if (sl.used) CUDA_CHECK(cudaEventSynchronize(sl.done));  // its previous chunk has left the staging buffer
    const int64_t* p = (const int64_t*)(src + r0 * 16);
    const int n_blocks = (int)((rows + NARROW_BLOCK_ROWS - 1) / NARROW_BLOCK_ROWS);
    int width = 0;
    for (int w : {4, 8}) {
      std::atomic<int> failed{0};
      e->pool->parallel_for(n_blocks, [&](int b) {
        if (failed.load(std::memory_order_relaxed)) return;
        const int64_t b0 = (int64_t)b * NARROW_BLOCK_ROWS, bn = std::min(NARROW_BLOCK_ROWS, rows - b0);
        const bool ok = w == 4 ? narrow_i128_to_i32(p + 2 * b0, bn, (int32_t*)sl.pinned + b0) : narrow_i128_to_i64(p + 2 * b0, bn, (int64_t*)sl.pinned + b0);
        if (!ok) failed.store(1, std::memory_order_relaxed);
      });
      if (!failed.load()) {
        width = w;
        break;
      }
    }
    if (width == 0) {  // genuinely wide values: ship the chunk unchanged
      CUDA_CHECK(cudaMemcpyAsync(dst + r0 * 16, src + r0 * 16, (size_t)rows * 16, cudaMemcpyHostToDevice, st));
      continue;
    }
    CUDA_CHECK(cudaMemcpyAsync(sl.dev, sl.pinned, (size_t)rows * width, cudaMemcpyHostToDevice, st));
    launch_widen_to_i128(sl.dev, width, dst + r0 * 16, rows, st);
    e->launches++;
    CUDA_CHECK(cudaEventRecord(sl.done, st));
    sl.used = true;
    e->narrowed_bytes_saved += (uint64_t)rows * (uint64_t)(16 - width);
  }
}

DevBatchPtr import_batch_impl(b200_engine* e, ArrowArray* arr, ArrowSchema* sch);

// Ownership of `arr` / `sch` moves to the engine on entry: they are released on success AND on failure (after the copies
// already issued from their buffers have drained), as the Arrow C Data Interface asks of a consumer.
DevBatchPtr import_batch(b200_engine* e, ArrowArray* arr, ArrowSchema* sch) {
  try {
    return import_batch_impl(e, arr, sch);
  } catch (...) {
    cudaStreamSynchronize(e->stream);
    if (arr && arr->release) arr->release(arr);
    if (sch && sch->release) sch->release(sch);
    throw;
  }
}

DevBatchPtr import_batch_impl(b200_engine* e, ArrowArray* arr, ArrowSchema* sch) {
  int64_t n = 0;
  std::vector<ImportedCol> ics = import_record_batch(arr, sch, &n);
  auto b = std::make_shared<DevBatch>();
  b->n = n;
  cudaStream_t st = e->stream;
  // Decimal128 columns of large batches go last, through the narrowing pipeline, so that the host pool
  // works while the plain copies of the other columns are on the bus
  bool narrow_on = n >= ((int64_t)1 << 20);
  {
    std::lock_guard<std::mutex> g(e->mu);
    auto it = e->config.find("b200.ingest.narrow_decimals");
    if (it != e->config.end()) narrow_on = it->second == "on" || (it->second != "off" && narrow_on);
  }
  struct Deferred { const uint8_t* src; uint8_t* dst; };
  std::vector<Deferred> deferred;
  for (auto& ic : ics) {
    DevColumn c;
    c.name = ic.name;
    c.type = ic.type;
    c.phys = phys_of(ic.type);
    c.n = n;
    c.nullable = ic.null_count > 0;
    if (ic.type.id == TypeId::Null) throw EngineError(B200_ERR_UNSUPPORTED, "Null-typed columns are not supported");
    if (ic.null_count > 0 && ic.validity) {
      int64_t b0 = ic.offset >> 3, b1 = (ic.offset + n + 7) >> 3;
      DevPtr bm = dev_alloc((size_t)(b1 - b0) + 16, st);
      CUDA_CHECK(cudaMemcpyAsync(bm->ptr, ic.validity + b0, (size_t)(b1 - b0), cudaMemcpyHostToDevice, st));
      DevPtr v = dev_alloc((size_t)n + 16, st);
      launch_bitmap_to_bytes((const uint8_t*)bm->ptr, ic.offset & 7, (uint8_t*)v->ptr, n, st);
      e->launches++;
      c.valid = (const uint8_t*)v->ptr;
      c.keep.push_back(v);
      c.keep.push_back(bm);
    }
    if (ic.type.id == TypeId::Bool) {
      int64_t b0 = ic.offset >> 3, b1 = (ic.offset + n + 7) >> 3;
      DevPtr bm = dev_alloc((size_t)(b1 - b0) + 16, st);
      CUDA_CHECK(cudaMemcpyAsync(bm->ptr, ic.data + b0, (size_t)(b1 - b0), cudaMemcpyHostToDevice, st));
      DevPtr v = dev_alloc((size_t)n + 16, st);
      launch_bitmap_to_bytes((const uint8_t*)bm->ptr, ic.offset & 7, (uint8_t*)v->ptr, n, st);
      e->launches++;
      c.data = (const uint8_t*)v->ptr;
      c.keep.push_back(v);
      c.keep.push_back(bm);
    } else if (ic.type.id == TypeId::Utf8) {
      if (ic.large_offsets) throw EngineError(B200_ERR_UNSUPPORTED, "LargeUtf8/LargeBinary input: cast to Utf8 on the host side");
      const int32_t* off = (const int32_t*)ic.data + ic.offset;
      int32_t first = off[0], last = off[n];
      DevPtr d_off = dev_alloc((size_t)(n + 1) * 4 + 64, st);
      CUDA_CHECK(cudaMemcpyAsync(d_off->ptr, off, (size_t)(n + 1) * 4, cudaMemcpyHostToDevice, st));
      DevPtr d_chars = dev_alloc((size_t)(last - first) + 64, st);
      if (last > first) CUDA_CHECK(cudaMemcpyAsync(d_chars->ptr, ic.extra + first, (size_t)(last - first), cudaMemcpyHostToDevice, st));
      c.data = (const uint8_t*)d_off->ptr;
      c.chars = (const uint8_t*)d_chars->ptr - first;
      c.chars_bytes = last - first;
      c.keep.push_back(d_off);
      c.keep.push_back(d_chars);
    } else {
      int w = c.width();
      DevPtr d = dev_alloc((size_t)n * w + 64, st);
      if (n && narrow_on && ic.type.id == TypeId::Decimal128 && w == 16) deferred.push_back(Deferred{ic.data + ic.offset * w, (uint8_t*)d->ptr});
      else if (n) CUDA_CHECK(cudaMemcpyAsync(d->ptr, ic.data + ic.offset * w, (size_t)n * w, cudaMemcpyHostToDevice, st));
      c.data = (const uint8_t*)d->ptr;
      c.keep.push_back(d);
    }
    b->cols.push_back(c);
  }
  for (auto& d : deferred) ingest_decimal_narrowed(e, d.src, d.dst, n, st);
  // the copies above read host memory owned by the Arrow arrays: wait before releasing them
  CUDA_CHECK(cudaStreamSynchronize(st));
  if (arr->release) arr->release(arr);
  if (sch->release) sch->release(sch);
  return b;
}

// ------------------------------------------------------------------------------------------------
// Arrow export (HBM -> host)
// ------------------------------------------------------------------------------------------------
// Small results (the tail of most queries is a handful of rows): ONE kernel packs every buffer of the batch
// (bitmaps + null counts, fixed-width values, string offsets and characters) into a device arena, one copy
// brings the arena to pinned host memory, one synchronisation in total.  Character areas are sized optimistically;
// a column that needs more sends the batch down the general path.
static const int64_t SMALL_EXPORT_ROWS = 4096;
static const size_t SMALL_EXPORT_ARENA = (size_t)1 << 20;
static const size_t SMALL_EXPORT_CHARS = (size_t)32 << 10;  // per string column

bool download_small(const Exec& x, const DevBatch& b, int64_t r0, int64_t r1, std::vector<HostCol>& hcs_out) {
  const int64_t n = r1 - r0;
  std::lock_guard<std::mutex> eg(x.e->export_mu);
  if (!x.e->export_arena && cudaHostAlloc((void**)&x.e->export_arena, SMALL_EXPORT_ARENA, cudaHostAllocDefault) != cudaSuccess) {
    x.e->export_arena = nullptr;
    return false;
  }
  uint8_t* arena = x.e->export_arena;
  cudaStream_t st = x.st();
  struct Slot { size_t validity = 0, count = 0, data = 0, chars = 0, chars_cap = 0; bool has_valid = false; };
  std::vector<Slot> slots(b.cols.size());
  std::vector<HostCol> hcs(b.cols.size());
  std::vector<DevColumn> cs(b.cols.size());
  size_t pos = 0;
  auto take = [&](size_t bytes) {
    size_t p = pos;
    pos += (bytes + 63) & ~(size_t)63;
    return p;
  };
  for (size_t ci = 0; ci < b.cols.size(); ci++) {
    cs[ci] = slice_column(b.cols[ci], r0, r1);
    const DevColumn& c = cs[ci];
    HostCol& h = hcs[ci];
    Slot& sl = slots[ci];
    h.name = c.name;
    h.type = c.type;
    h.nullable = true;
    h.n = n;
    if (c.valid && n) {
      sl.has_valid = true;
      sl.validity = take((size_t)(n + 7) / 8);
      sl.count = take(8);
    }
    if (c.type.id == TypeId::Bool) {
      h.data.assign((size_t)(n + 7) / 8, 0);
      sl.data = take(h.data.size());
    } else if (c.type.id == TypeId::Utf8) {
      h.data.resize((size_t)(n + 1) * 4);
      sl.data = take(h.data.size());
      sl.chars_cap = (c.phys == PH_UTF8 && c.chars_bytes >= 0) ? (size_t)c.chars_bytes : SMALL_EXPORT_CHARS;
      sl.chars = take(sl.chars_cap);
    } else {
      h.data.resize((size_t)n * c.width());
      sl.data = take(h.data.size());
    }
    if (pos > SMALL_EXPORT_ARENA) return false;
  }
  if (pos == 0) {
    hcs_out = std::move(hcs);
    return true;
  }
  DevPtr dev = dev_alloc(pos, st);
  uint8_t* d = (uint8_t*)dev->ptr;
  PackList pl;
  for (size_t ci = 0; ci < b.cols.size(); ci++) {
    const DevColumn& c = cs[ci];
    const Slot& sl = slots[ci];
    if (sl.has_valid) pl.bitmap(c.valid, n, d + sl.validity, d + sl.count);
    if (c.type.id == TypeId::Bool) {
      if (n) pl.bitmap(c.data, n, d + sl.data, nullptr);
    } else if (c.type.id == TypeId::Utf8) {
      pl.strings(c, d + sl.data, d + sl.chars, sl.chars_cap);
    } else if (n) {
      pl.copy(c.data, d + sl.data, (uint64_t)n * c.width());
    }
  }
  pl.run(x);
  CUDA_CHECK(cudaMemcpyAsync(arena, d, pos, cudaMemcpyDeviceToHost, st));
  x.sync();
  for (size_t ci = 0; ci < b.cols.size(); ci++)
    if (hcs[ci].type.id == TypeId::Utf8) {
      int32_t total = 0;
      memcpy(&total, arena + slots[ci].data + (size_t)n * 4, 4);
      if ((size_t)total > slots[ci].chars_cap) return false;  // optimistic character area too small: general path
    }
  for (size_t ci = 0; ci < b.cols.size(); ci++) {
    HostCol& h = hcs[ci];
    const Slot& sl = slots[ci];
    if (sl.has_valid) {
      unsigned long long nulls = 0;
      memcpy(&nulls, arena + sl.count, 8);
      h.null_count = (int64_t)nulls;
      if (nulls) h.validity.assign(arena + sl.validity, arena + sl.validity + (size_t)(n + 7) / 8);
    }
    if (!h.data.empty()) memcpy(h.data.data(), arena + sl.data, h.data.size());
    if (h.type.id == TypeId::Utf8) {
      const int32_t total = ((const int32_t*)h.data.data())[n];
      h.extra.assign(arena + sl.chars, arena + sl.chars + (size_t)total);
    }
  }
  hcs_out = std::move(hcs);
  return true;
}

// rows [r0, r1) of a device batch as host columns (Arrow buffers: bitmaps, values, offsets + characters)
std::vector<HostCol> download_batch(const Exec& x, const DevBatch& b, int64_t r0, int64_t r1) {
  const int64_t n = r1 - r0;
  std::vector<HostCol> hcs;
  if (n <= SMALL_EXPORT_ROWS && download_small(x, b, r0, r1, hcs)) return hcs;
  hcs.clear();
  cudaStream_t st = x.st();
  for (auto& c0 : b.cols) {
    DevColumn c = slice_column(c0, r0, r1);
    HostCol h;
    h.name = c.name;
    h.type = c.type;
    h.nullable = true;
    h.n = n;
    if (c.valid && n) {
      DevPtr bm = dev_alloc((size_t)(n + 7) / 8 + 16, st);
      DevPtr cnt = dev_alloc(8, st);
      CUDA_CHECK(cudaMemsetAsync(cnt->ptr, 0, 8, st));
      launch_bytes_to_bitmap(c.valid, (uint8_t*)bm->ptr, n, (unsigned long long*)cnt->ptr, st);
      x.count();
      h.validity.resize((size_t)(n + 7) / 8);
      CUDA_CHECK(cudaMemcpyAsync(h.validity.data(), bm->ptr, h.validity.size(), cudaMemcpyDeviceToHost, st));
      h.null_count = (int64_t)x.get<unsigned long long>(cnt->ptr);
      if (h.null_count == 0) h.validity.clear();
    }
    if (c.type.id == TypeId::Bool) {
      h.data.assign((size_t)(n + 7) / 8, 0);
      if (n) {
        DevPtr bm = dev_alloc((size_t)(n + 7) / 8 + 16, st);
        launch_bytes_to_bitmap(c.data, (uint8_t*)bm->ptr, n, nullptr, st);
        x.count();
        CUDA_CHECK(cudaMemcpyAsync(h.data.data(), bm->ptr, h.data.size(), cudaMemcpyDeviceToHost, st));
        x.wait();
      }
    } else if (c.type.id == TypeId::Utf8) {
      DevColumn u = c.phys == PH_STRVIEW ? as_utf8(x, c) : c;
      h.data.resize((size_t)(n + 1) * 4);
      CUDA_CHECK(cudaMemcpyAsync(h.data.data(), u.data, h.data.size(), cudaMemcpyDeviceToHost, st));
      x.wait();
      int32_t* off = (int32_t*)h.data.data();
      int32_t first = off[0], last = off[n];
      h.extra.resize((size_t)(last - first));
      if (last > first) CUDA_CHECK(cudaMemcpyAsync(h.extra.data(), u.chars + first, h.extra.size(), cudaMemcpyDeviceToHost, st));
      x.wait();
      for (int64_t i = 0; i <= n; i++) off[i] -= first;
    } else {
      h.data.resize((size_t)n * c.width());
      if (n) CUDA_CHECK(cudaMemcpyAsync(h.data.data(), c.data, h.data.size(), cudaMemcpyDeviceToHost, st));
      x.wait();
    }
    hcs.push_back(std::move(h));
  }
  return hcs;
}

void export_batch(const Exec& x, const DevBatch& b, int64_t r0, int64_t r1, ArrowArray* out, ArrowSchema* out_schema) {
  std::vector<HostCol> hcs = download_batch(x, b, r0, r1);
  export_record_batch(std::move(hcs), r1 - r0, out, out_schema);
}

// ------------------------------------------------------------------------------------------------
// Pipeline execution
// ------------------------------------------------------------------------------------------------
struct RunOutcome {
  RunStatus status;
  float ms = 0;
  const RunStatus* deferred = nullptr;          // wait == false: the status word, readable after the task's next sync
  const unsigned int* deferred_extra = nullptr;  // ... and the `extra_fetch` word
};

// the fused kernel's description of a program it can run instead of the tile VM (match_fused)
struct FusedPlan {
  FusedSpec spec;
  FusedShape shape;
  int block = 0;
  size_t smem = 0;
};

static void throw_run_error(unsigned int error) {
  if (error == 1) throw EngineError(B200_ERR_EXECUTION, "Arithmetic overflow");
  if (error == 2) throw EngineError(B200_ERR_EXECUTION, "Divide by zero");
  if (error) throw EngineError(B200_ERR_EXECUTION, "execution error in expression");
}

static bool program_filters(const Program& P) {
  for (int i = 0; i < P.n_instr; i++)
    if (P.code[i].op == OP_FILTER || (P.code[i].flags & IF_FILTER)) return true;
  return false;
}

// Enqueues the pipeline kernel.  wait == true: synchronises, checks the status word and returns it
// (`extra_fetch`, if given, is a device word read back in the same synchronisation).  wait == false:
// the caller already knows the output size; the status check (and the kernel time for the metrics)
// is deferred to the task's next synchronisation.
bool match_groupby(const Program& P, GroupBySpec& S);
bool match_fast_filter(const Program& P, FastFilterSpec& S);

// Partition-first aggregation (AggregateExec with more groups than the L2 can hold a table for): radix-partition the
// referenced columns by hash(keys) % K with the shuffle writer's kernels, so that bucket b's groups live in their own
// region of the table (cap / K slots, ~32 MB of touched cells) that stays in L2 while that bucket's CTAs run -- the
// random accesses of the upsert become L2 hits instead of 32-byte DRAM sectors.  Bytes: one extra read + write of the
// referenced columns (sequential) against three random sectors per row saved.  The bucket ranges are resolved on the
// device (launch_groupby_plan): no host synchronisation between the partition and the aggregation.
bool partition_for_groupby(const Exec& x, GroupBySpec& S, std::vector<DevPtr>& keep) {
  // b200.agg.partition_first.bucket_slots (default 2^19 slots ~ 32 MB of touched cells; 0 = never partition),
  // b200.agg.partition_first.min_rows (default 2^22)
  const uint64_t GB_PF_BUCKET_SLOTS = x.e->pf_bucket_slots;
  if (!GB_PF_BUCKET_SLOTS || S.n_keys < 1 || S.table.cap < GB_PF_BUCKET_SLOTS * 8 || S.n_rows < x.e->pf_min_rows || S.n_rows >= ((int64_t)1 << 32)) return false;
  for (int k = 0; k < S.n_keys; k++) {
    const uint32_t w = S.cols[S.key_col[k]].width;
    if (w != 4 && w != 8) return false;
  }
  const uint32_t K = (uint32_t)std::min<uint64_t>(S.table.cap / GB_PF_BUCKET_SLOTS, PART_MAX_FANOUT);
  const int64_t n = S.n_rows;
  PidSrc ps;
  memset(&ps, 0, sizeof ps);
  ps.salt = 0x5bd1e995;  // not the shuffle's partition function: the input may BE one shuffle partition of these very keys
  for (int k = 0; k < S.n_keys; k++) {
    const FusedCol& c = S.cols[S.key_col[k]];
    ps.keys[ps.n_keys++] = KeyCol{c.data, nullptr, (uint8_t)(c.width == 4 ? PH_I32 : PH_I64), (uint8_t)c.width};
  }
  const uint32_t n_tiles = partition_n_tiles(n);
  DevPtr acc = dev_alloc((size_t)K * 8 + 64, x.st());
  CUDA_CHECK(cudaMemsetAsync(acc->ptr, 0, (size_t)K * 8, x.st()));
  DevPtr tile_hist = dev_alloc((size_t)K * n_tiles * 4 + 64, x.st());
  PartStrCols sc;
  sc.n = 0;
  CUDA_CHECK(launch_partition_hist(ps, n, K, (uint32_t*)tile_hist->ptr, (unsigned long long*)acc->ptr, sc, (unsigned long long*)acc->ptr + K, x.st()));
  const int64_t hn = (int64_t)K * n_tiles;
  DevPtr offs = dev_alloc((size_t)(hn + 2) * 8, x.st());
  DevPtr scratch = dev_alloc((size_t)(hn / 1024 + 4) * 8, x.st());
  launch_scan_u32_to_u64((const uint32_t*)tile_hist->ptr, (uint64_t*)offs->ptr, hn, (uint64_t*)scratch->ptr, x.st());
  GatherCols gc;
  gc.n = 0;
  for (int c = 0; c < S.n_cols; c++) {
    DevPtr out = dev_alloc((size_t)n * S.cols[c].width + 64, x.st());
    GatherCol& g = gc.c[gc.n++];
    memset(&g, 0, sizeof g);
    g.in = S.cols[c].data;
    g.out = out->ptr;
    g.width = (int)S.cols[c].width;
    S.cols[c].data = out->ptr;
    keep.push_back(out);
  }
  CUDA_CHECK(launch_partition_scatter(ps, n, K, (const uint64_t*)offs->ptr, gc, nullptr, x.st()));
  DevPtr row_start = dev_alloc((size_t)(K + 1) * 8 + 64, x.st()), cta_start = dev_alloc((size_t)(K + 1) * 4 + 64, x.st());
  CUDA_CHECK(launch_groupby_plan((const unsigned long long*)acc->ptr, (int)K, (unsigned long long*)row_start->ptr, (unsigned int*)cta_start->ptr, x.st()));
  x.count(6);
  S.pf_K = (int)K;
  S.pf_slots = S.table.cap / K;
  S.pf_row_start = (const unsigned long long*)row_start->ptr;
  S.pf_cta_start = (const unsigned int*)cta_start->ptr;
  keep.push_back(row_start);
  keep.push_back(cta_start);
  keep.push_back(acc);
  keep.push_back(tile_hist);
  keep.push_back(offs);
  keep.push_back(scratch);
  x.e->n_groupby_pf++;
  return true;
}

RunOutcome launch_program(const Exec& x, PipelineBuilder& pb, int reg_groups, const FusedPlan* fused = nullptr, bool wait = true, OpMetrics* met = nullptr,
                          const unsigned int* extra_fetch = nullptr, unsigned int* extra_out = nullptr, const GroupBySpec* gb = nullptr,
                          const FastFilterSpec* ff = nullptr) {
  Program& P = pb.prog;
  DevPtr dstat = dev_alloc(sizeof(RunStatus), x.st());
  CUDA_CHECK(cudaMemsetAsync(dstat->ptr, 0, sizeof(RunStatus), x.st()));
  P.status = (RunStatus*)dstat->ptr;
  DevPtr tstate;
  if (P.sink == SINK_MATERIALIZE) {
    const int64_t tile_rows = ff ? 1024 : (int64_t)pb.block * VM_R;
    const int64_t nt = (P.n_rows + tile_rows - 1) / tile_rows;
    tstate = dev_alloc((size_t)std::max<int64_t>(nt, 1) * 8, x.st());
    CUDA_CHECK(cudaMemsetAsync(tstate->ptr, 0, (size_t)std::max<int64_t>(nt, 1) * 8, x.st()));
    P.tile_state = (unsigned long long*)tstate->ptr;
  }
  int grid;
  if (fused) {
    const int64_t warp_tile = 32 * fused->spec.rows_per_thread, nw = fused->block / 32;
    const int64_t n_wt = (P.n_rows + warp_tile - 1) / warp_tile;
    grid = (int)std::min<int64_t>(std::max<int64_t>((n_wt + nw - 1) / nw, 1), x.e->sm_count);
    if (!fused_rows_ok(P, grid, fused->block, fused->spec.rows_per_thread)) fused = nullptr;
  }
  if (!fused) {
    const int tile = pb.block * VM_R;
    int64_t n_tiles = (P.n_rows + tile - 1) / tile;
    grid = (int)std::min<int64_t>(std::max<int64_t>(n_tiles, 1), x.e->sm_count);
  }
  static const bool debug = getenv("B200_DEBUG") != nullptr;
  if (debug)
    fprintf(stderr, "[b200] pipeline sink=%d rows=%lld cols=%d instr=%d regs=%d block=%d stages=%u stage_bytes=%u regs_bytes=%u tma=%u grid=%d\n", (int)P.sink,
            (long long)P.n_rows, P.n_cols, P.n_instr, P.n_regs, pb.block, P.n_stages, P.stage_bytes, P.regs_bytes, P.use_tma, grid);
  if (debug) {
    for (int i = 0; i < P.n_instr; i++) {
      const VInstr& v = P.code[i];
      fprintf(stderr, "[b200]   %2d: op=%d t=%d fl=%d aux=%d dst=(%d,%d,%d) a=(%d,%d,%d) b=(%d,%d,%d) imm=%d\n", i, v.op, v.t, v.flags, v.aux, v.dst.kind, v.dst.vk,
              v.dst.idx, v.a.kind, v.a.vk, v.a.idx, v.b.kind, v.b.vk, v.b.idx, v.imm);
    }
    for (int i = 0; i < P.n_regs; i++) fprintf(stderr, "[b200]   reg %d: vk=%d off=%u valid_off=%u\n", i, P.regs[i].vk, P.regs[i].smem_off, P.regs[i].valid_off);
  }
  uint64_t kt_bytes = 0;
  for (int i = 0; i < P.n_cols; i++) kt_bytes += (uint64_t)P.cols[i].width * (uint64_t)P.n_rows;
  if (P.sink == SINK_MATERIALIZE)
    for (int j = 0; j < P.n_out; j++) kt_bytes += (uint64_t)phys_width((Phys)P.out[j].phys) * (uint64_t)P.n_rows;  // upper bound: every row kept
  KernelTimer kt(x, ff ? "filter_compact" : gb ? "groupby_hash_agg" : fused ? "pipeline_fused_agg" : P.sink == SINK_MATERIALIZE ? "pipeline_materialize" : P.sink == SINK_AGG_REG ? "pipeline_agg_reg" : "pipeline_agg_global", kt_bytes);
  cudaEvent_t e0, e1;
  CUDA_CHECK(cudaEventCreate(&e0));
  CUDA_CHECK(cudaEventCreate(&e1));
  CUDA_CHECK(cudaEventRecord(e0, x.st()));
  cudaError_t le;
  if (ff) {
    FastFilterSpec S = *ff;
    S.status = P.status;
    S.tile_state = P.tile_state;
    le = launch_fast_filter(S, x.e->sm_count, x.st());
    x.e->n_fastfilter++;
  } else if (gb) {
    GroupBySpec S = *gb;
    S.status = P.status;
    S.table = P.table;
    const bool allow_pf = gb->pf_K != -1;
    S.pf_K = 0;
    std::vector<DevPtr> pf_keep;  // stream-ordered: released after the launch below is enqueued
    if (allow_pf) partition_for_groupby(x, S, pf_keep);
    le = launch_groupby(S, x.e->sm_count, x.st());
    x.e->n_groupby++;
  } else if (fused) {
    int is_static = 0;
    le = launch_fused_pipeline(P, fused->spec, fused->shape, reg_groups, grid, fused->block, fused->smem, x.st(), &is_static);
    x.e->n_fused++;
    if (is_static) x.e->n_fused_static++;
    if (debug) {
      const FusedSpec& F = fused->spec;
      fprintf(stderr, "[b200]   fused kernel: static=%d shape=(%#llx,%#llx) block=%d R=%d stages=%d stage_bytes=%u smem=%zu grid=%d tma=%u\n", is_static,
              (unsigned long long)fused->shape.a, (unsigned long long)fused->shape.b, fused->block, F.rows_per_thread, F.n_stages, F.stage_bytes, fused->smem, grid,
              F.use_tma);
      for (int i = 0; i < F.n_filters; i++) fprintf(stderr, "[b200]     filter %d: w=%d op=%d\n", i, F.f[i].w, F.f[i].op - OP_CMP_EQ);
      for (int k = 0; k < F.n_keys; k++) fprintf(stderr, "[b200]     key %d: kind=%d w=%d max_len=%d shift=%d\n", k, F.k[k].kind, F.k[k].w, F.k[k].max_len, F.k[k].shift);
      for (int j = 0; j < F.n_prod; j++) fprintf(stderr, "[b200]     prod %d: kind=%d a_src=%d a_w=%d b_w=%d\n", j, F.p[j].kind, F.p[j].a_src, F.p[j].a_w, F.p[j].b_w);
      for (int a = 0; a < F.n_acc; a++) fprintf(stderr, "[b200]     acc %d: src=%d w=%d\n", a, F.a[a].src, F.a[a].w);
      fprintf(stderr, "[b200]     combine=%d\n", F.combine);
    }
  } else {
    le = launch_pipeline(P, reg_groups, grid, pb.block, pb.smem_bytes(), x.st());
    x.e->n_vm++;
  }
  if (le != cudaSuccess) {
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    CUDA_CHECK(le);
  }
  CUDA_CHECK(cudaEventRecord(e1, x.st()));
  x.count();
  RunOutcome o;
  const RunStatus* hs = x.fetch<RunStatus>(dstat->ptr);
  const unsigned int* he = extra_fetch ? x.fetch<unsigned int>(extra_fetch) : nullptr;
  if (!wait) {
    x.defer([hs, e0, e1, met, dstat, tstate]() {
      float ms = 0;
      cudaEventElapsedTime(&ms, e0, e1);
      cudaEventDestroy(e0);
      cudaEventDestroy(e1);
      if (met) met->elapsed_ns += (uint64_t)(ms * 1e6);
      throw_run_error(hs->error);
    });
    memset(&o.status, 0, sizeof o.status);
    o.deferred = hs;
    o.deferred_extra = he;
    return o;
  }
  try {
    x.sync();
  } catch (...) {
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    throw;
  }
  o.status = *hs;
  if (he && extra_out) *extra_out = *he;
  cudaEventElapsedTime(&o.ms, e0, e1);
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  if (met) met->elapsed_ns += (uint64_t)(o.ms * 1e6);
  throw_run_error(o.status.error);
  return o;
}

uint64_t source_bytes(const PipelineBuilder& pb) {
  uint64_t b = 0;
  for (int i = 0; i < pb.prog.n_cols; i++) b += (uint64_t)pb.prog.cols[i].width * (uint64_t)pb.prog.n_rows + (pb.prog.cols[i].valid ? (uint64_t)pb.prog.n_rows : 0);
  return b;
}

// materialise `outs` (current builder columns) -> new batch
DevBatchPtr run_materialize(const Exec& x, PipelineBuilder& pb, const std::vector<ColRef>& outs, const DevBatchPtr& src, OpMetrics* met) {
  Program& P = pb.prog;
  if (outs.size() > (size_t)VM_MAX_OUT) throw EngineError(B200_ERR_UNSUPPORTED, "too many output columns in one pipeline");
  auto out = std::make_shared<DevBatch>();
  const int64_t cap = src->n;
  P.sink = SINK_MATERIALIZE;
  P.n_out = (uint8_t)outs.size();
  for (size_t j = 0; j < outs.size(); j++) {
    const ColRef& c = outs[j];
    Phys ph = c.type.id == TypeId::Utf8 ? PH_STRVIEW : phys_of(c.type);
    DevColumn oc = make_out_column(c.name, c.type, ph, cap, c.nullable, x.st());
    for (auto& k : c.keep) oc.keep.push_back(k);
    OutCol& d = P.out[j];
    memset(&d, 0, sizeof d);
    d.src = pb.resolve(c);
    d.data = (void*)oc.data;
    d.valid = (uint8_t*)oc.valid;
    d.phys = ph;
    out->cols.push_back(oc);
  }
  pb.finalize_layout(4096);
  // without a filter every input row comes out: no need to wait for the row count
  const bool filters = program_filters(P);
  FastFilterSpec ffs;
  const bool use_ff = filters && match_fast_filter(P, ffs);
  RunOutcome r = launch_program(x, pb, 1, nullptr, filters, met, nullptr, nullptr, nullptr, use_ff ? &ffs : nullptr);
  out->n = filters ? (int64_t)r.status.out_rows : src->n;
  uint64_t wbytes = 0;
  for (auto& c : out->cols) {
    c.n = out->n;
    wbytes += (uint64_t)c.width() * (uint64_t)out->n;
  }
  // the views may point into the source batch's character buffers
  for (auto& c : out->cols)
    if (c.phys == PH_STRVIEW)
      for (auto& sc : src->cols)
        if (sc.phys == PH_UTF8 || sc.phys == PH_STRVIEW)
          for (auto& k : sc.keep) c.keep.push_back(k);
  for (auto& k : pb.keep)
    for (auto& c : out->cols)
      if (c.phys == PH_STRVIEW) c.keep.push_back(k);
  if (met) {
    met->bytes_read += source_bytes(pb);
    met->bytes_written += wbytes;
    met->launches += 1;
  }
  return out;
}

// ---- aggregate ------------------------------------------------------------------------------------
struct AggLowered {
  std::vector<ColRef> keys;          // what the group table stores (packed strings are Int64 values)
  std::vector<int> key_pack_shift;   // 0: plain key; 56 / 24: packed short string (bit position of the length)
  bool fast = false;                 // key_hash is an injective 64-bit image of the whole key
  ColRef combined;                   // valid when fast
  std::vector<AccDesc> accs;
  std::vector<ColRef> acc_src;
  struct OutRecipe {
    uint8_t kind, a, b;
    Phys phys;
    int imm;
    DataType type;
    std::string name;
    bool with_valid;
    int key_idx;
  };
  std::vector<OutRecipe> outs;
};

int add_acc(PipelineBuilder& pb, AggLowered& L, uint8_t kind, const ColRef* src) {
  Operand so;
  memset(&so, 0, sizeof so);
  bool nullable = false;
  if (src) {
    so = pb.resolve(*src);
    nullable = src->nullable;
  }
  for (size_t i = 0; i < L.accs.size(); i++) {
    const AccDesc& a = L.accs[i];
    if (a.kind == kind && (kind == ACC_COUNT_STAR || (a.src.kind == so.kind && a.src.idx == so.idx && a.src.vk == so.vk))) return (int)i;
  }
  if (L.accs.size() >= (size_t)VM_MAX_ACC) throw EngineError(B200_ERR_UNSUPPORTED, "too many aggregates in one AggregateExec");
  AccDesc a;
  memset(&a, 0, sizeof a);
  a.kind = kind;
  a.src = so;
  a.nullable = nullable ? 1 : 0;
  L.accs.push_back(a);
  if (src) {
    pb.pin(*src);
    L.acc_src.push_back(*src);
  }
  return (int)L.accs.size() - 1;
}

static bool narrowable(const DataType& t) {
  switch (t.id) {
    case TypeId::Utf8:
    case TypeId::Bool:
    case TypeId::Int8:
    case TypeId::Int16:
    case TypeId::Int32:
    case TypeId::UInt8:
    case TypeId::UInt16:
    case TypeId::UInt32:
    case TypeId::Date32: return true;
    default: return false;
  }
}

// pack_mode: 0 = keys as they are; 1 = short strings packed into Int64 (len<<56 | <=7 bytes);
//            2 = every key squeezed into 32 bits and combined injectively into one 64-bit value
// The packed forms are optimistic: the kernel raises pack_overflow when a string does not fit and
// the caller re-lowers with a smaller pack_mode.
void lower_aggregate(PipelineBuilder& pb, const PlanNode& node, AggLowered& L, int pack_mode) {
  const bool from_states = agg_mode_consumes_states(node.agg_mode);
  const bool emit_states = agg_mode_emits_states(node.agg_mode);
  const bool scalar = node.group_by.empty();
  std::vector<ColRef> narrow32;  // pack_mode 2: non-negative 32-bit images of the keys
  for (size_t g = 0; g < node.group_by.size(); g++) {
    ColRef k0 = pb.compile(*node.group_by[g].expr);
    pb.pin(k0);
    ColRef k = k0;
    int shift = 0;
    if (k0.type.id == TypeId::Utf8 && pack_mode > 0) {
      shift = pack_mode == 2 ? 24 : 56;
      k = pb.str_pack(k0, pack_mode == 2 ? 3 : 7, shift);
      pb.pin(k);
    }
    if (pack_mode == 2) {
      ColRef n32 = k;
      if (shift == 0 && (k0.type.is_signed_int() || k0.type.id == TypeId::Date32)) {
        n32 = pb.add_literal_i64(k, 2147483648ll);
        pb.pin(n32);
      }
      narrow32.push_back(n32);
    }
    k.name = node.group_by[g].name;
    L.keys.push_back(k);
    L.key_pack_shift.push_back(shift);
    AggLowered::OutRecipe r{};
    r.kind = shift ? AO_KEY_PACKED : AO_KEY;
    r.a = (uint8_t)g;
    r.b = 255;
    r.type = k0.type;
    r.phys = k0.type.id == TypeId::Utf8 ? PH_STRVIEW : phys_of(k0.type);
    r.name = k.name;
    r.with_valid = k0.nullable;
    r.key_idx = (int)g;
    r.imm = shift;
    L.outs.push_back(r);
  }
  // injective 64-bit key image => the register-cached group directory can be used
  {
    bool all_i64 = !L.keys.empty(), any_null = false;
    for (auto& k : L.keys) {
      all_i64 &= (k.type.pk() == PK::I64 || k.type.pk() == PK::Bool);
      any_null |= k.nullable;
    }
    if (all_i64 && !any_null) {
      if (L.keys.size() == 1) {
        L.fast = true;
        L.combined = L.keys[0];
      } else if (pack_mode == 2 && L.keys.size() == 2) {
        L.fast = true;
        L.combined = pb.combine32(narrow32[0], narrow32[1]);
        pb.pin(L.combined);
      }
    }
  }
  const int star = add_acc(pb, L, ACC_COUNT_STAR, nullptr);
  size_t state_col = node.group_by.size();
  (void)emit_states;
  auto push = [&](uint8_t kind, int a, int b, const DataType& t, const std::string& name, bool with_valid, int imm = 0) {
    AggLowered::OutRecipe r{};
    r.kind = kind;
    r.a = (uint8_t)a;
    r.b = (uint8_t)b;
    r.type = t;
    r.phys = phys_of(t);
    r.name = name;
    r.with_valid = with_valid;
    r.imm = imm;
    r.key_idx = -1;
    L.outs.push_back(r);
  };
  auto sum_out_kind = [](const DataType& t) -> uint8_t { return t.pk() == PK::F64 ? AO_ACC_F64 : (t.pk() == PK::I128 ? AO_ACC_I128 : AO_ACC_I64); };
  for (size_t ai = 0; ai < node.aggs.size(); ai++) {
    const AggExpr& ae = node.aggs[ai];
    const std::string& nm = ae.name;
    if (from_states) {
      ColRef s0 = pb.cols.at(state_col);
      switch (ae.fn) {
        case AggFn::Count: {
          int a = add_acc(pb, L, ACC_SUM_I128, &s0);
          push(AO_COUNT, a, 255, DataType(TypeId::Int64), nm, false);
          break;
        }
        case AggFn::Sum: {
          bool f = s0.type.pk() == PK::F64;
          int a = add_acc(pb, L, f ? ACC_SUM_F64 : ACC_SUM_I128, &s0);
          int c = s0.nullable ? add_acc(pb, L, ACC_COUNT, &s0) : star;
          push(sum_out_kind(ae.result_type), a, c, ae.result_type, nm, s0.nullable || scalar);
          break;
        }
        case AggFn::Min:
        case AggFn::Max: {
          if (s0.type.pk() == PK::Str) throw EngineError(B200_ERR_UNSUPPORTED, "MIN/MAX over Utf8");
          bool f = s0.type.pk() == PK::F64, mn = ae.fn == AggFn::Min;
          int a = add_acc(pb, L, f ? (mn ? ACC_MIN_F64 : ACC_MAX_F64) : (mn ? ACC_MIN_I128 : ACC_MAX_I128), &s0);
          int c = s0.nullable ? add_acc(pb, L, ACC_COUNT, &s0) : star;
          push(f ? AO_MINMAX_F64 : sum_out_kind(ae.result_type), a, c, ae.result_type, nm, s0.nullable || scalar);
          break;
        }
        case AggFn::Avg: {
          ColRef s1 = pb.cols.at(state_col + 1);
          int c = add_acc(pb, L, ACC_SUM_I128, &s0);
          bool f = s1.type.pk() == PK::F64;
          int a = add_acc(pb, L, f ? ACC_SUM_F64 : ACC_SUM_I128, &s1);
          if (f) push(AO_AVG_F64, a, c, ae.result_type, nm, true);
          else push(AO_AVG_DEC, a, c, ae.result_type, nm, true, ae.result_type.scale - ae.sum_type.scale);
          break;
        }
      }
      state_col += (size_t)ae.n_state_cols();
      continue;
    }
    ColRef arg;
    bool has_arg = ae.arg != nullptr;
    if (has_arg) arg = pb.compile(*ae.arg);
    switch (ae.fn) {
      case AggFn::Count: {
        int a = (has_arg && arg.nullable) ? add_acc(pb, L, ACC_COUNT, &arg) : star;
        push(AO_COUNT, a, 255, DataType(TypeId::Int64), emit_states ? nm + "[count]" : nm, false);
        break;
      }
      case AggFn::Sum: {
        ColRef v = arg;
        bool f = ae.sum_type.pk() == PK::F64;
        if (f) v = pb.cast_to(arg, DataType(TypeId::Float64));
        int a = add_acc(pb, L, f ? ACC_SUM_F64 : ACC_SUM_I128, &v);
        int c = v.nullable ? add_acc(pb, L, ACC_COUNT, &v) : star;
        push(sum_out_kind(ae.sum_type), a, c, ae.sum_type, emit_states ? nm + "[sum]" : nm, v.nullable || scalar);
        break;
      }
      case AggFn::Min:
      case AggFn::Max: {
        if (arg.type.pk() == PK::Str) throw EngineError(B200_ERR_UNSUPPORTED, "MIN/MAX over Utf8");
        if (arg.type.id == TypeId::UInt64) throw EngineError(B200_ERR_UNSUPPORTED, "MIN/MAX over UInt64");
        bool f = arg.type.pk() == PK::F64, mn = ae.fn == AggFn::Min;
        int a = add_acc(pb, L, f ? (mn ? ACC_MIN_F64 : ACC_MAX_F64) : (mn ? ACC_MIN_I128 : ACC_MAX_I128), &arg);
        int c = arg.nullable ? add_acc(pb, L, ACC_COUNT, &arg) : star;
        push(f ? AO_MINMAX_F64 : sum_out_kind(ae.sum_type), a, c, ae.sum_type, emit_states ? nm + (mn ? "[min]" : "[max]") : nm, arg.nullable || scalar);
        break;
      }
      case AggFn::Avg: {
        ColRef v = arg;
        bool f = !arg.type.is_decimal();
        if (f) v = pb.cast_to(arg, DataType(TypeId::Float64));
        int a = add_acc(pb, L, f ? ACC_SUM_F64 : ACC_SUM_I128, &v);
        int c = v.nullable ? add_acc(pb, L, ACC_COUNT, &v) : star;
        if (emit_states) {
          push(AO_COUNT, c, 255, DataType(TypeId::UInt64), nm + "[count]", false);
          push(sum_out_kind(ae.sum_type), a, c, ae.sum_type, nm + "[sum]", v.nullable || scalar);
        } else if (f) {
          push(AO_AVG_F64, a, c, ae.result_type, nm, true);
        } else {
          push(AO_AVG_DEC, a, c, ae.result_type, nm, true, ae.result_type.scale - ae.sum_type.scale);
        }
        break;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Pattern match of a lowered register-aggregate program against the fused fast path
// (filters on integer-like tile columns -> up to two decimal products -> <= 2 packed/integer keys ->
// SUM/COUNT accumulators).  Anything outside the pattern keeps the general VM path.
// ------------------------------------------------------------------------------------------------
static int env_int(const char* name, int dflt) {
  const char* v = getenv(name);
  return v && *v ? atoi(v) : dflt;
}

// Recognise the scan -> filter -> decimal products -> small SUM/COUNT aggregate shape in a lowered
// program and lay out the per-warp stage buffers of the fused kernel (fused.cuh).
bool match_fused(const Program& P, FusedPlan& FP) {
  FusedSpec& F = FP.spec;
  memset(&F, 0, sizeof F);
  if (P.sink != SINK_AGG_REG) return false;
  if (getenv("B200_NO_FUSED")) return false;
  for (int a = 0; a < P.n_acc; a++)
    if (!(P.acc[a].kind == ACC_SUM_I128 || P.acc[a].kind == ACC_COUNT || P.acc[a].kind == ACC_COUNT_STAR)) return false;
  // stage layout: every column of the program, one warp tile of 32*R rows each
  // measured on B200 (profiles/r01_summary.md): 4 rows per thread amortise the per-tile work (claim, TMA
  // issue, barrier wait) best; grouped shapes then fit 8 warps of up to 255 registers next to their
  // shared-memory partials, scalar shapes 12 warps
  const int R = env_int("B200_FUSED_R", 4);
  if (!(R == 2 || R == 4)) return false;
  int block = env_int("B200_FUSED_B", (R == 4 && P.n_keys) ? 256 : 384);
  if (block > (R == 4 ? 384 : 512) || block < 32 || (block & 31)) return false;
  const uint32_t TR = 32u * (uint32_t)R;
  if (P.n_cols > FUSED_MAX_COLS || P.n_cols == 0) return false;
  uint32_t fused_off[VM_MAX_COLS];
  uint32_t cur = 0, tx = 0, tx_utf8 = 0;
  bool aligned = true;
  // short-string keys with a pre-packed companion (prepack_short_strings) are read as 4-byte integer key columns
  bool prepacked[VM_MAX_COLS] = {false};
  if (!getenv("B200_NO_PREPACK"))
    for (int i = 0; i < P.n_instr; i++) {
      const VInstr& v = P.code[i];
      if (v.op == OP_STR_PACK8 && v.a.kind == OPD_COL && v.imm == 24 && v.aux <= 3 && P.cols[v.a.idx].phys == PH_UTF8 && P.cols[v.a.idx].packed32 &&
          (((uintptr_t)P.cols[v.a.idx].packed32) & 15) == 0)
        prepacked[v.a.idx] = true;
    }
  for (int c = 0; c < P.n_cols; c++) {
    const ColDesc& cd = P.cols[c];
    if (cd.valid) return false;
    FusedCol& fc = F.cols[c];
    fc.data = prepacked[c] ? cd.packed32 : cd.data;
    fc.width = prepacked[c] ? 4 : cd.width;
    fc.utf8 = (cd.phys == PH_UTF8 && !prepacked[c]) ? 1u : 0u;
    fc.tile_bytes = TR * fc.width + (fc.utf8 ? 16u : 0u);
    if (fc.tile_bytes & 15u) return false;
    fc.off = cur;
    fused_off[c] = cur;
    cur += fc.tile_bytes;
    if (fc.utf8) tx_utf8 += fc.tile_bytes;
    else tx += fc.tile_bytes;
    if (((uintptr_t)fc.data & 15) != 0) aligned = false;
  }
  F.n_cols = P.n_cols;
  F.rows_per_thread = R;
  F.stage_bytes = (cur + 127u) & ~127u;
  F.tile_tx = tx;
  F.tile_tx_utf8 = tx_utf8;
  F.use_tma = (aligned && !getenv("B200_NO_TMA")) ? 1u : 0u;
  {
    // shared memory: per-warp rings, then (grouped shapes) 8 bytes per (group, accumulator, thread)
    const size_t budget = 216 * 1024;
    const size_t acc_per_thread = P.n_keys ? (size_t)VM_REG_GROUPS * VM_REG_ACC * 8 : 0;
    const int want_S = std::min(env_int("B200_FUSED_S", FUSED_MAX_STAGES), (int)FUSED_MAX_STAGES);
    int S = 0;
    for (;; block -= 32) {
      if (block < 64) return false;
      const size_t acc = acc_per_thread * block;
      if (acc >= budget) continue;
      S = (int)((budget - acc) / ((size_t)(block / 32) * F.stage_bytes));
      if (S >= 2) break;
    }
    S = std::min(S, want_S);
    if (S < 2) return false;
    F.n_stages = S;
    FP.block = block;
    // the end-of-kernel reduction stages [VM_REG_ACC][block] 16-byte partials in the idle rings
    size_t ring = std::max((size_t)(block / 32) * S * F.stage_bytes, (size_t)VM_REG_ACC * block * 16);
    ring = (ring + 127) & ~(size_t)127;
    F.acc_off = (uint32_t)ring;
    FP.smem = ring + acc_per_thread * block;
  }
  auto int_col = [&](const Operand& o, uint32_t* off, uint8_t* w, bool want_i128) -> bool {
    if (o.kind != OPD_COL) return false;
    const ColDesc& cd = P.cols[o.idx];
    if (cd.valid) return false;
    if (!(cd.phys == PH_I32 || cd.phys == PH_I64 || cd.phys == PH_DEC128)) return false;
    if (want_i128 && o.vk == VK_I128 && cd.phys != PH_DEC128) return false;
    if (o.vk != VK_I128 && cd.phys == PH_DEC128) {
      // narrow view of a decimal: low word only
    }
    *off = fused_off[o.idx];
    *w = (o.vk == VK_I128) ? 16 : cd.width;
    return true;
  };
  int prod_reg[2] = {-1, -1};
  struct PackInfo { int reg; FusedKey k; };
  std::vector<PackInfo> packs;      // packed-string / biased-int key images by register
  int combined_reg = -1, comb_a = -1, comb_b = -1;
  for (int i = 0; i < P.n_instr; i++) {
    const VInstr& v = P.code[i];
    if (v.flags & IF_NULLCHK) return false;
    switch (v.op) {
      case OP_CMP_EQ: case OP_CMP_NE: case OP_CMP_LT: case OP_CMP_LE: case OP_CMP_GT: case OP_CMP_GE: {
        if (!(v.flags & IF_FILTER) || v.t != VK_I64 || v.aux == PH_U64) return false;
        if (F.n_filters >= FUSED_MAX_FILTERS) return false;
        FusedFilter& f = F.f[F.n_filters];
        Operand col = v.a, imm = v.b;
        uint8_t op = v.op;
        if (v.a.kind == OPD_IMM && v.b.kind == OPD_COL) {
          col = v.b;
          imm = v.a;
          op = v.op == OP_CMP_LT ? OP_CMP_GT : v.op == OP_CMP_LE ? OP_CMP_GE : v.op == OP_CMP_GT ? OP_CMP_LT : v.op == OP_CMP_GE ? OP_CMP_LE : v.op;
        }
        if (imm.kind != OPD_IMM || P.imms[imm.idx].is_null) return false;
        Operand c64 = col;
        c64.vk = VK_I64;
        if (!int_col(c64, &f.off, &f.w, false)) return false;
        if (P.cols[col.idx].phys == PH_DEC128) f.w = 16;
        f.op = op;
        f.imm = (int64_t)P.imms[imm.idx].lo;
        F.n_filters++;
        break;
      }
      case OP_DEC_MUL_LIT_MINUS: case OP_DEC_MUL_LIT_PLUS: case OP_MUL: {
        if (v.op == OP_MUL && v.t != VK_I128) return false;
        if (F.n_prod >= 2 || v.dst.kind != OPD_REG) return false;
        FusedProd& q = F.p[F.n_prod];
        q.kind = v.op == OP_DEC_MUL_LIT_MINUS ? 0 : v.op == OP_DEC_MUL_LIT_PLUS ? 1 : 2;
        if (v.a.kind == OPD_REG && F.n_prod == 1 && (int)v.a.idx == prod_reg[0]) {
          q.a_src = 1;
        } else if (!int_col(v.a, &q.a_off, &q.a_w, true)) {
          return false;
        }
        if (!int_col(v.b, &q.b_off, &q.b_w, true)) return false;
        if (q.kind != 2) {
          q.lit_lo = P.imms[v.imm].lo;
          q.lit_hi = P.imms[v.imm].hi;
        }
        prod_reg[F.n_prod++] = v.dst.idx;
        break;
      }
      case OP_STR_PACK8: {
        if (v.a.kind != OPD_COL || P.cols[v.a.idx].phys != PH_UTF8 || P.cols[v.a.idx].valid || v.dst.kind != OPD_REG) return false;
        PackInfo pi;
        pi.reg = v.dst.idx;
        memset(&pi.k, 0, sizeof pi.k);
        if (prepacked[v.a.idx]) {  // the image is already in the tile: an integer key column of width 4
          pi.k.kind = 0;
          pi.k.off = fused_off[v.a.idx];
          pi.k.w = 4;
          packs.push_back(pi);
          break;
        }
        pi.k.kind = 1;
        pi.k.off = fused_off[v.a.idx];
        pi.k.chars = P.cols[v.a.idx].chars;
        pi.k.offsets = (const int32_t*)P.cols[v.a.idx].data;
        pi.k.max_len = v.aux;
        pi.k.shift = (uint8_t)v.imm;
        pi.k.w = (pi.k.shift == 24 && pi.k.max_len <= 3) ? 4 : 8;
        packs.push_back(pi);
        break;
      }
      case OP_MADD_I64: {
        if (v.a.kind != OPD_REG || v.b.kind != OPD_REG || v.dst.kind != OPD_REG || P.imms[v.imm].lo != 4294967296ull) return false;
        combined_reg = v.dst.idx;
        comb_a = v.a.idx;
        comb_b = v.b.idx;
        break;
      }
      default: return false;
    }
  }
  // keys
  F.n_keys = P.n_keys;
  if (P.n_keys > 2) return false;
  if (P.n_keys > 0 && !P.keys_all_i64) return false;
  auto key_from = [&](const Operand& o, FusedKey& k) -> bool {
    if (o.kind == OPD_REG) {
      for (auto& pi : packs)
        if (pi.reg == (int)o.idx) {
          k = pi.k;
          return true;
        }
      return false;
    }
    if (o.kind == OPD_COL) {
      memset(&k, 0, sizeof k);
      uint32_t off;
      uint8_t w;
      Operand c64 = o;
      c64.vk = VK_I64;
      if (!int_col(c64, &off, &w, false) || P.cols[o.idx].phys == PH_DEC128) return false;
      k.kind = 0;
      k.off = off;
      k.w = w;
      return true;
    }
    return false;
  };
  for (int k = 0; k < P.n_keys; k++)
    if (!key_from(P.keys[k], F.k[k])) return false;
  if (P.n_keys == 1) {
    if (!(P.key_hash.kind == P.keys[0].kind && P.key_hash.idx == P.keys[0].idx)) return false;
    F.combine = 0;
  } else if (P.n_keys == 2) {
    // only the all-packed-string form: the 32-bit images are the pack registers themselves
    if (P.key_hash.kind != OPD_REG || (int)P.key_hash.idx != combined_reg) return false;
    if (!(P.keys[0].kind == OPD_REG && P.keys[1].kind == OPD_REG && comb_a == (int)P.keys[0].idx && comb_b == (int)P.keys[1].idx)) return false;
    F.combine = 1;
  }
  if (combined_reg >= 0 && P.n_keys != 2) return false;
  // accumulators
  if (P.n_acc > VM_REG_ACC) return false;
  F.n_acc = P.n_acc;
  for (int a = 0; a < P.n_acc; a++) {
    const AccDesc& ad = P.acc[a];
    FusedAcc& fa = F.a[a];
    if (ad.kind == ACC_COUNT_STAR || (ad.kind == ACC_COUNT && !ad.nullable)) {
      fa.src = 3;
      continue;
    }
    if (ad.kind != ACC_SUM_I128 || ad.nullable) return false;
    if (ad.src.kind == OPD_REG) {
      if ((int)ad.src.idx == prod_reg[0]) fa.src = 1;
      else if ((int)ad.src.idx == prod_reg[1]) fa.src = 2;
      else return false;
    } else if (ad.src.kind == OPD_COL) {
      if (!int_col(ad.src, &fa.off, &fa.w, true)) return false;
      if (ad.src.vk != VK_I128 && P.cols[ad.src.idx].phys == PH_DEC128) return false;
      fa.src = 0;
    } else {
      return false;
    }
  }
  // every packed register must be a key (no stray uses)
  for (auto& pi : packs) {
    bool used = false;
    for (int k = 0; k < P.n_keys; k++) used |= P.keys[k].kind == OPD_REG && (int)P.keys[k].idx == pi.reg;
    if (!used) return false;
  }
  // the code-shaping part of the spec (program.h FusedShape)
  FusedShapeDesc d;
  memset(&d, 0, sizeof d);
  d.nf = F.n_filters;
  for (int i = 0; i < F.n_filters; i++) {
    d.fw[i] = F.f[i].w;
    d.fop[i] = (uint8_t)(F.f[i].op - OP_CMP_EQ);
  }
  d.nk = F.n_keys;
  for (int k = 0; k < F.n_keys; k++) {
    d.kkind[k] = F.k[k].kind;
    d.kw[k] = F.k[k].w;
  }
  d.combine = F.combine;
  d.np = F.n_prod;
  for (int j = 0; j < F.n_prod; j++) {
    d.pkind[j] = F.p[j].kind;
    d.pasrc[j] = F.p[j].a_src;
    d.paw[j] = F.p[j].a_w;
    d.pbw[j] = F.p[j].b_w;
  }
  d.na = F.n_acc;
  for (int a = 0; a < F.n_acc; a++) {
    d.asrc[a] = F.a[a].src;
    d.aw[a] = F.a[a].w;
  }
  FP.shape = fused_shape_encode(d);
  return true;
}

// Recognise scan -> integer/date/decimal compares against literals -> up to two decimal products -> one or two integer-like
// key COLUMNS -> COUNT / SUM accumulators in a lowered aggregate program: the shape the dedicated high-cardinality kernel
// (groupby.cu) runs without the tile VM.  Hash instructions of the general key path are ignored (the kernel hashes the
// key image itself).
bool match_groupby(const Program& P, GroupBySpec& S) {
  memset(&S, 0, sizeof S);
  if (getenv("B200_NO_GROUPBY")) return false;
  if (P.n_keys < 1 || P.n_keys > 2 || P.n_acc > GB_MAX_ACC || P.n_cols > FUSED_MAX_COLS || P.n_cols == 0) return false;
  for (int c = 0; c < P.n_cols; c++) {
    const ColDesc& cd = P.cols[c];
    if (cd.valid) return false;
    if (!(cd.phys == PH_I32 || cd.phys == PH_I64 || cd.phys == PH_U64 || cd.phys == PH_DEC128)) return false;
    S.cols[c].data = cd.data;
    S.cols[c].width = cd.width;
  }
  S.n_cols = P.n_cols;
  auto col_of = [&](const Operand& o, int* out) -> bool {
    if (o.kind != OPD_COL || o.idx >= (unsigned)P.n_cols) return false;
    *out = (int)o.idx;
    return true;
  };
  int prod_reg[2] = {-1, -1};
  for (int i = 0; i < P.n_instr; i++) {
    const VInstr& v = P.code[i];
    switch (v.op) {
      case OP_HASH:
      case OP_HASH_COMBINE: break;  // the general path's row hash: not needed
      case OP_CMP_EQ: case OP_CMP_NE: case OP_CMP_LT: case OP_CMP_LE: case OP_CMP_GT: case OP_CMP_GE: {
        if (!(v.flags & IF_FILTER) || (v.flags & IF_NULLCHK) || v.t != VK_I64 || v.aux == PH_U64) return false;
        if (S.n_filters >= FUSED_MAX_FILTERS) return false;
        Operand col = v.a, imm = v.b;
        uint8_t op = v.op;
        if (v.a.kind == OPD_IMM && v.b.kind == OPD_COL) {
          col = v.b;
          imm = v.a;
          op = v.op == OP_CMP_LT ? OP_CMP_GT : v.op == OP_CMP_LE ? OP_CMP_GE : v.op == OP_CMP_GT ? OP_CMP_LT : v.op == OP_CMP_GE ? OP_CMP_LE : v.op;
        }
        if (imm.kind != OPD_IMM || P.imms[imm.idx].is_null) return false;
        if (!col_of(col, &S.f_col[S.n_filters])) return false;
        S.f_op[S.n_filters] = (int)op - (int)OP_CMP_EQ;
        S.f_imm[S.n_filters] = (int64_t)P.imms[imm.idx].lo;
        S.n_filters++;
        break;
      }
      case OP_DEC_MUL_LIT_MINUS: case OP_DEC_MUL_LIT_PLUS: case OP_MUL: {
        if ((v.flags & IF_NULLCHK) || (v.op == OP_MUL && v.t != VK_I128)) return false;
        if (S.n_prod >= 2 || v.dst.kind != OPD_REG) return false;
        const int j = S.n_prod;
        S.p_kind[j] = v.op == OP_DEC_MUL_LIT_MINUS ? 0 : v.op == OP_DEC_MUL_LIT_PLUS ? 1 : 2;
        if (v.a.kind == OPD_REG && j == 1 && (int)v.a.idx == prod_reg[0]) S.p_a_src[j] = 1;
        else if (!col_of(v.a, &S.p_a_col[j])) return false;
        if (!col_of(v.b, &S.p_b_col[j])) return false;
        if (S.p_kind[j] != 2) {
          const uint64_t lo = P.imms[v.imm].lo, hi = P.imms[v.imm].hi;
          if (hi != (uint64_t)((int64_t)lo >> 63)) return false;
          S.p_lit[j] = (int64_t)lo;
        }
        prod_reg[S.n_prod++] = v.dst.idx;
        break;
      }
      default: return false;
    }
  }
  S.n_keys = P.n_keys;
  for (int k = 0; k < P.n_keys; k++) {
    if (!col_of(P.keys[k], &S.key_col[k])) return false;
    if (P.cols[S.key_col[k]].phys == PH_DEC128) return false;
  }
  S.n_acc = P.n_acc;
  for (int a = 0; a < P.n_acc; a++) {
    const AccDesc& ad = P.acc[a];
    if (ad.kind == ACC_COUNT_STAR || (ad.kind == ACC_COUNT && !ad.nullable)) {
      S.a_src[a] = 3;
      continue;
    }
    if (ad.kind != ACC_SUM_I128 || ad.nullable) return false;
    if (ad.src.kind == OPD_REG) {
      if ((int)ad.src.idx == prod_reg[0]) S.a_src[a] = 1;
      else if ((int)ad.src.idx == prod_reg[1]) S.a_src[a] = 2;
      else return false;
    } else if (col_of(ad.src, &S.a_col[a])) {
      S.a_src[a] = 0;
    } else {
      return false;
    }
  }
  S.n_rows = P.n_rows;
  S.table = P.table;
  return true;
}

// Recognise a materialising program that only FILTERS (comparisons of plain columns with literals or with each other,
// combined with AND / OR / NOT) and forwards plain columns: the shape the dedicated FilterExec kernel (filter.cu) runs
// without the tile VM.  LIKE, arithmetic, casts, NULL-aware compares or computed outputs keep the VM.
bool match_fast_filter(const Program& P, FastFilterSpec& S) {
  if (P.sink != SINK_MATERIALIZE || getenv("B200_NO_FASTFILTER")) return false;
  if (P.n_cols > FF_MAX_COLS || P.n_cols == 0 || P.n_instr > FF_MAX_OPS || P.n_instr == 0 || P.n_imms > FF_MAX_IMMS || P.n_out > FF_MAX_OUT || P.n_regs > 64) return false;
  memset(&S, 0, sizeof S);
  auto int_phys = [](uint8_t ph) { return ph == PH_I8 || ph == PH_I16 || ph == PH_I32 || ph == PH_I64 || ph == PH_U8 || ph == PH_U16 || ph == PH_U32 || ph == PH_U64; };
  for (int c = 0; c < P.n_cols; c++) {
    const ColDesc& cd = P.cols[c];
    if (cd.valid) return false;
    if (!(int_phys(cd.phys) || cd.phys == PH_DEC128 || cd.phys == PH_UTF8 || cd.phys == PH_STRVIEW || cd.phys == PH_F64 || cd.phys == PH_F32 || cd.phys == PH_BOOL8)) return false;
    S.cols[c].data = cd.data;
    S.cols[c].chars = cd.chars;
    S.cols[c].phys = cd.phys;
    S.cols[c].width = cd.width;
  }
  S.n_cols = P.n_cols;
  for (int i = 0; i < P.n_imms; i++) {
    S.imms[i].lo = P.imms[i].lo;
    S.imms[i].hi = P.imms[i].hi;
  }
  auto bool_reg = [&](const Operand& o, uint8_t* out) {
    if (o.kind != OPD_REG || o.vk != VK_BOOL || o.idx >= 64) return false;
    *out = (uint8_t)o.idx;
    return true;
  };
  bool any_filter = false;
  for (int i = 0; i < P.n_instr; i++) {
    const VInstr& v = P.code[i];
    FfOp& op = S.ops[S.n_ops];
    memset(&op, 0, sizeof op);
    if (v.flags & IF_NULLCHK) return false;
    switch (v.op) {
      case OP_CMP_EQ: case OP_CMP_NE: case OP_CMP_LT: case OP_CMP_LE: case OP_CMP_GT: case OP_CMP_GE: {
        op.kind = FF_CMP;
        op.cmp = (uint8_t)(v.op - OP_CMP_EQ);
        if (!(v.t == VK_I64 || v.t == VK_I128 || v.t == VK_STR)) return false;
        if (v.t == VK_STR && !(v.op == OP_CMP_EQ || v.op == OP_CMP_NE)) return false;
        bool wide = v.t == VK_I128;
        const Operand* ops2[2] = {&v.a, &v.b};
        uint8_t idx[2], is_imm[2];
        for (int k = 0; k < 2; k++) {
          const Operand& o = *ops2[k];
          if (o.kind == OPD_IMM) {
            if (o.idx >= (unsigned)P.n_imms || P.imms[o.idx].is_null) return false;
            idx[k] = (uint8_t)o.idx;
            is_imm[k] = 1;
          } else if (o.kind == OPD_COL) {
            if (o.idx >= (unsigned)P.n_cols) return false;
            const uint8_t ph = P.cols[o.idx].phys;
            if (v.t == VK_STR) {
              if (!(ph == PH_UTF8 || ph == PH_STRVIEW)) return false;
            } else {
              if (!(int_phys(ph) || ph == PH_DEC128)) return false;
              wide = wide || ph == PH_DEC128;
            }
            idx[k] = (uint8_t)o.idx;
            is_imm[k] = 0;
          } else {
            return false;
          }
        }
        op.a = idx[0];
        op.b = idx[1];
        op.a_imm = is_imm[0];
        op.b_imm = is_imm[1];
        op.vt = v.t == VK_STR ? 2 : (wide ? 1 : (v.aux == PH_U64 ? 3 : 0));
        if (wide && v.aux == PH_U64) return false;
        // a 64-bit immediate compared as 128 bits needs its sign extension in `hi`
        for (int k = 0; k < 2; k++)
          if (op.vt == 1 && is_imm[k] && v.t != VK_I128) S.imms[idx[k]].hi = (uint64_t)((int64_t)S.imms[idx[k]].lo >> 63);
        if (v.flags & IF_FILTER) op.filter = 1;
        else if (!bool_reg(v.dst, &op.dst)) return false;
        break;
      }
      case OP_AND:
      case OP_OR:
        op.kind = v.op == OP_AND ? FF_AND : FF_OR;
        if (!bool_reg(v.a, &op.a) || !bool_reg(v.b, &op.b) || !bool_reg(v.dst, &op.dst)) return false;
        break;
      case OP_NOT:
        op.kind = FF_NOT;
        if (!bool_reg(v.a, &op.a) || !bool_reg(v.dst, &op.dst)) return false;
        break;
      case OP_FILTER:
        op.kind = FF_FILTER_REG;
        op.filter = 1;
        if (!bool_reg(v.a, &op.a)) return false;
        break;
      default: return false;
    }
    any_filter = any_filter || op.filter;
    S.n_ops++;
  }
  if (!any_filter) return false;
  for (int j = 0; j < P.n_out; j++) {
    const OutCol& oc = P.out[j];
    if (oc.src.kind != OPD_COL || oc.src.idx >= (unsigned)P.n_cols || oc.valid) return false;
    const uint8_t ph = P.cols[oc.src.idx].phys;
    const bool str = ph == PH_UTF8 || ph == PH_STRVIEW;
    if (str ? oc.phys != PH_STRVIEW : (oc.phys != ph)) return false;
    S.out_col[j] = (uint8_t)oc.src.idx;
    S.out_data[j] = oc.data;
  }
  S.n_out = P.n_out;
  S.n_rows = P.n_rows;
  return true;
}

struct TableMem {
  AggTable T;
  std::vector<DevPtr> keep;
};

TableMem alloc_table(const Exec& x, uint64_t cap, int n_keys, const std::vector<AccDesc>& accs) {
  TableMem tm;
  memset(&tm.T, 0, sizeof tm.T);
  // one allocation: [n_groups | hash | state | lock | acc] -- the part a fresh table needs initialised -- then the keys
  auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
  const size_t nk = std::max<size_t>(1, (size_t)n_keys), na = std::max<size_t>(1, accs.size());
  const size_t o_hash = 256, o_state = o_hash + up(cap * 8), o_lock = o_state + up(cap * 4), o_acc = o_lock + up(cap * 4);
  const size_t o_keys = o_acc + up(na * cap * 16), o_kv = o_keys + up(nk * cap * 16), bytes = o_kv + up(nk * cap);
  DevPtr blk = dev_alloc(bytes, x.st());
  tm.keep.push_back(blk);
  uint8_t* const b = (uint8_t*)blk->ptr;
  tm.T.cap = cap;
  tm.T.n_groups = (unsigned int*)b;
  tm.T.hash = (unsigned long long*)(b + o_hash);
  tm.T.state = (unsigned int*)(b + o_state);
  tm.T.lock = (unsigned int*)(b + o_lock);
  tm.T.acc = (unsigned long long*)(b + o_acc);
  tm.T.keys = (unsigned long long*)(b + o_keys);
  tm.T.key_valid = (unsigned char*)(b + o_kv);
  AccKinds k;
  memset(&k, 0, sizeof k);
  k.n = (int)accs.size();
  bool zero_init = true;  // SUM / COUNT / AVG states start at 0; MIN / MAX start at the type's extreme
  for (size_t i = 0; i < accs.size(); i++) {
    k.kind[i] = accs[i].kind;
    zero_init &= accs[i].kind != ACC_MIN_I128 && accs[i].kind != ACC_MAX_I128 && accs[i].kind != ACC_MIN_F64 && accs[i].kind != ACC_MAX_F64;
  }
  if (zero_init) {
    CUDA_CHECK(cudaMemsetAsync(b, 0, o_keys, x.st()));
  } else {
    launch_agg_table_init(tm.T, k, x.st());
    x.count();
  }
  return tm;
}

typedef std::function<std::unique_ptr<PipelineBuilder>()> BuilderFactory;

// Largest aggregate output that a task may extract on the group count of its last run, before the count is read back
// (the output block is zeroed so that rows the extraction does not write are empty values, never stray pointers).
static const uint64_t SPEC_MAX_GROUPS = 4096;

DevBatchPtr run_aggregate(const Exec& x, const BuilderFactory& make_pb, const PlanNode& node, const DevBatchPtr& src, OpMetrics* met, int part) {
  const int n_keys = (int)node.group_by.size();
  if (n_keys > VM_MAX_KEYS) throw EngineError(B200_ERR_UNSUPPORTED, "too many group-by columns");
  // initial optimism about the keys
  int pack_mode = 0;
  {
    bool any_str = false, all_narrow = n_keys > 0;
    for (auto& g : node.group_by) {
      any_str |= g.expr->type.id == TypeId::Utf8;
      all_narrow &= narrowable(g.expr->type);
    }
    if (n_keys == 2 && all_narrow) pack_mode = 2;
    else if (any_str) pack_mode = 1;
  }
  int node_idx = -1;
  if (x.s) {
    auto it = x.s->metric_index.find(&node);
    if (it != x.s->metric_index.end()) node_idx = it->second;
  }
  const std::string hint_key = (x.s ? x.s->fingerprint : std::string("?")) + "#" + std::to_string(node_idx);
  const std::string spec_key = hint_key + "@" + std::to_string(part);
  int level = 0;
  bool had_hint = false;
  uint64_t groups_hint = 0;
  // a shape whose last run on this partition got its groups from the hinted sink at the first attempt: enqueue the extraction
  // for that many groups without waiting; the status and the group count are checked at the task's final synchronisation
  bool speculate = false;
  uint64_t spec_groups = 0;
  {
    std::lock_guard<std::mutex> g(x.e->mu);
    auto it = x.e->agg_hint.find(hint_key);
    if (it != x.e->agg_hint.end()) {
      level = it->second / 4;
      pack_mode = std::min(pack_mode, it->second % 4);
      had_hint = true;
      auto ig = x.e->agg_groups.find(hint_key);
      if (ig != x.e->agg_groups.end()) groups_hint = ig->second;
      auto is = x.e->agg_spec.find(spec_key);
      if (x.speculate && is != x.e->agg_spec.end()) {
        speculate = true;
        spec_groups = is->second;
      }
    }
  }
  const int hinted_level = had_hint ? level : -1;
  bool sampled = false;
  // strategy ladder: register sink (<= 4 groups) -> global table of growing capacity; packed keys -> plain keys
  std::unique_ptr<PipelineBuilder> pbp;
  AggLowered L;
  TableMem tm;
  RunOutcome ro;
  unsigned int n_groups = 0;
  bool gb_bailed = false, pf_off = false;
  int attempts = 0;
  for (;;) {
    attempts++;
    x.check_cancel();
    ScopeTimer t_iter("  agg: lower+alloc+launch+sync");
    pbp = make_pb();
    PipelineBuilder& pb = *pbp;
    L = AggLowered();
    lower_aggregate(pb, node, L, pack_mode);
    Program& P = pb.prog;
    P.n_keys = (uint8_t)n_keys;
    P.n_acc = (uint8_t)L.accs.size();
    for (int k = 0; k < n_keys; k++) P.keys[k] = pb.resolve(L.keys[(size_t)k]);
    for (size_t a = 0; a < L.accs.size(); a++) P.acc[a] = L.accs[a];
    memset(&P.key_hash, 0, sizeof P.key_hash);
    P.keys_all_i64 = L.fast ? 1 : 0;
    if (n_keys) {
      if (L.fast) {
        P.key_hash = pb.resolve(L.combined);
      } else {
        ColRef h = pb.hash_of(L.keys);
        P.key_hash = h.op;
      }
    }
    const bool reg_ok = (int)L.accs.size() <= VM_REG_ACC;
    if (!reg_ok && level == 0) level = 1;
    // up to a few million input rows a table sized for "every row its own group" is cheap: no capacity ladder
    const bool small_input = src->n <= ((int64_t)1 << 22);
    if (level > 0 && small_input) level = 8;
    uint64_t cap;
    int reg_groups = 0;
    if (level == 0) {
      P.sink = SINK_AGG_REG;
      reg_groups = n_keys ? VM_REG_GROUPS : 1;
      cap = n_keys ? 64 : 2;
    } else {
      P.sink = SINK_AGG_GLOBAL;
      if (!n_keys) cap = 2;
      else cap = std::min<uint64_t>(next_pow2((uint64_t)std::max<int64_t>(src->n, 1) * 2), (uint64_t)1 << std::min(40, 12 + 4 * level));
      // a plan shape seen before: size the table for the groups its tasks produced (x2.5: load factor <= 0.4 with room for a
      // somewhat larger sibling task) instead of the whole class -- the classes are 16x apart, and every slot costs ~80 bytes
      // of memset and of extraction scan.  An overflow falls back to the class size (level++ below leaves hinted_level).
      if (groups_hint && level == hinted_level && n_keys) cap = std::min(cap, std::max<uint64_t>(next_pow2(groups_hint * 5 / 2), 4096));
      if (cap < 16) cap = 16;
    }
    {
      ScopeTimer t_alloc("    agg: alloc_table");
      tm = alloc_table(x, cap, n_keys, L.accs);
    }
    P.table = tm.T;
    pb.finalize_layout((size_t)VM_REG_ACC * 512 * 16 + 256);
    if (level == 0) {
      const size_t hi_bytes = (size_t)x.e->sm_count * 512 * VM_REG_GROUPS * VM_REG_ACC * 8;
      DevPtr hi = dev_alloc(hi_bytes, x.st());
      tm.keep.push_back(hi);
      P.acc_hi = (unsigned long long*)hi->ptr;
    }
    // First sight of a large integer-keyed aggregate: group the first 16 K rows on the hash kernel to learn whether the
    // 4-group register sink can apply at all and which table class to start with, instead of discovering it by running
    // (and abandoning) full passes up the capacity ladder.
    if (!sampled && !had_hint && level == 0 && n_keys > 0 && src->n > ((int64_t)1 << 20)) {
      sampled = true;
      GroupBySpec probe;
      const int64_t sample_rows = 16384;
      TableMem stm = alloc_table(x, 65536, n_keys, L.accs);
      P.table = stm.T;
      if (match_groupby(P, probe)) {
        probe.n_rows = sample_rows;
        probe.pf_K = -1;
        unsigned int seen = 0;
        RunOutcome so = launch_program(x, pb, 0, nullptr, true, nullptr, stm.T.n_groups, &seen, &probe);
        if (!so.status.pack_overflow && (so.status.overflow || seen > (unsigned)VM_REG_GROUPS)) {
          level = (so.status.overflow || (int64_t)seen * 2 > sample_rows) ? 3 : 2;  // (nearly) every row its own group: 16 M slots; else 1 M
          continue;
        }
      }
      P.table = tm.T;
    }
    FusedPlan fspec;
    const bool use_fused = level == 0 && match_fused(P, fspec);
    GroupBySpec gspec;
    const bool use_gb = level > 0 && !gb_bailed && match_groupby(P, gspec);
    gspec.pf_K = pf_off ? -1 : 0;
    {
      ScopeTimer t_l("    agg: launch_program (incl. sync)");
      ro = launch_program(x, pb, reg_groups, use_fused ? &fspec : nullptr, !speculate, met, tm.T.n_groups, &n_groups, use_gb ? &gspec : nullptr);
    }
    if (met) met->launches += 2;
    if (speculate) {
      const RunStatus* hs = ro.deferred;
      const unsigned int* hg = ro.deferred_extra;
      x.defer([hs, hg, spec_groups]() {
        if (hs->overflow || hs->pack_overflow || *hg != spec_groups) throw SpeculationMiss();
      });
      n_groups = (unsigned int)spec_groups;
      break;
    }
    if (ro.status.pack_overflow && use_gb) {
      gb_bailed = true;  // operands outside the dedicated kernel's ranges: same table size on the general sink
      continue;
    }
    if (ro.status.pack_overflow) {
      pack_mode = pack_mode == 2 ? 1 : 0;
      continue;
    }
    if (!ro.status.overflow) break;
    if (level > 0 && cap >= next_pow2((uint64_t)std::max<int64_t>(src->n, 1) * 2)) {
      if (use_gb && !pf_off) {
        pf_off = true;  // a bucket's region of the partitioned table filled up (skewed buckets): same table, unpartitioned
        continue;
      }
      throw EngineError(B200_ERR_EXECUTION, "aggregate hash table overflow");
    }
    level++;
  }
  if (!speculate) {
    // remember the smallest table class that holds this many groups (not the level that happened to be used: a small
    // input jumps straight to a table sized for its row count)
    int learnt = level;
    if (level > 0) {
      learnt = 1;
      while (learnt < 7 && ((uint64_t)1 << (12 + 4 * learnt)) < (uint64_t)n_groups * 2) learnt++;
    }
    std::lock_guard<std::mutex> g(x.e->mu);
    x.e->agg_hint[hint_key] = learnt * 4 + pack_mode;
    uint64_t& gh = x.e->agg_groups[hint_key];
    gh = std::max<uint64_t>(gh, n_groups);
    if (attempts == 1 && n_groups <= SPEC_MAX_GROUPS) x.e->agg_spec[spec_key] = n_groups;
    else x.e->agg_spec.erase(spec_key);
  }
  PipelineBuilder& pb = *pbp;
  // extraction
  ScopeTimer t_ex("  agg: extract");
  auto out = std::make_shared<DevBatch>();
  out->n = n_groups;
  AggExtractArgs A;
  memset(&A, 0, sizeof A);
  if (L.outs.size() > (size_t)VM_MAX_OUT) throw EngineError(B200_ERR_UNSUPPORTED, "too many aggregate output columns");
  A.n_out = (int)L.outs.size();
  A.n_keys = n_keys;
  // one block for the counter words and every output buffer: cleared as a whole when the group count is speculated, so
  // that rows the extraction leaves unwritten hold empty values (never stray string pointers) until the task's check
  const size_t rows = std::max<unsigned int>(n_groups, 1);
  auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
  struct Place { size_t data = 0, valid = 0, aux = 0; };
  std::vector<Place> place(L.outs.size());
  size_t blk_bytes = 256;
  for (size_t j = 0; j < L.outs.size(); j++) {
    const auto& r = L.outs[j];
    place[j].data = blk_bytes;
    blk_bytes += up(rows * phys_width(r.phys));
    if (r.with_valid) {
      place[j].valid = blk_bytes;
      blk_bytes += up(rows);
    }
    if (r.kind == AO_KEY_PACKED) {
      place[j].aux = blk_bytes;
      blk_bytes += up(rows * 8);
    }
  }
  DevPtr blk = dev_alloc(blk_bytes, x.st());
  uint8_t* const base = (uint8_t*)blk->ptr;
  CUDA_CHECK(cudaMemsetAsync(base, 0, speculate ? blk_bytes : 16, x.st()));
  A.counter = (unsigned long long*)base;
  A.error = (unsigned int*)(base + 8);
  A.cap = n_groups;
  uint64_t wbytes = 0;
  for (size_t j = 0; j < L.outs.size(); j++) {
    const auto& r = L.outs[j];
    DevColumn oc;
    oc.name = r.name;
    oc.type = r.type;
    oc.phys = r.phys;
    oc.n = n_groups;
    oc.data = base + place[j].data;
    if (r.with_valid) oc.valid = base + place[j].valid;
    oc.nullable = r.with_valid;
    oc.keep.push_back(blk);
    if (r.key_idx >= 0) {
      for (auto& k : L.keys[(size_t)r.key_idx].keep) oc.keep.push_back(k);
      if (r.phys == PH_STRVIEW) {
        for (auto& sc : src->cols)
          for (auto& k : sc.keep) oc.keep.push_back(k);
        for (auto& k : pb.keep) oc.keep.push_back(k);
      }
    }
    AggOut& o = A.out[j];
    o.data = (void*)oc.data;
    o.valid = (uint8_t*)oc.valid;
    o.aux = r.kind == AO_KEY_PACKED ? base + place[j].aux : nullptr;
    o.kind = r.kind;
    o.a = r.a;
    o.b = r.b;
    o.phys = r.phys;
    o.imm = r.imm;
    wbytes += (uint64_t)oc.width() * n_groups;
    out->cols.push_back(oc);
  }
  launch_agg_extract(tm.T, A, x.st());
  x.count();
  {
    // the extraction's overflow flag (decimal AVG / SUM precision) only has to be seen before the task returns
    const unsigned int* herr = x.fetch<unsigned int>(A.error);
    x.defer([herr, blk]() {
      if (*herr) throw EngineError(B200_ERR_EXECUTION, "Arithmetic overflow");
    });
  }
  for (size_t c = 0; c < out->cols.size() && c < node.schema.size(); c++) out->cols[c].name = node.schema[c].name;
  if (met) {
    met->bytes_read += source_bytes(pb);
    met->bytes_written += wbytes;
    met->input_rows += (uint64_t)src->n;
  }
  return out;
}

// ------------------------------------------------------------------------------------------------
// Operator tree execution
// ------------------------------------------------------------------------------------------------
struct Runner {
  Exec x;
  std::string job;

  int n_partitions(const PlanNode& n) {
    switch (n.op) {
      case PlanNode::Scan: {
        std::lock_guard<std::mutex> g(x.e->mu);
        auto it = x.e->tables.find(n.table);
        if (it == x.e->tables.end()) throw EngineError(B200_ERR_INVALID, "table not registered: " + n.table);
        return it->second.empty() ? 0 : it->second.rbegin()->first + 1;
      }
      case PlanNode::ShuffleReader: {
        std::lock_guard<std::mutex> g(x.e->mu);
        int mx = 0;
        for (auto& kv : x.e->shuffle)
          if (kv.first.job == job && kv.first.stage == n.reader_stage_id) mx = std::max(mx, (int)kv.first.part + 1);
        return mx;
      }
      case PlanNode::SortPreservingMerge: return 1;
      case PlanNode::Passthrough:
        if (n.op_name == "CoalescePartitionsExec") return 1;
        return n_partitions(*n.children[0]);
      case PlanNode::HashJoin: return n_partitions(*n.children[1]);
      default: return n_partitions(*n.children[0]);
    }
  }

  // Whether partition 0 of `n` is a single run of rows in the order its producer wrote them: false when a shuffle
  // reader (possibly under row-preserving operators) concatenates several map outputs, each sorted on its own.
  bool one_run(const PlanNode& n) {
    switch (n.op) {
      case PlanNode::ShuffleReader: {
        std::lock_guard<std::mutex> g(x.e->mu);
        auto it = x.e->shuffle.find(ShuffleKey{job, n.reader_stage_id, 0});
        int pieces = 0;
        if (it != x.e->shuffle.end())
          for (auto& p : it->second) pieces += p.r1 > p.r0 ? 1 : 0;
        return pieces <= 1;
      }
      case PlanNode::Passthrough:
        if (n.op_name == "CoalescePartitionsExec" && n_partitions(*n.children[0]) != 1) return false;
        return one_run(*n.children[0]);
      case PlanNode::Filter:
      case PlanNode::Projection:
      case PlanNode::Limit: return one_run(*n.children[0]);
      default: return true;
    }
  }

  DevBatchPtr concat(const std::vector<DevBatchPtr>& parts, const Schema& schema) {
    std::vector<std::pair<DevBatchPtr, std::pair<int64_t, int64_t>>> v;
    for (auto& p : parts) v.push_back({p, {0, p->n}});
    return concat_slices(v, schema);
  }

  DevBatchPtr concat_slices(const std::vector<std::pair<DevBatchPtr, std::pair<int64_t, int64_t>>>& parts, const Schema& schema) {
    auto out = std::make_shared<DevBatch>();
    int64_t total = 0;
    for (auto& p : parts) total += p.second.second - p.second.first;
    out->n = total;
    if (parts.size() == 1) {
      const DevBatch& b = *parts[0].first;
      for (auto& c : b.cols) out->cols.push_back(slice_column(c, parts[0].second.first, parts[0].second.second));
      return out;
    }
    // few rows (the tail of a query, reduce side of a small shuffle): all copies in one kernel launch
    const bool batched = total <= 65536;
    PackList pl;
    for (size_t ci = 0; ci < schema.size(); ci++) {
      bool any_valid = false;
      for (auto& p : parts) any_valid |= p.first->cols[ci].valid != nullptr;
      const DataType& t = schema[ci].type;
      Phys ph = t.id == TypeId::Utf8 ? PH_STRVIEW : phys_of(t);
      DevColumn oc = make_out_column(schema[ci].name, t, ph, total, any_valid, x.st());
      oc.n = total;
      int64_t pos = 0;
      for (auto& p : parts) {
        int64_t r0 = p.second.first, r1 = p.second.second, n = r1 - r0;
        if (n == 0) continue;
        DevColumn sc = slice_column(p.first->cols[ci], r0, r1);
        if (sc.type != t) throw EngineError(B200_ERR_INVALID, "concat: type mismatch in column " + schema[ci].name);
        if (batched && sc.phys == PH_UTF8) {
          // offsets + characters -> views, straight into the concatenated column (no temporary, no extra launch)
          pl.utf8_views(sc, (uint8_t*)oc.data + pos * oc.width());
          if (any_valid) {
            if (sc.valid) pl.copy(sc.valid, (uint8_t*)oc.valid + pos, (uint64_t)n);
            else CUDA_CHECK(cudaMemsetAsync((uint8_t*)oc.valid + pos, 1, (size_t)n, x.st()));
          }
          for (auto& k : sc.keep) oc.keep.push_back(k);
          pos += n;
          continue;
        }
        DevColumn v = as_views(x, sc);
        if (batched) pl.copy(v.data, (uint8_t*)oc.data + pos * oc.width(), (uint64_t)n * oc.width());
        else CUDA_CHECK(cudaMemcpyAsync((uint8_t*)oc.data + pos * oc.width(), v.data, (size_t)n * oc.width(), cudaMemcpyDeviceToDevice, x.st()));
        if (any_valid) {
          if (v.valid && batched) pl.copy(v.valid, (uint8_t*)oc.valid + pos, (uint64_t)n);
          else if (v.valid) CUDA_CHECK(cudaMemcpyAsync((uint8_t*)oc.valid + pos, v.valid, (size_t)n, cudaMemcpyDeviceToDevice, x.st()));
          else CUDA_CHECK(cudaMemsetAsync((uint8_t*)oc.valid + pos, 1, (size_t)n, x.st()));
        }
        if (ph == PH_STRVIEW)
          for (auto& k : v.keep) oc.keep.push_back(k);
        pos += n;
      }
      out->cols.push_back(oc);
    }
    pl.run(x);
    return out;
  }

  DevBatchPtr empty_batch(const Schema& s) {
    auto out = std::make_shared<DevBatch>();
    for (auto& f : s) {
      Phys ph = f.type.id == TypeId::Utf8 ? PH_STRVIEW : phys_of(f.type);
      DevColumn c = make_out_column(f.name, f.type, ph, 0, false, x.st());
      c.n = 0;
      out->cols.push_back(c);
    }
    return out;
  }

  DevBatchPtr exec_all(const PlanNode& n) {
    int np = n_partitions(n);
    std::vector<DevBatchPtr> parts;
    for (int p = 0; p < np; p++) parts.push_back(exec(n, p));
    if (parts.empty()) return empty_batch(n.schema);
    return concat(parts, n.schema);
  }

  // Walk down a Filter/Projection chain; returns the base node and the chain (top-down order).
  const PlanNode* chain_base(const PlanNode& top, std::vector<const PlanNode*>& chain) {
    const PlanNode* cur = &top;
    while (cur->op == PlanNode::Filter || cur->op == PlanNode::Projection ||
           (cur->op == PlanNode::Passthrough && cur->op_name != "CoalescePartitionsExec")) {
      if (cur->op == PlanNode::Filter && cur->fetch >= 0) break;
      if (cur->op != PlanNode::Passthrough) chain.push_back(cur);
      cur = cur->children[0].get();
    }
    return cur;
  }

  void apply_chain(PipelineBuilder& pb, const std::vector<const PlanNode*>& chain) {
    for (size_t i = chain.size(); i-- > 0;) {
      const PlanNode* n = chain[i];
      if (n->op == PlanNode::Filter) {
        pb.apply_filter(*n->predicate);
        if (n->has_projection) pb.apply_select(n->projection);
      } else {
        pb.apply_projection(n->exprs);
      }
    }
  }

  // Executes `top` (a Filter/Projection chain over some base) fused into one pipeline whose sink is
  // decided by the caller through `finish`.
  // Executes `top` (a Filter/Projection chain over some base) fused into one pipeline whose sink is
  // decided by the caller through `finish(make_builder, src)`; make_builder() returns a fresh
  // builder over `src` with the chain applied (sinks that retry with another lowering call it again).
  template <class F>
  DevBatchPtr with_chain(const PlanNode& top, int part, bool all_parts, F&& finish) {
    std::vector<const PlanNode*> chain;
    const PlanNode* base = chain_base(top, chain);
    DevBatchPtr src = all_parts ? exec_all(*base) : exec(*base, part);
    for (auto* n : chain)
      if (OpMetrics* m = x.m(n)) m->input_rows += (uint64_t)src->n;
    BuilderFactory make_pb = [&]() {
      std::unique_ptr<PipelineBuilder> pb(new PipelineBuilder(*src, x.st()));
      apply_chain(*pb, chain);
      return pb;
    };
    return finish(make_pb, src);
  }

  std::vector<ColRef> named_cols(PipelineBuilder& pb, const Schema& schema) {
    std::vector<ColRef> outs = pb.cols;
    for (size_t i = 0; i < outs.size() && i < schema.size(); i++) outs[i].name = schema[i].name;
    return outs;
  }

  // B200_TIMING=1: inclusive host wall time per operator (launch + synchronisation overheads)
  DevBatchPtr exec(const PlanNode& n, int part) {
    static const bool timing = getenv("B200_TIMING") != nullptr;
    if (!timing) return exec_impl(n, part);
    const auto t0 = std::chrono::steady_clock::now();
    const uint64_t l0 = x.e->launches;
    DevBatchPtr out = exec_impl(n, part);
    cudaStreamSynchronize(x.st());
    const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    fprintf(stderr, "[b200-time] op=%d part=%d rows_out=%lld host_ms=%.3f launches=%llu\n", (int)n.op, part, (long long)(out ? out->n : -1), ms,
            (unsigned long long)(x.e->launches - l0));
    return out;
  }
  DevBatchPtr exec_impl(const PlanNode& n, int part) {
    x.check_cancel();
    OpMetrics* met = x.m(&n);
    DevBatchPtr out;
    switch (n.op) {
      case PlanNode::Scan: {
        std::lock_guard<std::mutex> g(x.e->mu);
        auto it = x.e->tables.find(n.table);
        if (it == x.e->tables.end()) throw EngineError(B200_ERR_INVALID, "table not registered: " + n.table);
        auto pit = it->second.find(part);
        if (pit == it->second.end()) {
          out = empty_batch(n.schema);
          break;
        }
        out = std::make_shared<DevBatch>();
        out->n = pit->second->n;
        for (size_t k = 0; k < n.scan_projection.size(); k++) {
          int idx = n.scan_projection[k];
          if ((size_t)idx >= pit->second->cols.size()) throw EngineError(B200_ERR_INVALID, "scan projection out of range for " + n.table);
          DevColumn c = pit->second->cols[(size_t)idx];
          if (c.type != n.schema[k].type)
            throw EngineError(B200_ERR_INVALID, "scan: column " + n.schema[k].name + " has type " + c.type.str() + ", plan says " + n.schema[k].type.str());
          c.name = n.schema[k].name;
          out->cols.push_back(c);
        }
        break;
      }
      case PlanNode::ShuffleReader: {
        std::vector<std::pair<DevBatchPtr, std::pair<int64_t, int64_t>>> pieces;
        {
          std::lock_guard<std::mutex> g(x.e->mu);
          auto it = x.e->shuffle.find(ShuffleKey{job, n.reader_stage_id, n.broadcast ? 0 : part});
          if (it != x.e->shuffle.end())
            for (auto& p : it->second)
              if (p.r1 > p.r0) pieces.push_back({p.batch, {p.r0, p.r1}});
        }
        if (pieces.empty()) out = empty_batch(n.schema);
        else out = concat_slices(pieces, n.schema);
        for (size_t c = 0; c < out->cols.size() && c < n.schema.size(); c++) {
          if (out->cols[c].type != n.schema[c].type)
            throw EngineError(B200_ERR_INVALID, "shuffle reader: column " + n.schema[c].name + " has type " + out->cols[c].type.str() + ", plan says " + n.schema[c].type.str());
          out->cols[c].name = n.schema[c].name;
        }
        break;
      }
      case PlanNode::Filter:
      case PlanNode::Projection: {
        if (n.op == PlanNode::Filter && n.fetch >= 0) {
          // FilterExec { fetch } (datafusion.proto:1027-1034): the first `fetch` rows that pass, in input order -- the
          // materialising sinks keep the input order, so the prefix of the filtered batch is exactly that
          std::vector<const PlanNode*> chain;
          chain.push_back(&n);
          const PlanNode* base = chain_base(*n.children[0], chain);
          DevBatchPtr src = exec(*base, part);
          for (auto* c : chain)
            if (OpMetrics* m = x.m(c)) m->input_rows += (uint64_t)src->n;
          PipelineBuilder pb(*src, x.st());
          apply_chain(pb, chain);
          DevBatchPtr all = run_materialize(x, pb, named_cols(pb, n.schema), src, met);
          const int64_t keep = std::min<int64_t>(all->n, n.fetch);
          out = std::make_shared<DevBatch>();
          out->n = keep;
          for (auto& c : all->cols) out->cols.push_back(slice_column(c, 0, keep));
          break;
        }
        out = with_chain(n, part, false, [&](const BuilderFactory& mk, DevBatchPtr& src) {
          auto pb = mk();
          return run_materialize(x, *pb, named_cols(*pb, n.schema), src, met);
        });
        break;
      }
      case PlanNode::Aggregate: {
        const PlanNode& child = *n.children[0];
        bool all = (n.agg_mode == AggMode::Final || n.agg_mode == AggMode::Single) && part == 0 && n_partitions(child) > 1;
        out = with_chain(child, part, all, [&](const BuilderFactory& mk, DevBatchPtr& src) { return run_aggregate(x, mk, n, src, met, part); });
        break;
      }
      case PlanNode::HashJoin:
        out = exec_join(n, part, met);
        if (!n.sort_keys.empty()) out = do_sort(n.sort_keys, -1, out, met);  // SortMergeJoinExec: ordered by the join keys
        break;
      case PlanNode::Sort: {
        DevBatchPtr in = exec(*n.children[0], part);
        out = do_sort(n.sort_keys, n.fetch, in, met);
        break;
      }
      case PlanNode::SortPreservingMerge: {
        const PlanNode& child = *n.children[0];
        if (n_partitions(child) == 1 && one_run(child)) {
          // one sorted input: the merge passes it through (DataFusion's SortPreservingMergeExec over one partition)
          DevBatchPtr in = exec(child, 0);
          if (met) met->input_rows += (uint64_t)in->n;
          const int64_t m = n.fetch >= 0 ? std::min<int64_t>(n.fetch, in->n) : in->n;
          if (m == in->n) {
            out = in;
            break;
          }
          out = std::make_shared<DevBatch>();
          out->n = m;
          for (auto& c : in->cols) out->cols.push_back(slice_column(c, 0, m));
          break;
        }
        DevBatchPtr in = exec_all(child);
        out = do_sort(n.sort_keys, n.fetch, in, met);
        break;
      }
      case PlanNode::Passthrough:
        out = (n.op_name == "CoalescePartitionsExec") ? exec_all(*n.children[0]) : exec(*n.children[0], part);
        break;
      case PlanNode::Limit: {
        DevBatchPtr in = (n.op_name == "GlobalLimitExec") ? exec_all(*n.children[0]) : exec(*n.children[0], part);
        int64_t r0 = std::min<int64_t>(std::max<int64_t>(0, n.skip), in->n);
        int64_t r1 = n.fetch >= 0 ? std::min<int64_t>(in->n, r0 + n.fetch) : in->n;
        out = std::make_shared<DevBatch>();
        out->n = r1 - r0;
        for (auto& c : in->cols) out->cols.push_back(slice_column(c, r0, r1));
        break;
      }
      case PlanNode::ShuffleWriter: throw EngineError(B200_ERR_INVALID, "nested ShuffleWriterExec");
    }
    if (met) met->output_rows += (uint64_t)out->n;
    return out;
  }

  // ---- sort -----------------------------------------------------------------------------------
  DevBatchPtr do_sort(const std::vector<SortKey>& keys, int64_t fetch, DevBatchPtr in, OpMetrics* met) {
    const int64_t n = in->n;
    auto t0 = std::chrono::steady_clock::now();
    // key columns: plain column references are used in place, anything else is computed first
    std::vector<DevColumn> kcols;
    bool need_eval = false;
    for (auto& k : keys) need_eval |= k.expr->kind != Expr::Col;
    DevBatchPtr work = in;
    size_t n_in_cols = in->cols.size();
    if (need_eval && n > 0) {
      PipelineBuilder pb(*in, x.st());
      std::vector<ColRef> outs = pb.cols;
      for (auto& k : keys) {
        ColRef c = pb.compile(*k.expr);
        pb.pin(c);
        outs.push_back(c);
      }
      work = run_materialize(x, pb, outs, in, met);
      for (size_t k = 0; k < keys.size(); k++) kcols.push_back(work->cols[n_in_cols + k]);
    } else {
      for (auto& k : keys) kcols.push_back(in->cols.at((size_t)(k.expr->kind == Expr::Col ? k.expr->col : 0)));
    }
    if (n <= 1 || keys.empty()) {
      auto out = std::make_shared<DevBatch>();
      int64_t m = fetch >= 0 ? std::min<int64_t>(fetch, n) : n;
      out->n = m;
      for (size_t c = 0; c < n_in_cols; c++) out->cols.push_back(slice_column(in->cols[c], 0, m));
      return out;
    }
    if (n >= ((int64_t)1 << 32)) throw EngineError(B200_ERR_UNSUPPORTED, "sort of more than 2^32 rows");
    if (n <= SMALL_SORT_MAX_ROWS && keys.size() <= (size_t)SMALL_SORT_MAX_KEYS) {
      // the tail of a query (ORDER BY over a few groups): one comparison-sort launch, no length read-backs
      SmallSortKeys K;
      K.n_keys = (int)keys.size();
      std::vector<DevColumn> kv;  // keeps the view buffers alive until the launch is enqueued
      for (size_t ki = 0; ki < keys.size(); ki++) {
        kv.push_back(as_views(x, kcols[ki]));
        const DevColumn& kc = kv.back();
        SortWordArgs& A = K.k[ki];
        A.data = kc.data;
        A.valid = kc.valid;
        A.phys = kc.phys;
        A.asc = keys[ki].asc;
        A.nulls_first = keys[ki].nulls_first;
        A.word = 0;
      }
      DevPtr idx = dev_alloc((size_t)n * 8, x.st());
      launch_small_sort(K, (int64_t*)idx->ptr, n, x.st());
      x.count();
      const int64_t m = fetch >= 0 ? std::min<int64_t>(fetch, n) : n;
      DevBatch proj;
      proj.n = n;
      for (size_t c = 0; c < n_in_cols; c++) proj.cols.push_back(in->cols[c]);
      DevBatchPtr out = gather_batch(x, proj, (const int64_t*)idx->ptr, m, false);
      if (met) {
        met->elapsed_ns += (uint64_t)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t0).count();
        met->input_rows += (uint64_t)n;
      }
      return out;
    }
    const uint32_t n_blocks = (uint32_t)((n + 2047) / 2048);
    DevPtr ka = dev_alloc((size_t)n * 8, x.st()), kb = dev_alloc((size_t)n * 8, x.st());
    DevPtr va = dev_alloc((size_t)n * 4, x.st()), vb = dev_alloc((size_t)n * 4, x.st());
    DevPtr hist = dev_alloc((size_t)256 * n_blocks * 4 + 64, x.st());
    DevPtr scan = dev_alloc(((size_t)256 * n_blocks + 1 + (size_t)(256 * n_blocks) / 1024 + 8) * 8, x.st());
    uint32_t* perm = (uint32_t*)va->ptr;
    uint32_t* perm_alt = (uint32_t*)vb->ptr;
    launch_iota_u32(perm, n, x.st());
    x.count();
    for (size_t ki = keys.size(); ki-- > 0;) {
      DevColumn kc = as_views(x, kcols[ki]);
      int n_words = 1;
      if (kc.phys == PH_DEC128) n_words = 2;
      if (kc.phys == PH_STRVIEW) {
        DevPtr mx = dev_alloc(16, x.st());
        CUDA_CHECK(cudaMemsetAsync(mx->ptr, 0, 16, x.st()));
        launch_max_view_len((const unsigned long long*)kc.data, kc.valid, n, (unsigned int*)mx->ptr, x.st());
        x.count();
        unsigned int maxlen = x.get<unsigned int>(mx->ptr);
        n_words = (int)(maxlen / 7) + 1;
      }
      // least significant word first; the NULL-rank word is the most significant
      for (int w = n_words - 1; w >= (kc.valid ? -1 : 0); w--) {
        x.check_cancel();
        SortWordArgs A;
        A.data = kc.data;
        A.valid = kc.valid;
        A.phys = kc.phys;
        A.asc = keys[ki].asc;
        A.nulls_first = keys[ki].nulls_first;
        A.word = w;
        uint64_t* kin = (uint64_t*)ka->ptr;
        launch_sort_word(A, perm, kin, n, x.st());
        x.count();
        bool in_a;
        uint64_t ln = 0;
        if (perm == (uint32_t*)va->ptr) {
          radix_sort_pairs_u64((uint64_t*)ka->ptr, (uint32_t*)va->ptr, (uint64_t*)kb->ptr, (uint32_t*)vb->ptr, n, (uint32_t*)hist->ptr, (uint64_t*)scan->ptr, x.st(), &in_a, &ln);
          perm = in_a ? (uint32_t*)va->ptr : (uint32_t*)vb->ptr;
        } else {
          // current permutation lives in vb: sort with roles swapped (keys were written to ka)
          radix_sort_pairs_u64((uint64_t*)ka->ptr, (uint32_t*)vb->ptr, (uint64_t*)kb->ptr, (uint32_t*)va->ptr, n, (uint32_t*)hist->ptr, (uint64_t*)scan->ptr, x.st(), &in_a, &ln);
          perm = in_a ? (uint32_t*)vb->ptr : (uint32_t*)va->ptr;
        }
        x.count(ln);
        (void)perm_alt;
      }
    }
    int64_t m = fetch >= 0 ? std::min<int64_t>(fetch, n) : n;
    DevPtr idx = dev_alloc((size_t)std::max<int64_t>(m, 1) * 8, x.st());
    launch_u32_to_i64(perm, (int64_t*)idx->ptr, m, x.st());
    x.count();
    DevBatch proj;
    proj.n = n;
    for (size_t c = 0; c < n_in_cols; c++) proj.cols.push_back(in->cols[c]);
    DevBatchPtr out = gather_batch(x, proj, (const int64_t*)idx->ptr, m, false);
    x.wait();
    if (met) {
      met->elapsed_ns += (uint64_t)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t0).count();
      met->input_rows += (uint64_t)n;
    }
    return out;
  }

  // ---- hash join --------------------------------------------------------------------------------
  // Evaluates `outs` of a pipeline: columns the chain forwards untouched (and that no filter compacts) are taken
  // from the source batch as they are, only computed columns go through the materialising kernel.
  struct Mixed {
    std::vector<DevColumn> cols;  // one per entry of `outs`
    int64_t n = 0;
  };
  Mixed materialize_mixed(PipelineBuilder& pb, const std::vector<ColRef>& outs, const DevBatchPtr& src, OpMetrics* met) {
    Mixed m;
    const bool filters = program_filters(pb.prog);
    std::vector<int> direct(outs.size(), -1);
    std::vector<ColRef> mouts;
    for (size_t c = 0; c < outs.size(); c++) {
      if (!filters) direct[c] = pb.source_index(outs[c]);
      if (direct[c] < 0) mouts.push_back(outs[c]);
    }
    DevBatchPtr mat;
    m.n = src->n;
    if (!mouts.empty()) {
      mat = run_materialize(x, pb, mouts, src, met);
      m.n = mat->n;
    }
    size_t mi = 0;
    for (size_t c = 0; c < outs.size(); c++) {
      DevColumn col = direct[c] >= 0 ? src->cols[(size_t)direct[c]] : mat->cols[mi++];
      col.name = outs[c].name;
      m.cols.push_back(col);
    }
    return m;
  }

  struct JoinSide {
    DevBatch payload;              // output columns of the side
    std::vector<DevColumn> keys;   // evaluated join keys (strings as views)
    const uint64_t* hash = nullptr;
    DevColumn hash_col;
    int64_t n = 0;
  };
  JoinSide prepare_side(const PlanNode& child, int part, bool all, const std::vector<ExprPtr>& key_exprs, bool need_hash, OpMetrics* met) {
    JoinSide js;
    with_chain(child, part, all, [&](const BuilderFactory& mk, DevBatchPtr& src) {
      auto pbp = mk();
      PipelineBuilder& pb = *pbp;
      std::vector<ColRef> outs = named_cols(pb, child.schema);
      const size_t n_payload = outs.size();
      std::vector<ColRef> keys;
      for (auto& ke : key_exprs) {
        ColRef k = pb.compile(*ke);
        pb.pin(k);
        keys.push_back(k);
      }
      for (auto& k : keys) outs.push_back(k);
      if (need_hash) {
        ColRef h = pb.hash_of(keys);
        h.name = "__hash";
        outs.push_back(h);
      }
      Mixed m = materialize_mixed(pb, outs, src, met);
      js.n = m.n;
      js.payload.n = m.n;
      for (size_t c = 0; c < n_payload; c++) js.payload.cols.push_back(m.cols[c]);
      for (size_t k = 0; k < keys.size(); k++) js.keys.push_back(as_views(x, m.cols[n_payload + k]));
      if (need_hash) {
        js.hash_col = m.cols.back();
        js.hash = (const uint64_t*)js.hash_col.data;
      }
      return src;
    });
    return js;
  }

  static bool exact_key(const DataType& t) {
    switch (t.id) {
      case TypeId::Int8: case TypeId::Int16: case TypeId::Int32: case TypeId::Int64: case TypeId::UInt8: case TypeId::UInt16: case TypeId::UInt32:
      case TypeId::UInt64: case TypeId::Date32: case TypeId::Timestamp: return true;
      default: return false;
    }
  }

  DevBatchPtr exec_join(const PlanNode& n, int part, OpMetrics* met) {
    const bool collect_left = n.partition_mode == "CollectLeft";
    std::vector<ExprPtr> lk, rk;
    for (auto& on : n.on) {
      lk.push_back(on.first);
      rk.push_back(on.second);
    }
    const size_t nk = lk.size();
    if (nk > (size_t)VM_MAX_KEYS) throw EngineError(B200_ERR_UNSUPPORTED, "too many join keys");
    // CollectLeft replays the whole build side in every probe task; a join type that also EMITS build rows
    // (unmatched or semi/anti) would then emit them once per task.  DataFusion shares a visited bitmap across
    // the probe partitions of one process; tasks here are independent, so those shapes are only legal with a
    // single probe partition.
    if (collect_left && (n.join_type == JoinType::Left || n.join_type == JoinType::Full || n.join_type == JoinType::LeftSemi || n.join_type == JoinType::LeftAnti) &&
        n_partitions(*n.children[1]) > 1)
      throw EngineError(B200_ERR_UNSUPPORTED, "CollectLeft hash join that emits build-side rows over more than one probe partition: plan it as Partitioned");
    // one integer-like key: the table is keyed by the key itself (no hash column, no second look at the keys)
    const bool exact = nk == 1 && exact_key(lk[0]->type) && lk[0]->type.id == rk[0]->type.id;
    JoinSide L = prepare_side(*n.children[0], part, collect_left, lk, !exact, met);
    JoinSide R = prepare_side(*n.children[1], part, false, rk, !exact, met);
    const int64_t nb = L.n, np = R.n;
    if (nb >= ((int64_t)1 << 31)) throw EngineError(B200_ERR_UNSUPPORTED, "hash join build side exceeds 2^31 rows");
    auto t0 = std::chrono::steady_clock::now();
    JoinKeys K;
    memset(&K, 0, sizeof K);
    K.n_keys = (int)nk;
    K.null_equals_null = n.null_equals_null ? 1 : 0;
    uint64_t key_bytes_b = 0, key_bytes_p = 0;
    for (size_t k = 0; k < nk; k++) {
      const DevColumn& b = L.keys[k];
      const DevColumn& p = R.keys[k];
      if (b.phys != p.phys) throw EngineError(B200_ERR_UNSUPPORTED, "join key physical types differ (" + b.type.str() + " vs " + p.type.str() + "): add casts");
      K.build[k] = KeyCol{b.data, b.valid, (uint8_t)b.phys, (uint8_t)b.width()};
      K.probe[k] = KeyCol{p.data, p.valid, (uint8_t)p.phys, (uint8_t)p.width()};
      key_bytes_b += (uint64_t)b.width();
      key_bytes_p += (uint64_t)p.width();
    }
    const bool exact_ok = exact && !(n.null_equals_null && (L.keys[0].valid || R.keys[0].valid));
    if (exact && !exact_ok) throw EngineError(B200_ERR_UNSUPPORTED, "null_equals_null join on a nullable integer key");
    x.check_cancel();
    const uint64_t n_buckets = next_pow2((uint64_t)std::max<int64_t>(nb, 1) * 2);
    DevPtr heads = dev_alloc((size_t)n_buckets * 4, x.st());
    DevPtr nodes = dev_alloc((size_t)std::max<int64_t>(nb, 1) * sizeof(JoinNode), x.st());
    {
      KernelTimer kt(x, "join_build", (uint64_t)nb * (key_bytes_b + sizeof(JoinNode)) + n_buckets * 4);
      CUDA_CHECK(cudaMemsetAsync(heads->ptr, 0xFF, (size_t)n_buckets * 4, x.st()));
      launch_join_build2(K, exact, L.hash, nb, (int32_t*)heads->ptr, n_buckets, (JoinNode*)nodes->ptr, x.st());
      x.count();
    }
    x.check_cancel();
    const bool has_filter = n.join_filter != nullptr;
    const JoinType jt = n.join_type;
    const bool semi_anti = jt == JoinType::LeftSemi || jt == JoinType::LeftAnti || jt == JoinType::RightSemi || jt == JoinType::RightAnti;
    const bool left_outer = jt == JoinType::Left || jt == JoinType::Full, right_outer = jt == JoinType::Right || jt == JoinType::Full;
    const bool want_bmark = jt == JoinType::LeftSemi || jt == JoinType::LeftAnti || left_outer;
    const bool want_pmark = jt == JoinType::RightSemi || jt == JoinType::RightAnti || right_outer;
    // with a residual filter the marks must come from the pairs that survive it
    const bool need_pairs = has_filter || !semi_anti;
    int mode = need_pairs ? 1 : 0;
    DevPtr bmark, pmark;
    if (!has_filter && want_bmark) {
      bmark = dev_alloc((size_t)std::max<int64_t>(nb, 1), x.st());
      CUDA_CHECK(cudaMemsetAsync(bmark->ptr, 0, (size_t)std::max<int64_t>(nb, 1), x.st()));
      mode |= 4;
    }
    if (!has_filter && want_pmark) {
      pmark = dev_alloc((size_t)std::max<int64_t>(np, 1), x.st());
      CUDA_CHECK(cudaMemsetAsync(pmark->ptr, 0, (size_t)std::max<int64_t>(np, 1), x.st()));
      mode |= 2;
    }
    int64_t n_pairs = 0;
    DevPtr bi, pi;
    if (mode) {
      DevPtr counter = dev_alloc(16, x.st());
      uint64_t cap = need_pairs ? (uint64_t)std::max<int64_t>(np + nb / 8 + 1024, 1) : 0;
      for (int attempt = 0;; attempt++) {
        if (need_pairs) {
          bi = dev_alloc((size_t)std::max<uint64_t>(cap, 1) * 8, x.st());
          pi = dev_alloc((size_t)std::max<uint64_t>(cap, 1) * 8, x.st());
        }
        CUDA_CHECK(cudaMemsetAsync(counter->ptr, 0, 16, x.st()));
        {
          KernelTimer kt(x, "join_probe", (uint64_t)np * (key_bytes_p + 4 + sizeof(JoinNode)));
          launch_join_probe2(K, exact, mode, (const JoinNode*)nodes->ptr, (const int32_t*)heads->ptr, n_buckets, R.hash, np, (unsigned long long*)counter->ptr, cap,
                             need_pairs ? (int64_t*)bi->ptr : nullptr, need_pairs ? (int64_t*)pi->ptr : nullptr, pmark ? (uint8_t*)pmark->ptr : nullptr,
                             bmark ? (uint8_t*)bmark->ptr : nullptr, x.st());
          x.count();
        }
        if (!need_pairs) break;
        n_pairs = (int64_t)x.get<unsigned long long>(counter->ptr);
        if ((uint64_t)n_pairs <= cap) break;
        if (attempt) throw EngineError(B200_ERR_EXECUTION, "hash join: pair count changed between passes");
        cap = (uint64_t)n_pairs;  // many-to-many join: run again with the exact size
      }
    }
    x.check_cancel();
    const int64_t* bidx = need_pairs ? (const int64_t*)bi->ptr : nullptr;
    const int64_t* pidx = need_pairs ? (const int64_t*)pi->ptr : nullptr;
    const DevBatch& Lp = L.payload;
    const DevBatch& Rp = R.payload;
    DevPtr fbi, fpi;  // filtered pair lists
    if (has_filter && n_pairs > 0) {
      // evaluate the residual filter on the candidate pairs, carrying the pair indices through
      DevBatchPtr lg = gather_batch(x, Lp, bidx, n_pairs, false), rg = gather_batch(x, Rp, pidx, n_pairs, false);
      auto cat = std::make_shared<DevBatch>();
      cat->n = n_pairs;
      for (auto& c : lg->cols) cat->cols.push_back(c);
      for (auto& c : rg->cols) cat->cols.push_back(c);
      DevColumn ib, ip;
      ib.type = ip.type = DataType(TypeId::Int64);
      ib.phys = ip.phys = PH_I64;
      ib.n = ip.n = n_pairs;
      ib.data = (const uint8_t*)bi->ptr;
      ip.data = (const uint8_t*)pi->ptr;
      ib.keep.push_back(bi);
      ip.keep.push_back(pi);
      ib.name = "__bi";
      ip.name = "__pi";
      cat->cols.push_back(ib);
      cat->cols.push_back(ip);
      PipelineBuilder pb(*cat, x.st());
      pb.apply_filter(*n.join_filter);
      std::vector<ColRef> outs = {pb.cols[cat->cols.size() - 2], pb.cols[cat->cols.size() - 1]};
      DevBatchPtr kept = run_materialize(x, pb, outs, cat, met);
      n_pairs = kept->n;
      fbi = kept->cols[0].keep[0];
      fpi = kept->cols[1].keep[0];
      bidx = (const int64_t*)kept->cols[0].data;
      pidx = (const int64_t*)kept->cols[1].data;
    }
    auto flags_to_indices = [&](const uint8_t* marks, int64_t nrows, bool want, int64_t* n_sel) {
      DevPtr f = dev_alloc((size_t)(nrows + 1) * 4, x.st());
      DevPtr o = dev_alloc((size_t)(nrows + 2) * 8, x.st());
      DevPtr sc = dev_alloc((size_t)(nrows / 1024 + 4) * 8, x.st());
      launch_flag_to_u32(marks, want ? 1 : 0, (uint32_t*)f->ptr, nrows, x.st());
      launch_scan_u32_to_u64((const uint32_t*)f->ptr, (uint64_t*)o->ptr, nrows, (uint64_t*)sc->ptr, x.st());
      x.count(4);
      *n_sel = (int64_t)x.get<uint64_t>((const uint64_t*)o->ptr + nrows);
      DevPtr idx = dev_alloc((size_t)std::max<int64_t>(*n_sel, 1) * 8, x.st());
      launch_select_indices((const uint32_t*)f->ptr, (const uint64_t*)o->ptr, (int64_t*)idx->ptr, nrows, x.st());
      x.count();
      return idx;
    };
    auto marks_of = [&](const int64_t* idx, int64_t nrows, const DevPtr& from_probe) {
      if (!has_filter && from_probe) return from_probe;  // the probe pass already marked them
      DevPtr m = dev_alloc((size_t)std::max<int64_t>(nrows, 1), x.st());
      CUDA_CHECK(cudaMemsetAsync(m->ptr, 0, (size_t)std::max<int64_t>(nrows, 1), x.st()));
      if (n_pairs > 0) {
        launch_mark_from_idx(idx, n_pairs, (uint8_t*)m->ptr, x.st());
        x.count();
      }
      return m;
    };
    DevBatchPtr out;
    switch (jt) {
      case JoinType::LeftSemi:
      case JoinType::LeftAnti: {
        DevPtr m = marks_of(bidx, nb, bmark);
        int64_t ns = 0;
        DevPtr idx = flags_to_indices((const uint8_t*)m->ptr, nb, jt == JoinType::LeftSemi, &ns);
        out = gather_batch(x, Lp, (const int64_t*)idx->ptr, ns, false);
        break;
      }
      case JoinType::RightSemi:
      case JoinType::RightAnti: {
        DevPtr m = marks_of(pidx, np, pmark);
        int64_t ns = 0;
        DevPtr idx = flags_to_indices((const uint8_t*)m->ptr, np, jt == JoinType::RightSemi, &ns);
        out = gather_batch(x, Rp, (const int64_t*)idx->ptr, ns, false);
        break;
      }
      default: {
        // inner pairs (+ unmatched rows for outer joins, index -1 on the missing side)
        int64_t extra_l = 0, extra_r = 0;
        DevPtr ul, ur;
        if (left_outer) {
          DevPtr m = marks_of(bidx, nb, bmark);
          ul = flags_to_indices((const uint8_t*)m->ptr, nb, false, &extra_l);
        }
        if (right_outer) {
          DevPtr m = marks_of(pidx, np, pmark);
          ur = flags_to_indices((const uint8_t*)m->ptr, np, false, &extra_r);
        }
        const int64_t total = n_pairs + extra_l + extra_r;
        const int64_t* li_p = bidx;
        const int64_t* ri_p = pidx;
        DevPtr li, ri;
        if (extra_l || extra_r) {
          li = dev_alloc((size_t)std::max<int64_t>(total, 1) * 8, x.st());
          ri = dev_alloc((size_t)std::max<int64_t>(total, 1) * 8, x.st());
          if (n_pairs) {
            CUDA_CHECK(cudaMemcpyAsync(li->ptr, bidx, (size_t)n_pairs * 8, cudaMemcpyDeviceToDevice, x.st()));
            CUDA_CHECK(cudaMemcpyAsync(ri->ptr, pidx, (size_t)n_pairs * 8, cudaMemcpyDeviceToDevice, x.st()));
          }
          if (extra_l) {
            CUDA_CHECK(cudaMemcpyAsync((int64_t*)li->ptr + n_pairs, ul->ptr, (size_t)extra_l * 8, cudaMemcpyDeviceToDevice, x.st()));
            CUDA_CHECK(cudaMemsetAsync((int64_t*)ri->ptr + n_pairs, 0xFF, (size_t)extra_l * 8, x.st()));
          }
          if (extra_r) {
            CUDA_CHECK(cudaMemsetAsync((int64_t*)li->ptr + n_pairs + extra_l, 0xFF, (size_t)extra_r * 8, x.st()));
            CUDA_CHECK(cudaMemcpyAsync((int64_t*)ri->ptr + n_pairs + extra_l, ur->ptr, (size_t)extra_r * 8, cudaMemcpyDeviceToDevice, x.st()));
          }
          li_p = (const int64_t*)li->ptr;
          ri_p = (const int64_t*)ri->ptr;
        }
        // only the columns the join's projection keeps are gathered
        std::vector<int> want;
        const size_t nl = Lp.cols.size(), nr = Rp.cols.size();
        if (n.has_projection) want = n.projection;
        else
          for (size_t c = 0; c < nl + nr; c++) want.push_back((int)c);
        DevBatch Ls, Rs;
        Ls.n = nb;
        Rs.n = np;
        std::vector<std::pair<int, size_t>> where;  // per wanted column: (side, index inside the side's gathered batch)
        for (int idx : want) {
          if ((size_t)idx < nl) {
            where.push_back({0, Ls.cols.size()});
            Ls.cols.push_back(Lp.cols[(size_t)idx]);
          } else {
            where.push_back({1, Rs.cols.size()});
            Rs.cols.push_back(Rp.cols.at((size_t)idx - nl));
          }
        }
        KernelTimer kt(x, "join_gather", 0);
        DevBatchPtr lg = gather_batch(x, Ls, li_p, total, right_outer);
        DevBatchPtr rg = gather_batch(x, Rs, ri_p, total, left_outer);
        out = std::make_shared<DevBatch>();
        out->n = total;
        for (auto& w : where) out->cols.push_back(w.first == 0 ? lg->cols[w.second] : rg->cols[w.second]);
        for (size_t c = 0; c < out->cols.size() && c < n.schema.size(); c++) out->cols[c].name = n.schema[c].name;
        if (met) {
          met->elapsed_ns += (uint64_t)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t0).count();
          met->input_rows += (uint64_t)(nb + np);
        }
        return out;
      }
    }
    if (n.has_projection) {
      auto p = std::make_shared<DevBatch>();
      p->n = out->n;
      for (int idx : n.projection) p->cols.push_back(out->cols.at((size_t)idx));
      out = p;
    }
    for (size_t c = 0; c < out->cols.size() && c < n.schema.size(); c++) out->cols[c].name = n.schema[c].name;
    if (met) {
      met->elapsed_ns += (uint64_t)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t0).count();
      met->input_rows += (uint64_t)(nb + np);
    }
    return out;
  }

  // ---- shuffle writer -----------------------------------------------------------------------------
  uint64_t slice_bytes(const DevBatch& b, int64_t rows, const std::vector<int64_t>& chars_bytes) {
    uint64_t t = 0;
    size_t si = 0;
    for (auto& c : b.cols) {
      if (c.type.id == TypeId::Bool) t += (uint64_t)(rows + 7) / 8;
      else if (c.type.id == TypeId::Utf8) t += 4ull * (uint64_t)(rows + 1) + (uint64_t)chars_bytes[si++];
      else t += (uint64_t)c.width() * (uint64_t)rows;
    }
    return t;
  }

  // character bytes of every Utf8 column of `b` (rows [0, b.n)), one read-back for all of them; known values are reused
  std::vector<int64_t> string_bytes(const DevBatch& b) {
    std::vector<int64_t> out;
    queue_string_bytes(b, out);
    x.sync();
    return out;
  }
  // the same, with the read-back queued: `out` is complete after the task's next x.sync()
  void queue_string_bytes(const DevBatch& b, std::vector<int64_t>& out) {
    PartStrCols sc;
    sc.n = 0;
    std::vector<size_t> unknown;
    for (auto& c : b.cols) {
      if (c.type.id != TypeId::Utf8) continue;
      if (c.phys == PH_UTF8 && c.chars_bytes >= 0) {
        out.push_back(c.chars_bytes);
        continue;
      }
      out.push_back(-1);
      if (b.n == 0) {
        out.back() = 0;
        continue;
      }
      if (sc.n == PART_MAX_STR_COLS) throw EngineError(B200_ERR_UNSUPPORTED, "more than 16 string columns in one shuffle output");
      sc.c[sc.n++] = PartStrCol{c.data, c.valid, c.phys == PH_STRVIEW ? 1 : 0, 0};
      unknown.push_back(out.size() - 1);
    }
    if (sc.n) {
      DevPtr acc = dev_alloc((size_t)(1 + sc.n) * 8, x.st());
      CUDA_CHECK(cudaMemsetAsync(acc->ptr, 0, (size_t)(1 + sc.n) * 8, x.st()));
      PidSrc none;
      memset(&none, 0, sizeof none);
      CUDA_CHECK(launch_partition_hist(none, b.n, 1, nullptr, (unsigned long long*)acc->ptr, sc, (unsigned long long*)acc->ptr + 1, x.st()));
      x.count();
      const unsigned long long* h = (const unsigned long long*)x.fetch_bytes((const unsigned long long*)acc->ptr + 1, (size_t)sc.n * 8);
      x.defer([h, unknown, &out]() {
        for (size_t k = 0; k < unknown.size(); k++) out[unknown[k]] = (int64_t)h[k];
      });
    }
  }

  struct FusedExchange {
    bool done = false;  // the rows were scattered into their owners' windows (nothing left to exchange)
    uint64_t sent = 0, recvd = 0;
  };

  // ------------------------------------------------------------------------------------------------
  // Fused shuffle writer + exchange (gang collective; ShuffleWriterExec's repartition, shuffle_writer.rs:214-330, and
  // the readers' remote fetch, shuffle_reader.rs:522-602, as ONE kernel pass).  After the histogram every executor
  // knows how many rows every map task holds for every output partition (one small NCCL all-gather), so every row has a
  // known final address in the window of the executor that owns its partition: the scatter kernel stores it there
  // directly -- local partitions through HBM, remote ones as peer stores over NVLink.  The reduce side finds its input
  // already laid out partition by partition, map task by map task (the order sort_shuffle and the NCCL exchange produce).
  // Returns false (nothing written) when some window cannot hold this exchange: the caller then takes the two-step path;
  // the decision is taken from the all-gathered matrix, i.e. identically on every executor.
  // ------------------------------------------------------------------------------------------------
  bool scatter_to_owners(const PlanNode& root, int input_partition, const std::vector<DevColumn>& pay, const PidSrc& pid, int64_t n, uint32_t P,
                         uint32_t n_tiles, const DevPtr& mat, const DevPtr& tile_hist, uint64_t row_bytes, FusedExchange* fx,
                         std::vector<b200_shuffle_write_partition>& res, OpMetrics* met) {
    b200_engine* e = x.e;
    NcclApi& N = NcclApi::get();
    const int W = e->world, me = e->rank;
    const size_t mrow = (size_t)P + 3;
    const size_t ncols = pay.size();
    auto al = [](uint64_t v) { return (v + 255) & ~255ull; };
    std::lock_guard<std::mutex> cg(e->comm_mu);
    // my row of the matrix: the counts are already there (histogram); add validity mask, window fill, map task id
    uint64_t* extra = (uint64_t*)x.stage_bytes(24);
    extra[0] = 0;
    for (size_t c = 0; c < ncols; c++)
      if (pay[c].valid) extra[0] |= 1ull << c;
    extra[1] = al(e->win_used);
    extra[2] = (uint64_t)(int64_t)input_partition;
    unsigned long long* mrows = (unsigned long long*)mat->ptr;
    CUDA_CHECK(cudaMemcpyAsync(mrows + mrow * (size_t)me + P, extra, 24, cudaMemcpyHostToDevice, x.st()));
    NCCL_CHECK(N.GroupStart());
    for (int d = 0; d < W; d++) {
      if (d == me) continue;
      NCCL_CHECK(N.Send(mrows + mrow * (size_t)me, mrow * 8, kNcclUint8, d, e->comm, x.st()));
      NCCL_CHECK(N.Recv(mrows + mrow * (size_t)d, mrow * 8, kNcclUint8, d, e->comm, x.st()));
    }
    NCCL_CHECK(N.GroupEnd());
    x.count(1);
    // (the matrix and the base table below can exceed the task's pinned arena at large fan-outs: plain host vectors)
    std::vector<unsigned long long> Mv(mrow * (size_t)W);
    CUDA_CHECK(cudaMemcpyAsync(Mv.data(), mat->ptr, Mv.size() * 8, cudaMemcpyDeviceToHost, x.st()));
    const unsigned long long* M = Mv.data();
    // while the matrix travels: per-tile offsets of the local rows
    const int64_t hn = (int64_t)P * n_tiles;
    DevPtr offs = dev_alloc((size_t)(hn + 2) * 8, x.st());
    DevPtr scratch = dev_alloc((size_t)(hn / 1024 + 4) * 8, x.st());
    if (hn > 0) {
      launch_scan_u32_to_u64((const uint32_t*)tile_hist->ptr, (uint64_t*)offs->ptr, hn, (uint64_t*)scratch->ptr, x.st());
      x.count(3);
    }
    x.sync();
    auto cnt = [&](int s, uint32_t p) { return (uint64_t)M[mrow * (size_t)s + p]; };
    uint64_t any_valid = 0;
    for (int s = 0; s < W; s++) any_valid |= M[mrow * (size_t)s + P];
    // layout of every owner's window for this exchange: per owned partition, per column, all map tasks back to back
    std::vector<uint64_t> tot(P, 0), before(P, 0);
    for (uint32_t p = 0; p < P; p++)
      for (int s = 0; s < W; s++) {
        if (s < me) before[p] += cnt(s, p);
        tot[p] += cnt(s, p);
      }
    const size_t nslots = ncols * 2;  // [c] data, [ncols + c] validity
    std::vector<uint64_t> region(nslots * P, 0);
    std::vector<uint64_t> cursor((size_t)W);
    for (int r = 0; r < W; r++) cursor[(size_t)r] = M[mrow * (size_t)r + P + 1];
    for (uint32_t p = 0; p < P; p++) {
      uint64_t& cur = cursor[(size_t)(p % (uint32_t)W)];
      for (size_t c = 0; c < ncols; c++) {
        region[c * P + p] = cur;
        cur += al(tot[p] * (uint64_t)pay[c].width());
        if (any_valid >> c & 1) {
          region[(ncols + c) * P + p] = cur;
          cur += al(tot[p]);
        }
      }
    }
    for (int r = 0; r < W; r++)
      if (cursor[(size_t)r] > e->win_bytes) return false;  // same verdict everywhere; nothing was written
    // destination bases: byte address of row 0 of (column, partition) as the scatter kernel numbers the rows, i.e.
    // shifted back by this task's prefix of the partition-contiguous order
    std::vector<int64_t> bounds(P + 1, 0);
    for (uint32_t p = 0; p < P; p++) bounds[p + 1] = bounds[p] + (int64_t)cnt(me, p);
    std::vector<uint64_t> hbv(nslots * P);
    uint64_t* hb = hbv.data();
    for (size_t sl = 0; sl < nslots; sl++) {
      const size_t c = sl % ncols;
      const int64_t w = sl < ncols ? (int64_t)pay[c].width() : 1;
      for (uint32_t p = 0; p < P; p++) {
        const uint8_t* base = e->win_peer[(size_t)(p % (uint32_t)W)] + region[sl * P + p];
        hb[sl * P + p] = (uint64_t)(base + ((int64_t)before[p] - bounds[p]) * w);
      }
    }
    DevPtr bases = dev_alloc(nslots * P * 8 + 64, x.st());
    CUDA_CHECK(cudaMemcpyAsync(bases->ptr, hb, nslots * P * 8, cudaMemcpyHostToDevice, x.st()));
    std::vector<DevPtr> ones_keep;
    {
      GatherCols gc;
      gc.n = 0;
      auto flush = [&]() {
        if (gc.n && n > 0) {
          uint64_t b = 0;
          for (int k = 0; k < gc.n; k++) b += (uint64_t)gc.c[k].width;
          KernelTimer kt(x, "partition_scatter_peer", (uint64_t)n * (2 * b + 4));
          CUDA_CHECK(launch_partition_scatter(pid, n, P, (const uint64_t*)offs->ptr, gc, nullptr, x.st()));
          x.count();
        }
        gc.n = 0;
      };
      auto add = [&](const void* in, size_t slot, int width) {
        GatherCol& g = gc.c[gc.n++];
        memset(&g, 0, sizeof g);
        g.in = in;
        g.width = width;
        g.part_base = (const unsigned long long*)bases->ptr + slot * P;
        if (gc.n == GATHER_MAX_COLS) flush();
      };
      for (size_t c = 0; c < ncols; c++) {
        add(pay[c].data, c, pay[c].width());
        if (any_valid >> c & 1) {
          const uint8_t* v = pay[c].valid;
          if (!v && n > 0) {  // another map task has nulls in this column: this one contributes all-valid bytes
            DevPtr ones = dev_alloc((size_t)n + 64, x.st());
            CUDA_CHECK(cudaMemsetAsync(ones->ptr, 1, (size_t)n, x.st()));
            ones_keep.push_back(ones);
            v = (const uint8_t*)ones->ptr;
          }
          add(v, ncols + c, 1);
        }
      }
      flush();
    }
    // every executor's stores must have landed before anyone reads its window: a zero-payload all-to-all on the same
    // stream completes only after every peer's scatter kernel did
    {
      DevPtr bar = dev_alloc((size_t)W * 16 + 64, x.st());
      NCCL_CHECK(N.GroupStart());
      for (int d = 0; d < W; d++) {
        if (d == me) continue;
        NCCL_CHECK(N.Send((const uint8_t*)bar->ptr + 8 * (size_t)W, 8, kNcclUint8, d, e->comm, x.st()));
        NCCL_CHECK(N.Recv((uint8_t*)bar->ptr + 8 * (size_t)d, 8, kNcclUint8, d, e->comm, x.st()));
      }
      NCCL_CHECK(N.GroupEnd());
      x.count(1);
    }
    e->win_used = cursor[(size_t)me];
    // the reduce side's view: one batch per owned partition, one piece per map task
    const int64_t bs = e->batch_size;
    uint64_t total_bytes = 0;
    {
      std::lock_guard<std::mutex> g(e->mu);
      for (uint32_t p = 0; p < P; p++) {
        const uint64_t rows = cnt(me, p);
        if (rows) {
          b200_shuffle_write_partition w{};
          w.partition_id = p;
          w.num_rows = rows;
          w.num_batches = (rows + (uint64_t)bs - 1) / (uint64_t)bs;
          w.num_bytes = rows * row_bytes;
          w.file_id = input_partition;
          w.is_sort_shuffle = root.sort_shuffle ? 1 : 0;
          total_bytes += w.num_bytes;
          res.push_back(w);
          if ((int)(p % (uint32_t)W) != me) fx->sent += w.num_bytes;
        }
        if ((int)(p % (uint32_t)W) != me) continue;
        auto& v = e->shuffle[ShuffleKey{job, root.stage_id, (int64_t)p}];
        if (tot[p] == 0) {
          if (v.empty()) e->shuffle.erase(ShuffleKey{job, root.stage_id, (int64_t)p});
          continue;
        }
        auto b = std::make_shared<DevBatch>();
        b->n = (int64_t)tot[p];
        for (size_t c = 0; c < ncols; c++) {
          DevColumn col;
          col.name = root.schema[c].name;
          col.type = pay[c].type;
          col.phys = pay[c].phys;
          col.n = b->n;
          col.data = e->win_local + region[c * P + p];
          col.nullable = (any_valid >> c & 1) != 0;
          if (col.nullable) col.valid = e->win_local + region[(ncols + c) * P + p];
          b->cols.push_back(col);
        }
        int64_t at = 0;
        for (int s = 0; s < W; s++) {
          const int64_t rs = (int64_t)cnt(s, p);
          const int64_t fid = (int64_t)M[mrow * (size_t)s + P + 2];
          if (rs) {
            v.erase(std::remove_if(v.begin(), v.end(), [&](const Piece& pc) { return pc.file_id == fid && pc.src_rank == s; }), v.end());
            v.push_back(Piece{fid, b, at, at + rs, s, {}});
            if (s != me) fx->recvd += (uint64_t)rs * row_bytes;
          }
          at += rs;
        }
        std::stable_sort(v.begin(), v.end(), [](const Piece& a, const Piece& b2) { return a.src_rank != b2.src_rank ? a.src_rank < b2.src_rank : a.file_id < b2.file_id; });
      }
    }
    x.sync();
    if (met) {
      met->output_rows += (uint64_t)n;
      met->bytes_written += total_bytes;
      met->bytes_read += total_bytes;
    }
    e->fused_exchanges++;
    fx->done = true;
    return true;
  }

  std::vector<b200_shuffle_write_partition> execute_stage(const PlanNode& root, int input_partition, FusedExchange* fx = nullptr) {
    if (root.op != PlanNode::ShuffleWriter) throw EngineError(B200_ERR_INVALID, "stage plan root must be a ShuffleWriterExec");
    OpMetrics* met = x.m(&root);
    const PlanNode& child = *root.children[0];
    const int64_t bs = x.e->batch_size;
    const int32_t my_rank = x.e->rank;
    auto nbatches = [&](uint64_t rows) { return (rows + (uint64_t)bs - 1) / (uint64_t)bs; };
    std::vector<b200_shuffle_write_partition> res;
    // no repartitioning; also hash partitioning into ONE partition (hash % 1 == 0 for every row), which
    // keeps the rows of this task together as output partition 0
    const bool single = root.n_out_partitions == 1;
    if (root.n_out_partitions == 0 || single) {
      DevBatchPtr in = exec(child, input_partition);
      // stored as produced: strings stay views into kept-alive character buffers; they are laid out as Arrow
      // Utf8 only when the partition leaves the device (export) or the GPU (exchange)
      auto st = std::make_shared<DevBatch>();
      st->n = in->n;
      for (size_t c = 0; c < in->cols.size(); c++) {
        DevColumn col = in->cols[c];
        col.name = root.schema[c].name;
        st->cols.push_back(col);
      }
      std::vector<int64_t> cb;
      {
        ScopeTimer t2("writer: string bytes + final sync");
        queue_string_bytes(*st, cb);
        x.sync();  // the string byte counts and the deferred status checks of this task's kernels
      }
      b200_shuffle_write_partition w{};
      w.partition_id = single ? 0u : (uint64_t)input_partition;
      w.num_rows = (uint64_t)st->n;
      w.num_batches = nbatches(w.num_rows);
      w.num_bytes = slice_bytes(*st, st->n, cb);
      w.file_id = single ? (int64_t)input_partition : -1;
      w.is_sort_shuffle = (single && root.sort_shuffle) ? 1 : 0;
      {
        std::lock_guard<std::mutex> g(x.e->mu);
        auto& v = x.e->shuffle[ShuffleKey{job, root.stage_id, single ? 0 : input_partition}];
        if (single) {
          const int64_t fid = (int64_t)input_partition;
          v.erase(std::remove_if(v.begin(), v.end(), [&](const Piece& pc) { return pc.file_id == fid && pc.src_rank == my_rank; }), v.end());
          if (st->n > 0) v.push_back(Piece{fid, st, 0, st->n, my_rank, cb});
          else if (v.empty()) x.e->shuffle.erase(ShuffleKey{job, root.stage_id, 0});
        } else {
          v.clear();
          v.push_back(Piece{-1, st, 0, st->n, my_rank, cb});
        }
      }
      if (met) {
        met->output_rows += w.num_rows;
        met->input_rows += w.num_rows;
        met->bytes_written += w.num_bytes;
      }
      if (!(single && st->n == 0)) res.push_back(w);  // only partitions with rows are reported
      return res;
    }
    // hash repartition: pid = hash(keys) % P computed by the child's pipeline kernel, then ONE stable radix
    // partition pass (per-tile histogram -> scan -> ranked scatter of every column)
    const uint32_t P = (uint32_t)root.n_out_partitions;
    if (P > PART_MAX_FANOUT) throw EngineError(B200_ERR_UNSUPPORTED, "more than 4096 output partitions in one shuffle");
    size_t n_payload = 0;
    std::vector<DevColumn> pay;   // payload columns (strings as views)
    PidSrc ps;
    memset(&ps, 0, sizeof ps);
    std::vector<DevColumn> key_keep;
    DevBatchPtr mat_keep;
    int64_t n = 0;
    with_chain(child, input_partition, false, [&](const BuilderFactory& mk, DevBatchPtr& src) {
      auto pbp = mk();
      PipelineBuilder& pb = *pbp;
      std::vector<ColRef> outs = named_cols(pb, root.schema);
      n_payload = outs.size();
      std::vector<ColRef> keys;
      for (auto& e : root.part_exprs) {
        ColRef k = pb.compile(*e);
        pb.pin(k);
        keys.push_back(k);
      }
      // shuffle keys that are plain integer-like columns of an unfiltered input: the partition kernels hash them on
      // the fly; otherwise the pipeline kernel materialises the partition id next to the computed payload columns
      // integer-like shuffle keys travel as columns (forwarded untouched, or compacted with the payload when the chain
      // filters) and the partition kernels hash them on the fly; other key types get a materialised partition id
      bool direct_keys = !keys.empty() && keys.size() <= (size_t)VM_MAX_KEYS;
      for (auto& k : keys) direct_keys = direct_keys && exact_key(k.type) && (k.op.kind == OPD_NONE || k.op.kind == OPD_COL);
      if (direct_keys) {
        for (auto& k : keys) outs.push_back(k);
      } else {
        ColRef h = pb.hash_of(keys);
        ColRef pid = pb.mod_u64(h, P);
        pid.name = "__pid";
        outs.push_back(pid);
      }
      Mixed m = materialize_mixed(pb, outs, src, met);
      n = m.n;
      for (size_t c = 0; c < n_payload; c++) {
        DevColumn col = as_views(x, m.cols[c]);
        col.name = root.schema[c].name;
        pay.push_back(col);
      }
      if (direct_keys) {
        for (size_t k = 0; k < keys.size(); k++) {
          const DevColumn& kc = m.cols[n_payload + k];
          ps.keys[ps.n_keys++] = KeyCol{kc.data, kc.valid, (uint8_t)kc.phys, (uint8_t)kc.width()};
          key_keep.push_back(kc);
        }
      } else {
        key_keep.push_back(m.cols.back());
        ps.pid = (const uint32_t*)m.cols.back().data;
      }
      return src;
    });
    if (n >= ((int64_t)1 << 32)) throw EngineError(B200_ERR_UNSUPPORTED, "more than 2^32 rows in one shuffle-writer task");
    const PidSrc& pid = ps;
    // histogram (+ string bytes per partition for ShuffleWritePartition.num_bytes)
    PartStrCols sc;
    sc.n = 0;
    for (auto& c : pay)
      if (c.type.id == TypeId::Utf8) {
        if (sc.n == PART_MAX_STR_COLS) throw EngineError(B200_ERR_UNSUPPORTED, "more than 16 string columns in one shuffle output");
        sc.c[sc.n++] = PartStrCol{c.data, c.valid, c.phys == PH_STRVIEW ? 1 : 0, 0};
      }
    if ((size_t)P * (1 + sc.n) * 4 > 200 * 1024) throw EngineError(B200_ERR_UNSUPPORTED, "shuffle fan-out x string columns exceeds the histogram's shared memory");
    const uint32_t n_tiles = partition_n_tiles(n);
    const size_t acc_words = (size_t)P * (1 + sc.n);
    // fused shuffle: decided from the schema and the engine's configuration only, so that every executor of the gang
    // takes the same branch
    const int W = x.e->world, me = x.e->rank;
    const bool fuse = fx && W > 1 && x.e->comm && x.e->win_local && sc.n == 0 && n_payload <= 60;
    const size_t mrow = (size_t)P + 3;  // per executor: P row counts, validity mask, window fill, map task id
    DevPtr acc = dev_alloc((fuse ? mrow * (size_t)W : acc_words) * 8, x.st());
    CUDA_CHECK(cudaMemsetAsync(acc->ptr, 0, (fuse ? mrow * (size_t)W : acc_words) * 8, x.st()));
    unsigned long long* const acc_ptr = (unsigned long long*)acc->ptr + (fuse ? mrow * (size_t)me : 0);
    DevPtr tile_hist = dev_alloc((size_t)std::max<uint64_t>((uint64_t)P * n_tiles, 1) * 4 + 64, x.st());
    uint64_t row_bytes = 0;
    for (auto& c : pay) row_bytes += (uint64_t)c.width() + (c.valid ? 1 : 0);
    {
      uint64_t kb = pid.pid ? 4 : 0;
      for (int k = 0; k < pid.n_keys; k++) kb += pid.keys[k].width;
      KernelTimer kt(x, "partition_hist", (uint64_t)n * kb);
      CUDA_CHECK(launch_partition_hist(pid, n, P, (uint32_t*)tile_hist->ptr, acc_ptr, sc, acc_ptr + P, x.st()));
      x.count();
    }
    if (fuse) {
      std::vector<b200_shuffle_write_partition> fr;
      if (scatter_to_owners(root, input_partition, pay, pid, n, P, n_tiles, acc, tile_hist, row_bytes, fx, fr, met)) return fr;
    }
    const unsigned long long* hc = (const unsigned long long*)x.fetch_bytes(acc_ptr, acc_words * 8);
    // while the counts travel: scan the per-tile histogram and scatter
    const int64_t hn = (int64_t)P * n_tiles;
    DevPtr offs = dev_alloc((size_t)(hn + 2) * 8, x.st());
    DevPtr scratch = dev_alloc((size_t)(hn / 1024 + 4) * 8, x.st());
    if (hn > 0) {
      launch_scan_u32_to_u64((const uint32_t*)tile_hist->ptr, (uint64_t*)offs->ptr, hn, (uint64_t*)scratch->ptr, x.st());
      x.count(3);
    }
    auto st = std::make_shared<DevBatch>();
    st->n = n;
    {
      GatherCols gc;
      gc.n = 0;
      auto flush = [&]() {
        if (gc.n && n > 0) {
          uint64_t b = 0;
          for (int k = 0; k < gc.n; k++) b += (uint64_t)gc.c[k].width;
          KernelTimer kt(x, "partition_scatter", (uint64_t)n * (2 * b + 4));
          CUDA_CHECK(launch_partition_scatter(pid, n, P, (const uint64_t*)offs->ptr, gc, nullptr, x.st()));
          x.count();
        }
        gc.n = 0;
      };
      auto add = [&](const void* in, void* out, int width) {
        GatherCol& g = gc.c[gc.n++];
        memset(&g, 0, sizeof g);
        g.in = in;
        g.out = out;
        g.width = width;
        if (gc.n == GATHER_MAX_COLS) flush();
      };
      for (size_t c = 0; c < n_payload; c++) {
        const DevColumn& scn = pay[c];
        DevColumn oc = make_out_column(root.schema[c].name, scn.type, scn.phys, n, scn.valid != nullptr, x.st());
        oc.n = n;
        add(scn.data, (void*)oc.data, scn.width());
        if (scn.valid) add(scn.valid, (void*)oc.valid, 1);
        for (auto& k : scn.keep) oc.keep.push_back(k);
        st->cols.push_back(oc);
      }
      flush();
    }
    x.sync();
    std::vector<int64_t> bounds(P + 1, 0);
    for (uint32_t p = 0; p < P; p++) bounds[p + 1] = bounds[p] + (int64_t)hc[p];
    std::vector<std::vector<int64_t>> chars_per_part((size_t)sc.n, std::vector<int64_t>(P));  // [string col][p]
    for (int c = 0; c < sc.n; c++)
      for (uint32_t p = 0; p < P; p++) chars_per_part[(size_t)c][p] = (int64_t)hc[(size_t)P * (1 + c) + p];
    uint64_t total_bytes = 0;
    {
      std::lock_guard<std::mutex> g(x.e->mu);
      for (uint32_t p = 0; p < P; p++) {
        auto& v = x.e->shuffle[ShuffleKey{job, root.stage_id, (int64_t)p}];
        // a re-run of the same map task replaces its previous output (task retry)
        v.erase(std::remove_if(v.begin(), v.end(), [&](const Piece& pc) { return pc.file_id == input_partition && pc.src_rank == my_rank; }), v.end());
        const int64_t rows = bounds[p + 1] - bounds[p];
        if (rows == 0) {
          if (v.empty()) x.e->shuffle.erase(ShuffleKey{job, root.stage_id, (int64_t)p});
          continue;  // only partitions with rows are reported (sort_shuffle/writer.rs:357-369)
        }
        std::vector<int64_t> cb;
        for (auto& cp : chars_per_part) cb.push_back(cp[p]);
        v.push_back(Piece{input_partition, st, bounds[p], bounds[p + 1], my_rank, cb});
        b200_shuffle_write_partition w{};
        w.partition_id = p;
        w.num_rows = (uint64_t)rows;
        w.num_batches = nbatches(w.num_rows);
        w.num_bytes = slice_bytes(*st, rows, cb);
        w.file_id = input_partition;
        w.is_sort_shuffle = root.sort_shuffle ? 1 : 0;
        total_bytes += w.num_bytes;
        res.push_back(w);
      }
    }
    if (met) {
      met->output_rows += (uint64_t)n;
      met->bytes_written += total_bytes;
      met->bytes_read += total_bytes;
    }
    return res;
  }
};

// ------------------------------------------------------------------------------------------------
// Exchange between the box's GPU executors (ShuffleReaderExec's remote fetch, shuffle_reader.rs:522-602 /
// client.rs:143-220, as an all-to-all-v over NVLink).  Gang collective: every executor of the communicator calls
// it for the same (job, stage) after its map tasks finished.
//
// Round 1: every pair exchanges one fixed-size slot = [header | inline payload].  The header lists, per piece,
// (partition, file id, rows, byte size of every column buffer) -- the ShuffleWritePartition / PartitionLocation
// metadata the reference sends through the scheduler -- so no separate size collective is needed, and messages
// of up to EXCH_INLINE bytes (the partial-aggregate states of q1: a few hundred bytes) are complete after it.
// Round 2 (only for pairs whose payload is larger): grouped ncclSend/ncclRecv straight from the stored column
// slices into the receiver's final column buffers -- no packing copy on either side.
// ------------------------------------------------------------------------------------------------
static const uint64_t EXCH_MAGIC = 0xB200E8C4A11ull;
static const size_t EXCH_INLINE = 16 << 10;
enum ExchangeMode { EXCH_HASH = 0, EXCH_GATHER = 1, EXCH_BROADCAST = 2 };

struct ExchEntry {
  int64_t partition, file_id, rows;
  std::vector<uint64_t> sizes;  // 3 per column: validity bytes, data bytes, chars bytes
};

struct Exchange {
  Exec x;
  Runner r;
  b200_engine* e;
  std::string job;
  int64_t stage;
  int P, mode, root;
  Schema schema;
  size_t ncols;

  bool goes_to(int p, int d) const {
    if (mode == EXCH_BROADCAST) return true;
    if (mode == EXCH_GATHER) return d == root;
    return p % e->world == d;
  }
  int n_owned(int d) const {
    int k = 0;
    for (int p = 0; p < P; p++) k += goes_to(p, d) ? 1 : 0;
    return k;
  }
  size_t entry_bytes() const { return (3 + 3 * ncols) * 8; }
  size_t hdr_bytes(int d) const { return (32 + (size_t)n_owned(d) * entry_bytes() + 255) & ~(size_t)255; }
  size_t slot_bytes() const {
    size_t h = 0;
    for (int d = 0; d < e->world; d++) h = std::max(h, hdr_bytes(d));
    return h + EXCH_INLINE;
  }
  static uint64_t al16(uint64_t v) { return (v + 15) & ~15ull; }

  void run(uint64_t* sent_out, uint64_t* recv_out) {
    NcclApi& N = NcclApi::get();
    const int W = e->world, me = e->rank;
    // ---- local pieces: one (coalesced) piece per partition ------------------------------------------------
    struct Local {
      int p;
      Piece piece;
    };
    std::vector<Local> locals;
    {
      std::vector<std::pair<int, std::vector<Piece>>> snap;
      {
        std::lock_guard<std::mutex> g(e->mu);
        for (int p = 0; p < P; p++) {
          auto it = e->shuffle.find(ShuffleKey{job, stage, (int64_t)p});
          if (it == e->shuffle.end()) continue;
          std::vector<Piece> mine;
          for (auto& pc : it->second)
            if (pc.src_rank == me && pc.r1 > pc.r0) mine.push_back(pc);
          if (!mine.empty()) snap.push_back({p, mine});
        }
      }
      for (auto& kv : snap) {
        if (kv.second.size() == 1) {
          locals.push_back(Local{kv.first, kv.second[0]});
          continue;
        }
        std::vector<std::pair<DevBatchPtr, std::pair<int64_t, int64_t>>> v;
        for (auto& pc : kv.second) v.push_back({pc.batch, {pc.r0, pc.r1}});
        Piece c;
        c.file_id = kv.second[0].file_id;
        c.batch = r.concat_slices(v, schema);
        c.r0 = 0;
        c.r1 = c.batch->n;
        c.src_rank = me;
        bool known = true;
        for (auto& pc : kv.second) known &= !pc.str_bytes.empty() || pc.batch->cols.empty();
        if (known && !kv.second[0].str_bytes.empty()) {
          c.str_bytes.assign(kv.second[0].str_bytes.size(), 0);
          for (auto& pc : kv.second)
            for (size_t k = 0; k < c.str_bytes.size(); k++) c.str_bytes[k] += pc.str_bytes[k];
        }
        locals.push_back(Local{kv.first, c});
      }
    }
    // string bytes of every outgoing slice must be known on the host (they normally are: the writer recorded them)
    for (auto& L : locals) {
      size_t n_str = 0;
      for (auto& c : L.piece.batch->cols) n_str += c.type.id == TypeId::Utf8 ? 1 : 0;
      if (L.piece.batch->cols.size() != ncols) throw EngineError(B200_ERR_INVALID, "exchange: stored partition does not match the given schema");
      if (n_str && L.piece.str_bytes.size() != n_str) {
        DevBatch sl;
        sl.n = L.piece.r1 - L.piece.r0;
        for (auto& c : L.piece.batch->cols) sl.cols.push_back(slice_column(c, L.piece.r0, L.piece.r1));
        L.piece.str_bytes = r.string_bytes(sl);
      }
    }
    if (W <= 1) {
      *sent_out = *recv_out = 0;
      return;
    }
    if (!e->comm) throw EngineError(B200_ERR_INVALID, "exchange: communicator not initialised (b200_engine_comm_init)");
    const size_t slot = slot_bytes();
    DevPtr sendbuf = dev_alloc(slot * W, x.st()), recvbuf = dev_alloc(slot * W, x.st());
    // ---- compose headers and the payload layout per destination -----------------------------------------------
    struct Out {
      std::vector<ExchEntry> entries;
      std::vector<const Local*> src;
      uint64_t payload = 0;
      bool inl = true;
    };
    std::vector<Out> outs((size_t)W);
    for (int d = 0; d < W; d++) {
      if (d == me) continue;
      Out& o = outs[(size_t)d];
      for (auto& L : locals) {
        if (!goes_to(L.p, d)) continue;
        ExchEntry en;
        en.partition = L.p;
        en.file_id = L.piece.file_id;
        en.rows = L.piece.r1 - L.piece.r0;
        size_t si = 0;
        for (auto& c : L.piece.batch->cols) {
          en.sizes.push_back(c.valid ? (uint64_t)en.rows : 0);
          if (c.type.id == TypeId::Utf8) {
            en.sizes.push_back((uint64_t)(en.rows + 1) * 4);
            en.sizes.push_back((uint64_t)L.piece.str_bytes[si++]);
          } else {
            en.sizes.push_back((uint64_t)en.rows * c.width());
            en.sizes.push_back(0);
          }
        }
        for (uint64_t b : en.sizes) o.payload += al16(b);
        o.entries.push_back(en);
        o.src.push_back(&L);
      }
      o.inl = o.payload <= EXCH_INLINE;
    }
    // headers -> one staging block -> device; inline payloads packed by the same kernel that places the headers
    size_t hdr_total = 0;
    std::vector<size_t> hdr_at((size_t)W, 0);
    for (int d = 0; d < W; d++) {
      hdr_at[(size_t)d] = hdr_total;
      hdr_total += d == me ? 0 : hdr_bytes(d);
    }
    uint8_t* hstage = (uint8_t*)x.stage_bytes(hdr_total ? hdr_total : 16);
    memset(hstage, 0, hdr_total);
    for (int d = 0; d < W; d++) {
      if (d == me) continue;
      const Out& o = outs[(size_t)d];
      uint64_t* h = (uint64_t*)(hstage + hdr_at[(size_t)d]);
      h[0] = EXCH_MAGIC;
      h[1] = o.entries.size();
      h[2] = o.inl ? 1 : 0;
      h[3] = o.payload;
      uint64_t* q = h + 4;
      for (auto& en : o.entries) {
        *q++ = (uint64_t)en.partition;
        *q++ = (uint64_t)en.file_id;
        *q++ = (uint64_t)en.rows;
        for (uint64_t b : en.sizes) *q++ = b;
      }
    }
    DevPtr hdev = dev_alloc(hdr_total + 16, x.st());
    if (hdr_total) CUDA_CHECK(cudaMemcpyAsync(hdev->ptr, hstage, hdr_total, cudaMemcpyHostToDevice, x.st()));
    PackList pl;
    std::vector<DevColumn> keep_cols;  // converted string columns of large messages, alive until the sends are enqueued
    struct SendOp { const void* ptr; uint64_t bytes; int peer; };
    std::vector<SendOp> sends;
    uint64_t sent = 0;
    for (int d = 0; d < W; d++) {
      if (d == me) continue;
      const Out& o = outs[(size_t)d];
      uint8_t* sl = (uint8_t*)sendbuf->ptr + (size_t)d * slot;
      pl.copy((const uint8_t*)hdev->ptr + hdr_at[(size_t)d], sl, hdr_bytes(d));
      uint8_t* cur = sl + hdr_bytes(d);
      sent += o.payload;
      for (size_t k = 0; k < o.entries.size(); k++) {
        const Piece& pc = o.src[k]->piece;
        const ExchEntry& en = o.entries[k];
        size_t si = 0;
        for (size_t c = 0; c < ncols; c++) {
          DevColumn col = slice_column(pc.batch->cols[c], pc.r0, pc.r1);
          const uint64_t bv = en.sizes[3 * c], bd = en.sizes[3 * c + 1], bc = en.sizes[3 * c + 2];
          if (o.inl) {
            if (bv) pl.copy(col.valid, cur, bv);
            cur += al16(bv);
            if (col.type.id == TypeId::Utf8) {
              pl.strings(col, cur, cur + al16(bd), bc);
            } else if (bd) {
              pl.copy(col.data, cur, bd);
            }
            cur += al16(bd) + al16(bc);
          } else {
            if (bv) sends.push_back(SendOp{col.valid, bv, d});
            if (col.type.id == TypeId::Utf8) {
              DevColumn u = col.phys == PH_STRVIEW ? as_utf8(x, col, (int64_t)pc.str_bytes[si]) : col;
              const uint8_t* chars = u.chars;
              if (col.phys != PH_STRVIEW) {
                // Arrow slice: the receiver wants offsets that start at 0
                DevPtr ro = dev_alloc((size_t)(u.n + 1) * 4 + 64, x.st());
                DevPtr fl = dev_alloc(16, x.st());
                launch_rebase_offsets((const int32_t*)u.data, u.n + 1, (int32_t*)ro->ptr, (int32_t*)fl->ptr, x.st());
                x.count();
                // first offset of the slice: needed on the host to position the chars pointer
                const int32_t first = x.get<int32_t>(fl->ptr);
                chars = u.chars + first;
                u.data = (const uint8_t*)ro->ptr;
                u.keep.push_back(ro);
              }
              keep_cols.push_back(u);
              sends.push_back(SendOp{u.data, bd, d});
              if (bc) sends.push_back(SendOp{chars, bc, d});
            } else if (bd) {
              sends.push_back(SendOp{col.data, bd, d});
            }
          }
          if (col.type.id == TypeId::Utf8) si++;
        }
      }
    }
    pl.run(x);
    // ---- round 1: fixed-size slots ---------------------------------------------------------------------------
    std::lock_guard<std::mutex> cg(e->comm_mu);
    NCCL_CHECK(N.GroupStart());
    for (int d = 0; d < W; d++) {
      if (d == me) continue;
      NCCL_CHECK(N.Send((const uint8_t*)sendbuf->ptr + (size_t)d * slot, slot, kNcclUint8, d, e->comm, x.st()));
      NCCL_CHECK(N.Recv((uint8_t*)recvbuf->ptr + (size_t)d * slot, slot, kNcclUint8, d, e->comm, x.st()));
    }
    NCCL_CHECK(N.GroupEnd());
    x.count(1);
    // incoming headers: every peer used hdr_bytes(me)
    const size_t hb = hdr_bytes(me);
    std::vector<const uint64_t*> rh((size_t)W, nullptr);
    for (int d = 0; d < W; d++)
      if (d != me) rh[(size_t)d] = (const uint64_t*)x.fetch_bytes((const uint8_t*)recvbuf->ptr + (size_t)d * slot, hb);
    x.sync();
    // ---- parse, allocate, round 2 ------------------------------------------------------------------------------
    struct RecvOp { void* ptr; uint64_t bytes; int peer; };
    std::vector<RecvOp> recvs;
    struct Incoming { int p; Piece piece; };
    std::vector<Incoming> incoming;
    uint64_t recvd = 0;
    for (int d = 0; d < W; d++) {
      if (d == me) continue;
      const uint64_t* h = rh[(size_t)d];
      if (h[0] != EXCH_MAGIC) throw EngineError(B200_ERR_CUDA, "exchange: bad header from rank " + std::to_string(d));
      const uint64_t n_ent = h[1];
      const bool inl = h[2] != 0;
      recvd += h[3];
      if (32 + n_ent * entry_bytes() > hb) throw EngineError(B200_ERR_INVALID, "exchange: header overflow");
      const uint64_t* q = h + 4;
      const uint8_t* cur = (const uint8_t*)recvbuf->ptr + (size_t)d * slot + hb;
      for (uint64_t k = 0; k < n_ent; k++) {
        const int64_t part = (int64_t)*q++, fid = (int64_t)*q++, rows = (int64_t)*q++;
        auto b = std::make_shared<DevBatch>();
        b->n = rows;
        std::vector<int64_t> sb;
        for (size_t c = 0; c < ncols; c++) {
          const uint64_t bv = *q++, bd = *q++, bc = *q++;
          DevColumn col;
          col.name = schema[c].name;
          col.type = schema[c].type;
          col.phys = phys_of(col.type);
          col.n = rows;
          col.nullable = bv != 0;
          auto place = [&](uint64_t bytes) -> const uint8_t* {
            if (inl) {
              const uint8_t* ptr = cur;
              cur += al16(bytes);
              col.keep.push_back(recvbuf);
              return ptr;
            }
            DevPtr dp = dev_alloc((size_t)bytes + 64, x.st());
            col.keep.push_back(dp);
            if (bytes) recvs.push_back(RecvOp{dp->ptr, bytes, d});
            return (const uint8_t*)dp->ptr;
          };
          const uint8_t* pv = place(bv);
          if (bv) col.valid = pv;
          col.data = place(bd);
          if (col.type.id == TypeId::Utf8) {
            col.chars = place(bc);
            col.chars_bytes = (int64_t)bc;
            sb.push_back((int64_t)bc);
          } else if (inl) {
            cur += al16(bc);
          }
          b->cols.push_back(col);
        }
        Incoming in;
        in.p = (int)part;
        in.piece.file_id = fid;
        in.piece.batch = b;
        in.piece.r0 = 0;
        in.piece.r1 = rows;
        in.piece.src_rank = d;
        in.piece.str_bytes = sb;
        incoming.push_back(in);
      }
    }
    if (!sends.empty() || !recvs.empty()) {
      NCCL_CHECK(N.GroupStart());
      for (auto& so : sends) NCCL_CHECK(N.Send(so.ptr, so.bytes, kNcclUint8, so.peer, e->comm, x.st()));
      for (auto& ro : recvs) NCCL_CHECK(N.Recv(ro.ptr, ro.bytes, kNcclUint8, ro.peer, e->comm, x.st()));
      NCCL_CHECK(N.GroupEnd());
      x.count(1);
    }
    // ---- install ---------------------------------------------------------------------------------------------
    {
      std::lock_guard<std::mutex> g(e->mu);
      for (int p = 0; p < P; p++) {
        if (goes_to(p, me)) continue;
        e->shuffle.erase(ShuffleKey{job, stage, (int64_t)p});  // handed over to its owner
      }
      for (auto& in : incoming) {
        auto& v = e->shuffle[ShuffleKey{job, stage, (int64_t)in.p}];
        v.erase(std::remove_if(v.begin(), v.end(), [&](const Piece& pc) { return pc.src_rank == in.piece.src_rank && pc.file_id == in.piece.file_id; }), v.end());
        v.push_back(in.piece);
        std::stable_sort(v.begin(), v.end(), [](const Piece& a, const Piece& b) { return a.src_rank != b.src_rank ? a.src_rank < b.src_rank : a.file_id < b.file_id; });
      }
    }
    *sent_out = sent;
    *recv_out = recvd;
  }
};

// ------------------------------------------------------------------------------------------------
// Parquet scan: DataSourceExec + ParquetSource with the page decode on the device
// (ballista/core/proto/datafusion.proto:1058-1077; registration path benchmarks/src/bin/tpch.rs:684-693).
// The host parses the footer and the page headers (parquet_meta.hpp), ships the raw bytes of the REQUESTED column chunks
// to HBM (projection push-down: other columns never cross the bus) and csrc/device/parquet.cu decodes them.
// ------------------------------------------------------------------------------------------------
struct PqHostColumn {
  pq::SchemaElement se;
  int leaf = -1;
  bool optional = false;
  std::vector<PqPage> pages, dicts;
  int64_t rows = 0, dict_entries = 0;
  DevPtr raw;  // the column's chunks, back to back (as stored in the file: possibly compressed)
  DevPtr dec;  // Snappy-compressed chunks: the pages' payloads rebuilt uncompressed
  std::vector<PqDecompJob> jobs;
  std::vector<uint8_t> page_in_dec, dict_in_dec;  // per page: its payload pointer is an offset into `dec` until `dec` exists
  size_t dec_bytes = 0;
};

static DataType pq_arrow_type(const pq::SchemaElement& se, int* out_kind) {
  const bool is_decimal = se.logical == 5 || se.converted == 5;
  const bool is_date = se.logical == 6 || se.converted == 6;
  switch (se.type) {
    case pq::T_BOOLEAN: *out_kind = PQ_OUT_BOOL8; return DataType(TypeId::Bool);
    case pq::T_INT32:
      if (is_decimal) { *out_kind = PQ_OUT_DEC128; return DataType::decimal(se.precision, se.scale); }
      *out_kind = PQ_OUT_I32;
      return DataType(is_date ? TypeId::Date32 : TypeId::Int32);
    case pq::T_INT64:
      if (is_decimal) { *out_kind = PQ_OUT_DEC128; return DataType::decimal(se.precision, se.scale); }
      *out_kind = PQ_OUT_I64;
      return DataType(TypeId::Int64);
    case pq::T_DOUBLE: *out_kind = PQ_OUT_F64; return DataType(TypeId::Float64);
    case pq::T_BYTE_ARRAY: *out_kind = PQ_OUT_STRVIEW; return DataType(TypeId::Utf8);
    case pq::T_FLBA:
      if (is_decimal && se.type_length >= 1 && se.type_length <= 16) { *out_kind = PQ_OUT_DEC128; return DataType::decimal(se.precision, se.scale); }
      break;
    default: break;
  }
  throw EngineError(B200_ERR_UNSUPPORTED, "parquet column '" + se.name + "': physical/logical type not supported by the device scan");
}

DevBatchPtr scan_parquet(const Exec& x, const std::string& path, const std::vector<std::string>& want) {
  ScopeTimer tm("parquet_scan");
  FILE* f = fopen(path.c_str(), "rb");
  if (!f) throw EngineError(B200_ERR_NOT_FOUND, "cannot open " + path);
  fseek(f, 0, SEEK_END);
  const size_t fsize = (size_t)ftell(f);
  fseek(f, 0, SEEK_SET);
  struct Pinned {
    uint8_t* p = nullptr;
    ~Pinned() {
      if (p) cudaFreeHost(p);
    }
  } file;
  if (cudaHostAlloc((void**)&file.p, fsize + 64, cudaHostAllocDefault) != cudaSuccess) {
    fclose(f);
    throw EngineError(B200_ERR_OOM, "pinned staging for the parquet file");
  }
  const size_t got = fread(file.p, 1, fsize, f);
  fclose(f);
  if (got != fsize) throw EngineError(B200_ERR_INVALID, "short read on " + path);
  pq::FileMeta fm;
  try {
    fm = pq::read_file_meta(file.p, fsize);
  } catch (const std::runtime_error& ex) {
    throw EngineError(B200_ERR_INVALID, ex.what());
  }
  if (fm.schema.empty()) throw EngineError(B200_ERR_INVALID, "parquet: empty schema");
  const size_t n_leaves = fm.schema.size() - 1;
  if ((size_t)fm.schema[0].num_children != n_leaves) throw EngineError(B200_ERR_UNSUPPORTED, "parquet: nested schemas are not supported by the device scan");
  std::vector<PqHostColumn> cols;
  std::vector<std::string> names = want;
  if (names.empty())
    for (size_t i = 1; i < fm.schema.size(); i++) names.push_back(fm.schema[i].name);
  for (auto& nm : names) {
    PqHostColumn c;
    for (size_t i = 1; i < fm.schema.size(); i++)
      if (fm.schema[i].name == nm) c.leaf = (int)i - 1;
    if (c.leaf < 0) throw EngineError(B200_ERR_INVALID, "parquet: no column named " + nm);
    c.se = fm.schema[(size_t)c.leaf + 1];
    if (c.se.num_children) throw EngineError(B200_ERR_UNSUPPORTED, "parquet: nested column " + nm);
    if (c.se.repetition == 2) throw EngineError(B200_ERR_UNSUPPORTED, "parquet: repeated column " + nm);
    c.optional = c.se.repetition == 1;
    cols.push_back(c);
  }
  cudaStream_t st = x.st();
  int64_t n_rows = 0;
  for (auto& rg : fm.row_groups) n_rows += rg.num_rows;
  // ---- raw bytes to HBM + page tables ---------------------------------------------------------------------------------
  for (auto& c : cols) {
    size_t total = 0;
    for (auto& rg : fm.row_groups) {
      if ((size_t)c.leaf >= rg.columns.size()) throw EngineError(B200_ERR_INVALID, "parquet: row group without column " + c.se.name);
      total += (size_t)rg.columns[(size_t)c.leaf].total_compressed;
    }
    c.raw = dev_alloc(total + 64, st);
    size_t dpos = 0;
    for (auto& rg : fm.row_groups) {
      const pq::ColumnChunkMeta& cm = rg.columns[(size_t)c.leaf];
      if (cm.codec != 0 && cm.codec != 1)
        throw EngineError(B200_ERR_UNSUPPORTED, "parquet: column " + c.se.name + " uses compression codec " + std::to_string(cm.codec) + " (the device scan reads UNCOMPRESSED and SNAPPY pages)");
      const bool snappy = cm.codec == 1;
      int64_t start = cm.data_page_offset;
      if (cm.dictionary_page_offset > 0 && cm.dictionary_page_offset < start) start = cm.dictionary_page_offset;
      if (start < 0 || (size_t)start + (size_t)cm.total_compressed > fsize) throw EngineError(B200_ERR_INVALID, "parquet: column chunk outside the file");
      CUDA_CHECK(cudaMemcpyAsync((uint8_t*)c.raw->ptr + dpos, file.p + start, (size_t)cm.total_compressed, cudaMemcpyHostToDevice, st));
      const uint8_t* hp = file.p + start;
      const uint8_t* hend = hp + cm.total_compressed;
      const uint8_t* dbase = (const uint8_t*)c.raw->ptr + dpos;
      int64_t chunk_dict_base = c.dict_entries, chunk_values = 0;
      while (hp < hend && chunk_values < cm.num_values) {
        pq::PageHeader h;
        try {
          h = pq::read_page_header(hp, hend);
        } catch (const std::runtime_error& ex) {
          throw EngineError(B200_ERR_INVALID, ex.what());
        }
        const uint8_t* payload = hp + h.header_bytes;
        if (payload + h.compressed_size > hend) throw EngineError(B200_ERR_INVALID, "parquet: page overruns its chunk");
        const uint8_t* dev_payload = dbase + (payload - (file.p + start));
        PqPage pg;
        memset(&pg, 0, sizeof pg);
        pg.n_values = (uint32_t)h.num_values;
        uint32_t plen = (uint32_t)h.compressed_size;   // bytes of the payload the decode kernels will see
        const bool is_data = h.type == pq::P_DATA || h.type == pq::P_DATA_V2;
        const uint32_t v2_levels = h.type == pq::P_DATA_V2 ? (uint32_t)(h.rep_bytes + h.def_bytes) : 0;
        const bool in_dec = snappy && (h.type == pq::P_DICTIONARY || is_data);
        if (in_dec) {
          // the page payload is rebuilt, uncompressed, at c.dec + dec_bytes (the addresses are patched in once c.dec exists)
          plen = (uint32_t)h.uncompressed_size;
          if (v2_levels > (uint32_t)h.compressed_size || v2_levels > plen) throw EngineError(B200_ERR_INVALID, "parquet: level section overruns the page");
          PqDecompJob lv, vj;
          memset(&lv, 0, sizeof lv);
          memset(&vj, 0, sizeof vj);
          if (v2_levels) {  // V2: the levels are never compressed
            lv.src = dev_payload;
            lv.dst = (uint8_t*)c.dec_bytes;
            lv.src_len = lv.dst_len = v2_levels;
            lv.raw_copy = 1;
            c.jobs.push_back(lv);
          }
          vj.src = dev_payload + v2_levels;
          vj.dst = (uint8_t*)(c.dec_bytes + v2_levels);
          vj.src_len = (uint32_t)h.compressed_size - v2_levels;
          vj.dst_len = plen - v2_levels;
          vj.raw_copy = (h.type == pq::P_DATA_V2 && !h.v2_compressed) ? 1 : 0;
          c.jobs.push_back(vj);
          pg.data = (const uint8_t*)c.dec_bytes;   // offset for now
          c.dec_bytes += ((size_t)plen + 15) & ~(size_t)15;
        } else {
          pg.data = dev_payload;
        }
        if (h.type == pq::P_DICTIONARY) {
          if (h.encoding != pq::E_PLAIN && h.encoding != pq::E_PLAIN_DICTIONARY) throw EngineError(B200_ERR_UNSUPPORTED, "parquet: dictionary page encoding");
          pg.val_off = 0;
          pg.val_len = plen;
          pg.row0 = c.dict_entries;
          chunk_dict_base = c.dict_entries;
          c.dict_entries += h.num_values;
          c.dicts.push_back(pg);
          c.dict_in_dec.push_back(in_dec ? 1 : 0);
        } else if (is_data) {
          if (h.type == pq::P_DATA) {
            if (c.optional) {
              if (h.def_encoding != pq::E_RLE) throw EngineError(B200_ERR_UNSUPPORTED, "parquet: definition levels not RLE encoded");
              if (plen < 4) throw EngineError(B200_ERR_INVALID, "parquet: page too short for its level section");
              pg.v1_levels = 1;   // [u32 length][levels][values]: resolved on the device
            }
            pg.val_off = 0;
            pg.val_len = plen;
          } else {
            if (v2_levels > plen) throw EngineError(B200_ERR_INVALID, "parquet: level section overruns the page");
            pg.def_off = (uint32_t)h.rep_bytes;
            pg.def_len = c.optional ? (uint32_t)h.def_bytes : 0;
            pg.val_off = v2_levels;
            pg.val_len = plen - v2_levels;
          }
          if (h.encoding == pq::E_PLAIN) pg.encoding = 0;
          else if (h.encoding == pq::E_PLAIN_DICTIONARY || h.encoding == pq::E_RLE_DICTIONARY) pg.encoding = 1;
          else if (h.encoding == pq::E_RLE && c.se.type == pq::T_BOOLEAN) pg.encoding = 2;
          else throw EngineError(B200_ERR_UNSUPPORTED, "parquet: column " + c.se.name + " uses encoding " + std::to_string(h.encoding) + " (supported: PLAIN, RLE_DICTIONARY)");
          pg.row0 = c.rows;
          pg.dict_base = chunk_dict_base;
          c.rows += h.num_values;
          chunk_values += h.num_values;
          c.pages.push_back(pg);
          c.page_in_dec.push_back(in_dec ? 1 : 0);
        }  // index pages etc.: skipped
        hp = payload + h.compressed_size;
      }
      dpos += (size_t)cm.total_compressed;
    }
    if (c.rows != n_rows) throw EngineError(B200_ERR_INVALID, "parquet: column " + c.se.name + " has " + std::to_string(c.rows) + " values, the file " + std::to_string(n_rows) + " rows");
    if (c.dec_bytes) {
      // Snappy: rebuild every page payload uncompressed in HBM (one warp per page), then decode as usual
      c.dec = dev_alloc(c.dec_bytes + 64, st);
      uint8_t* base = (uint8_t*)c.dec->ptr;
      for (auto& j : c.jobs) j.dst = base + (size_t)j.dst;
      for (size_t i = 0; i < c.pages.size(); i++)
        if (c.page_in_dec[i]) c.pages[i].data = base + (size_t)c.pages[i].data;
      for (size_t i = 0; i < c.dicts.size(); i++)
        if (c.dict_in_dec[i]) c.dicts[i].data = base + (size_t)c.dicts[i].data;
      DevPtr dj = dev_alloc(c.jobs.size() * sizeof(PqDecompJob), st);
      CUDA_CHECK(cudaMemcpyAsync(dj->ptr, c.jobs.data(), c.jobs.size() * sizeof(PqDecompJob), cudaMemcpyHostToDevice, st));
      DevPtr err = dev_alloc(16, st);
      CUDA_CHECK(cudaMemsetAsync(err->ptr, 0, 16, st));
      {
        KernelTimer kt(x, "parquet_snappy", (uint64_t)c.raw->bytes + (uint64_t)c.dec_bytes);
        launch_pq_snappy((const PqDecompJob*)dj->ptr, (int)c.jobs.size(), (unsigned int*)err->ptr, st);
        x.count();
      }
      const unsigned int* herr = x.fetch<unsigned int>(err->ptr);
      const std::string cname = c.se.name;
      x.defer([herr, cname, dj, err]() {
        if (*herr) throw EngineError(B200_ERR_INVALID, "parquet: corrupt Snappy data in column " + cname);
      });
    }
  }
  // ---- decode ------------------------------------------------------------------------------------------------------------
  struct ColWork {
    PqColumn pc;
    DataType type;
    DevPtr d_pages, d_dicts, valid, nonnull, dense_base, total, dict, out;
    const unsigned long long* h_total = nullptr;
    int width = 0;
  };
  std::vector<ColWork> work(cols.size());
  auto upload = [&](const std::vector<PqPage>& v) {
    DevPtr d = dev_alloc(std::max<size_t>(v.size(), 1) * sizeof(PqPage), st);
    if (!v.empty()) CUDA_CHECK(cudaMemcpyAsync(d->ptr, v.data(), v.size() * sizeof(PqPage), cudaMemcpyHostToDevice, st));  // pageable: staged before returning
    return d;
  };
  for (size_t ci = 0; ci < cols.size(); ci++) {
    PqHostColumn& c = cols[ci];
    ColWork& w = work[ci];
    memset(&w.pc, 0, sizeof w.pc);
    int kind = 0;
    w.type = pq_arrow_type(c.se, &kind);
    w.pc.phys = c.se.type;
    w.pc.type_length = c.se.type_length;
    w.pc.out_kind = kind;
    w.width = kind == PQ_OUT_I32 ? 4 : (kind == PQ_OUT_I64 || kind == PQ_OUT_F64) ? 8 : kind == PQ_OUT_BOOL8 ? 1 : 16;
    w.d_pages = upload(c.pages);
    w.d_dicts = upload(c.dicts);
    if (c.dict_entries) {
      w.dict = dev_alloc((size_t)c.dict_entries * (size_t)w.width + 64, st);
      w.pc.dict = w.dict->ptr;
      launch_pq_dict(w.pc, (const PqPage*)w.d_dicts->ptr, (int)c.dicts.size(), st);
      x.count();
    }
    if (c.optional) {
      w.valid = dev_alloc((size_t)std::max<int64_t>(n_rows, 1) + 64, st);
      w.nonnull = dev_alloc(std::max<size_t>(c.pages.size(), 1) * 4, st);
      w.dense_base = dev_alloc(std::max<size_t>(c.pages.size(), 1) * 8, st);
      w.total = dev_alloc(16, st);
      CUDA_CHECK(cudaMemsetAsync(w.total->ptr, 0, 16, st));
      launch_pq_levels((const PqPage*)w.d_pages->ptr, (int)c.pages.size(), (uint8_t*)w.valid->ptr, (uint32_t*)w.nonnull->ptr, (unsigned long long*)w.total->ptr, st);
      launch_pq_page_scan((const uint32_t*)w.nonnull->ptr, (int)c.pages.size(), (unsigned long long*)w.dense_base->ptr, st);
      x.count(2);
      w.h_total = x.fetch<unsigned long long>(w.total->ptr);
    }
  }
  x.sync();  // one read-back for all nullable columns: which of them really contain NULLs
  auto out = std::make_shared<DevBatch>();
  out->n = n_rows;
  for (size_t ci = 0; ci < cols.size(); ci++) {
    PqHostColumn& c = cols[ci];
    ColWork& w = work[ci];
    const bool has_nulls = c.optional && (int64_t)*w.h_total != n_rows;
    w.out = dev_alloc((size_t)std::max<int64_t>(n_rows, 1) * (size_t)w.width + 64, st);
    {
      KernelTimer kt(x, "parquet_decode_values", (uint64_t)n_rows * (uint64_t)w.width);
      if (!has_nulls) {
        launch_pq_values(w.pc, (const PqPage*)w.d_pages->ptr, (int)c.pages.size(), nullptr, nullptr, w.out->ptr, st);
        x.count();
      } else {
        DevPtr dense = dev_alloc((size_t)std::max<int64_t>(n_rows, 1) * (size_t)w.width + 64, st);
        launch_pq_values(w.pc, (const PqPage*)w.d_pages->ptr, (int)c.pages.size(), (const unsigned long long*)w.dense_base->ptr, (const uint32_t*)w.nonnull->ptr, dense->ptr, st);
        launch_pq_expand((const PqPage*)w.d_pages->ptr, (int)c.pages.size(), (const unsigned long long*)w.dense_base->ptr, (const uint8_t*)w.valid->ptr, dense->ptr,
                         w.out->ptr, w.width, st);
        x.count(2);
      }
    }
    DevColumn col;
    col.name = c.se.name;
    col.type = w.type;
    col.n = n_rows;
    col.nullable = has_nulls;
    col.phys = w.pc.out_kind == PQ_OUT_STRVIEW ? PH_STRVIEW : phys_of(w.type);
    col.data = (const uint8_t*)w.out->ptr;
    col.keep.push_back(w.out);
    if (has_nulls) {
      col.valid = (const uint8_t*)w.valid->ptr;
      col.keep.push_back(w.valid);
    }
    if (col.phys == PH_STRVIEW) {
      // registered tables use the canonical Arrow layout (offsets + contiguous characters): the views into the raw pages
      // are compacted once, here, and the raw pages are released
      col.keep.push_back(c.raw);
      if (c.dec) col.keep.push_back(c.dec);
      if (w.dict) col.keep.push_back(w.dict);
      col = as_utf8(x, col);
    }
    out->cols.push_back(col);
  }
  prepack_short_strings(x, *out);
  x.sync();
  return out;
}

void collect_nodes(const PlanNode& n, b200_stage* s) {
  s->metric_index[&n] = (int)s->metrics.size();
  OpMetrics m;
  m.name = n.op_name;
  s->metrics.push_back(m);
  for (auto& c : n.children) collect_nodes(*c, s);
}

int table_id(const std::string& name) {
  static const char* names[] = {"lineitem", "orders", "customer", "supplier", "part", "partsupp", "nation", "region"};
  for (int i = 0; i < 8; i++)
    if (name == names[i]) return i;
  return -1;
}

template <class F>
int guard(F&& f) {
  try {
    f();
    return B200_OK;
  } catch (const EngineError& e) {
    g_err = e.what();
    return e.code;
  } catch (const std::bad_alloc&) {
    g_err = "host out of memory";
    return B200_ERR_OOM;
  } catch (const std::exception& e) {
    g_err = e.what();
    return B200_ERR_INVALID;
  } catch (...) {
    g_err = "unknown error";
    return B200_ERR_INVALID;
  }
}

}  // namespace

// ================================================================================================
// C ABI
// ================================================================================================
// ---- exchange window (fused shuffle): allocate, publish through CUDA IPC, map every peer's ---------------------------------
static void release_window(b200_engine* e) {
  for (size_t d = 0; d < e->win_peer.size(); d++)
    if (e->win_peer[d] && (int)d != e->rank) cudaIpcCloseMemHandle(e->win_peer[d]);
  e->win_peer.clear();
  if (e->win_local) cudaFree(e->win_local);
  e->win_local = nullptr;
  e->win_bytes = e->win_used = 0;
}

// all-gather of one fixed-size record per executor over the exchange communicator (setup path only)
static void comm_allgather(b200_engine* e, const void* mine, void* all, size_t rec) {
  NcclApi& N = NcclApi::get();
  const int W = e->world, me = e->rank;
  uint8_t* dev = nullptr;
  CUDA_CHECK(cudaMalloc((void**)&dev, rec * (size_t)W));
  try {
    CUDA_CHECK(cudaMemcpyAsync(dev + rec * (size_t)me, mine, rec, cudaMemcpyHostToDevice, e->stream));
    NCCL_CHECK(N.GroupStart());
    for (int d = 0; d < W; d++) {
      if (d == me) continue;
      NCCL_CHECK(N.Send(dev + rec * (size_t)me, rec, kNcclUint8, d, e->comm, e->stream));
      NCCL_CHECK(N.Recv(dev + rec * (size_t)d, rec, kNcclUint8, d, e->comm, e->stream));
    }
    NCCL_CHECK(N.GroupEnd());
    CUDA_CHECK(cudaMemcpyAsync(all, dev, rec * (size_t)W, cudaMemcpyDeviceToHost, e->stream));
    CUDA_CHECK(cudaStreamSynchronize(e->stream));
  } catch (...) {
    cudaFree(dev);
    throw;
  }
  cudaFree(dev);
}

// Collective (called from b200_engine_comm_init on every executor).  Any executor that cannot provide or map a window
// makes all of them run without one: the fused shuffle needs every peer, the two-step exchange none.
static void setup_window(b200_engine* e) {
  const int W = e->world, me = e->rank;
  struct Rec {
    cudaIpcMemHandle_t h;
    uint64_t bytes, ok;
  };
  Rec mine;
  memset(&mine, 0, sizeof mine);
  const size_t want = (e->win_config_bytes + 4095) & ~(size_t)4095;
  uint8_t* ptr = nullptr;
  if (cudaMalloc((void**)&ptr, want) == cudaSuccess && cudaIpcGetMemHandle(&mine.h, ptr) == cudaSuccess) {
    mine.bytes = want;
    mine.ok = 1;
  } else {
    cudaGetLastError();
    if (ptr) cudaFree(ptr);
    ptr = nullptr;
  }
  std::vector<Rec> all((size_t)W);
  comm_allgather(e, &mine, all.data(), sizeof(Rec));
  bool ok = true;
  for (auto& r : all) ok = ok && r.ok && r.bytes == want;
  std::vector<uint8_t*> peer((size_t)W, nullptr);
  if (ok) {
    for (int d = 0; d < W && ok; d++) {
      if (d == me) {
        peer[(size_t)d] = ptr;
        continue;
      }
      void* m = nullptr;
      if (cudaIpcOpenMemHandle(&m, all[(size_t)d].h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
        cudaGetLastError();
        ok = false;
      }
      peer[(size_t)d] = (uint8_t*)m;
    }
  }
  // second round: did everyone manage to map everyone?
  uint64_t flag = ok ? 1 : 0;
  std::vector<uint64_t> flags((size_t)W, 0);
  comm_allgather(e, &flag, flags.data(), sizeof flag);
  for (uint64_t f : flags) ok = ok && f;
  if (!ok) {
    for (int d = 0; d < W; d++)
      if (d != me && peer[(size_t)d]) cudaIpcCloseMemHandle(peer[(size_t)d]);
    if (ptr) cudaFree(ptr);
    return;
  }
  e->win_local = ptr;
  e->win_bytes = want;
  e->win_used = 0;
  e->win_peer = peer;
}


extern "C" {

const char* b200_version(void) { return "b200exec 0.1 sm_100a"; }
const char* b200_last_error(void) { return g_err.c_str(); }

// Ingest is a host<->GPU pipeline (pinned staging, a pool of narrowing threads, DMA): it only reaches the PCIe rate when
// the host side runs on the NUMA node the GPU hangs off -- across the socket interconnect the same copies run at about
// half speed.  The thread that creates the engine (and every thread it starts later, e.g. the ingest pool) is therefore
// bound to the CPUs of the GPU's node; pinned buffers it allocates afterwards are first-touched there.
// B200_NUMA_BIND=0 keeps the caller's affinity.
static void bind_to_gpu_numa_node(int device) {
  const char* env = getenv("B200_NUMA_BIND");
  if (env && env[0] == '0') return;
  char busid[64] = {0};
  if (cudaDeviceGetPCIBusId(busid, sizeof busid, device) != cudaSuccess) return;
  for (char* c = busid; *c; c++) *c = (char)tolower(*c);
  char path[256];
  snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", busid);
  int node = -1;
  if (FILE* f = fopen(path, "r")) {
    if (fscanf(f, "%d", &node) != 1) node = -1;
    fclose(f);
  }
  if (node < 0) return;
  snprintf(path, sizeof path, "/sys/devices/system/node/node%d/cpulist", node);
  FILE* f = fopen(path, "r");
  if (!f) return;
  char list[4096] = {0};
  const size_t got = fread(list, 1, sizeof list - 1, f);
  fclose(f);
  if (!got) return;
  cpu_set_t want, cur, both;
  CPU_ZERO(&want);
  for (char* p = list; *p;) {
    char* end = nullptr;
    long a = strtol(p, &end, 10);
    if (end == p) break;
    long b = a;
    if (*end == '-') b = strtol(end + 1, &end, 10);
    for (long c = a; c <= b && c < CPU_SETSIZE; c++) CPU_SET((int)c, &want);
    p = (*end == ',') ? end + 1 : end;
    if (*end != ',' ) break;
  }
  if (sched_getaffinity(0, sizeof cur, &cur) != 0) return;
  CPU_AND(&both, &want, &cur);
  if (CPU_COUNT(&both) == 0) return;
  sched_setaffinity(0, sizeof both, &both);
}

int b200_engine_create(int device, uint64_t pool_bytes, int rank, int world, b200_engine** out) {
  return guard([&] {
    if (!out) throw EngineError(B200_ERR_INVALID, "null out pointer");
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0)
      throw EngineError(B200_ERR_CUDA, std::string("no CUDA device available: the B200 engine has no CPU path (") + cudaGetErrorString(ce) + ")");
    if (device < 0 || device >= ndev) throw EngineError(B200_ERR_INVALID, "bad device ordinal");
    CUDA_CHECK(cudaSetDevice(device));
    bind_to_gpu_numa_node(device);
    auto* e = new b200_engine();
    e->device = device;
    e->rank = rank;
    e->world = world;
    cudaDeviceProp prop;
    CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
    e->sm_count = prop.multiProcessorCount;
    CUDA_CHECK(cudaStreamCreateWithFlags(&e->own_stream, cudaStreamNonBlocking));
    e->stream = e->own_stream;
    cudaMemPool_t pool;
    CUDA_CHECK(cudaDeviceGetDefaultMemPool(&pool, device));
    uint64_t thr = pool_bytes ? pool_bytes : UINT64_MAX;
    CUDA_CHECK(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr));
    *out = e;
  });
}

void b200_engine_destroy(b200_engine* e) {
  if (!e) return;
  cudaSetDevice(e->device);
  cudaStreamSynchronize(e->stream);
  e->tables.clear();
  e->shuffle.clear();
  e->packed_cache.clear();
  e->plan_cache.clear();
  cudaStreamSynchronize(e->stream);
  for (auto& sl : e->nslot) {
    if (sl.pinned) cudaFreeHost(sl.pinned);
    if (sl.dev) cudaFree(sl.dev);
    if (sl.done) cudaEventDestroy(sl.done);
  }
  release_window(e);
  if (e->comm && NcclApi::get().ok()) NcclApi::get().CommDestroy(e->comm);
  if (e->export_arena) cudaFreeHost(e->export_arena);
  if (e->own_stream) cudaStreamDestroy(e->own_stream);
  delete e;
}

int b200_engine_set_stream(b200_engine* e, void* cuda_stream) {
  return guard([&] {
    CUDA_CHECK(cudaStreamSynchronize(e->stream));
    e->stream = cuda_stream ? (cudaStream_t)cuda_stream : e->own_stream;
  });
}
int b200_engine_synchronize(b200_engine* e) {
  return guard([&] {
    CUDA_CHECK(cudaSetDevice(e->device));
    CUDA_CHECK(cudaStreamSynchronize(e->stream));
  });
}
uint64_t b200_engine_kernel_launches(b200_engine* e) { return e->launches; }
uint64_t b200_engine_counter(b200_engine* e, const char* name) {
  const std::string n = name ? name : "";
  if (n == "fused") return e->n_fused;
  if (n == "groupby_partition_first") return e->n_groupby_pf;
  if (n == "fused_static") return e->n_fused_static;
  if (n == "fused_exchanges") return e->fused_exchanges;
  if (n == "exchange_window_bytes") return e->win_bytes;
  if (n == "vm") return e->n_vm;
  if (n == "groupby") return e->n_groupby;
  if (n == "fastfilter") return e->n_fastfilter;
  if (n == "ingest_bytes_saved") return e->narrowed_bytes_saved;
  if (n == "stream_syncs") return e->stream_syncs;
  return 0;
}

int b200_engine_set_config(b200_engine* e, const char* key, const char* value) {
  return guard([&] {
    std::lock_guard<std::mutex> g(e->mu);
    e->config[key] = value;
    if (std::string(key) == "datafusion.execution.batch_size") e->batch_size = std::max<int64_t>(1, atoll(value));
    if (std::string(key) == "b200.ingest.chunk_rows") e->ingest_chunk_rows = std::max<int64_t>(1 << 16, atoll(value));
    if (std::string(key) == "b200.ingest.slots") e->ingest_slots = atoi(value);
    if (std::string(key) == "b200.exchange.window_bytes") e->win_config_bytes = (size_t)strtoull(value, nullptr, 10);  // read by b200_engine_comm_init
    if (std::string(key) == "b200.ingest.threads") e->pool.reset();  // re-created with the new size at the next ingest
    if (std::string(key) == "b200.agg.partition_first.bucket_slots") {
      const uint64_t v = strtoull(value, nullptr, 10);
      e->pf_bucket_slots = v ? std::max<uint64_t>(next_pow2(v), 64) : 0;
    }
    if (std::string(key) == "b200.agg.partition_first.min_rows") e->pf_min_rows = std::max<int64_t>(1, atoll(value));
    if (std::string(key) == "b200.agg.reset_hints") {
      e->agg_hint.clear();
      e->agg_groups.clear();
      e->agg_spec.clear();
    }  // forget which aggregate strategy each plan shape needed
    if (std::string(key) == "b200.metrics.kernel_timing") e->kernel_timing = std::string(value) == "on" || std::string(value) == "1" || std::string(value) == "true";
  });
}

int b200_engine_register_batch(b200_engine* e, const char* table, int partition, struct ArrowArray* batch, struct ArrowSchema* schema) {
  return guard([&] {
    CUDA_CHECK(cudaSetDevice(e->device));
    DevBatchPtr b = import_batch(e, batch, schema);
    Exec x{e, nullptr, nullptr};
    prepack_short_strings(x, *b);
    DevBatchPtr prev;
    {
      std::lock_guard<std::mutex> g(e->mu);
      auto& slot = e->tables[table][partition];
      prev = slot;
      if (!prev) slot = b;
    }
    if (prev) {  // append
      Runner r{x, ""};
      Schema s;
      for (auto& c : prev->cols) s.push_back(Field{c.name, c.type, true});
      DevBatchPtr cat = r.concat({prev, b}, s);
      CUDA_CHECK(cudaStreamSynchronize(e->stream));
      std::lock_guard<std::mutex> g(e->mu);
      e->tables[table][partition] = cat;
    }
  });
}

int b200_engine_drop_table(b200_engine* e, const char* table) {
  return guard([&] {
    CUDA_CHECK(cudaSetDevice(e->device));
    std::lock_guard<std::mutex> g(e->mu);
    e->tables.erase(table);
  });
}

int b200_engine_tpch_generate(b200_engine* e, const char* table, int64_t msf, int partition, int64_t row_begin, int64_t row_end, const char* columns_csv) {
  return guard([&] {
    CUDA_CHECK(cudaSetDevice(e->device));
    int t = table_id(table);
    if (t < 0) throw EngineError(B200_ERR_INVALID, std::string("unknown TPC-H table ") + table);
    std::vector<int> cols;
    if (columns_csv && *columns_csv) {
      std::string s(columns_csv);
      size_t p = 0;
      while (p <= s.size()) {
        size_t q = s.find(',', p);
        if (q == std::string::npos) q = s.size();
        std::string nm = s.substr(p, q - p);
        int found = -1;
        for (int c = 0; c < tpch::kNumCols[t]; c++)
          if (nm == tpch::kCols[t][c].name) found = c;
        if (found < 0) throw EngineError(B200_ERR_INVALID, "unknown column " + nm);
        cols.push_back(found);
        p = q + 1;
      }
    } else {
      for (int c = 0; c < tpch::kNumCols[t]; c++) cols.push_back(c);
    }
    const int64_t n = row_end - row_begin;
    if (n < 0) throw EngineError(B200_ERR_INVALID, "bad row range");
    cudaStream_t st = e->stream;
    auto b = std::make_shared<DevBatch>();
    b->n = n;
    for (int c : cols) {
      const tpch::ColDef& cd = tpch::kCols[t][c];
      DevColumn col;
      col.name = cd.name;
      col.n = n;
      col.nullable = false;
      switch (cd.kind) {
        case tpch::K_I64: col.type = DataType(TypeId::Int64); break;
        case tpch::K_I32: col.type = DataType(TypeId::Int32); break;
        case tpch::K_DEC: col.type = DataType::decimal(15, 2); break;
        case tpch::K_DATE: col.type = DataType(TypeId::Date32); break;
        default: col.type = DataType(TypeId::Utf8);
      }
      col.phys = phys_of(col.type);
      if (cd.kind == tpch::K_STR) {
        DevPtr lens = dev_alloc((size_t)(n + 1) * 4, st);
        DevPtr offs64 = dev_alloc((size_t)(n + 2) * 8, st);
        DevPtr scratch = dev_alloc((size_t)(n / 1024 + 4) * 8, st);
        launch_tpch_str_len(t, c, msf, row_begin, n, (uint32_t*)lens->ptr, st);
        launch_scan_u32_to_u64((const uint32_t*)lens->ptr, (uint64_t*)offs64->ptr, n, (uint64_t*)scratch->ptr, st);
        e->launches += 4;
        uint64_t total = Exec{e, nullptr, nullptr}.get<uint64_t>((const uint64_t*)offs64->ptr + n);
        if (total > 0x7FFFFFFFull) throw EngineError(B200_ERR_UNSUPPORTED, "generated string column exceeds 2 GiB; use more partitions");
        DevPtr offsets = dev_alloc((size_t)(n + 1) * 4 + 64, st);
        DevPtr chars = dev_alloc((size_t)total + 64, st);
        launch_tpch_str_fill(t, c, msf, row_begin, n, (const uint64_t*)offs64->ptr, (int32_t*)offsets->ptr, (uint8_t*)chars->ptr, st);
        e->launches++;
        col.data = (const uint8_t*)offsets->ptr;
        col.chars = (const uint8_t*)chars->ptr;
        col.chars_bytes = (int64_t)total;
        col.keep.push_back(offsets);
        col.keep.push_back(chars);
      } else {
        DevPtr d = dev_alloc((size_t)std::max<int64_t>(n, 1) * col.width() + 64, st);
        launch_tpch_fixed(t, c, cd.kind, msf, row_begin, n, d->ptr, st);
        e->launches++;
        col.data = (const uint8_t*)d->ptr;
        col.keep.push_back(d);
      }
      b->cols.push_back(col);
    }
    prepack_short_strings(Exec{e, nullptr, nullptr}, *b);
    CUDA_CHECK(cudaStreamSynchronize(st));
    std::lock_guard<std::mutex> g(e->mu);
    e->tables[table][partition] = b;
  });
}

// Host-only view of what the device scan would be handed: schema, row counts and the page inventory of every column
// (JSON).  No CUDA call: used by the CPU tests to pin the Thrift footer / page-header reader against pyarrow's metadata.
int b200_parquet_describe(const char* path, char* out, uint64_t cap) {
  return guard([&] {
    if (!path || !out || cap < 2) throw EngineError(B200_ERR_INVALID, "bad argument");
    FILE* f = fopen(path, "rb");
    if (!f) throw EngineError(B200_ERR_NOT_FOUND, std::string("cannot open ") + path);
    fseek(f, 0, SEEK_END);
    const size_t fsize = (size_t)ftell(f);
    fseek(f, 0, SEEK_SET);
    std::vector<uint8_t> buf(fsize);
    const size_t got = fread(buf.data(), 1, fsize, f);
    fclose(f);
    if (got != fsize) throw EngineError(B200_ERR_INVALID, "short read");
    pq::FileMeta fm;
    try {
      fm = pq::read_file_meta(buf.data(), fsize);
    } catch (const std::runtime_error& ex) {
      throw EngineError(B200_ERR_INVALID, ex.what());
    }
    std::string j = "{\"num_rows\":" + std::to_string(fm.num_rows) + ",\"row_groups\":" + std::to_string(fm.row_groups.size()) + ",\"columns\":[";
    for (size_t i = 1; i < fm.schema.size(); i++) {
      const pq::SchemaElement& se = fm.schema[i];
      int64_t data_pages = 0, dict_pages = 0, values = 0, dict_encoded = 0, codec = 0;
      for (auto& rg : fm.row_groups) {
        if (i - 1 >= rg.columns.size()) continue;
        const pq::ColumnChunkMeta& cm = rg.columns[i - 1];
        codec = cm.codec;
        int64_t start = cm.data_page_offset;
        if (cm.dictionary_page_offset > 0 && cm.dictionary_page_offset < start) start = cm.dictionary_page_offset;
        const uint8_t* hp = buf.data() + start;
        const uint8_t* hend = hp + cm.total_compressed;
        int64_t seen = 0;
        while (hp < hend && seen < cm.num_values) {
          pq::PageHeader h = pq::read_page_header(hp, hend);
          if (h.type == pq::P_DICTIONARY) dict_pages++;
          else if (h.type == pq::P_DATA || h.type == pq::P_DATA_V2) {
            data_pages++;
            seen += h.num_values;
            values += h.num_values;
            if (h.encoding == pq::E_PLAIN_DICTIONARY || h.encoding == pq::E_RLE_DICTIONARY) dict_encoded++;
          }
          hp += h.header_bytes + (size_t)h.compressed_size;
        }
      }
      if (i > 1) j += ",";
      j += "{\"name\":\"" + se.name + "\",\"physical\":" + std::to_string(se.type) + ",\"type_length\":" + std::to_string(se.type_length) + ",\"optional\":" +
           (se.repetition == 1 ? "true" : "false") + ",\"logical\":" + std::to_string(se.logical) + ",\"converted\":" + std::to_string(se.converted) +
           ",\"precision\":" + std::to_string(se.precision) + ",\"scale\":" + std::to_string(se.scale) + ",\"codec\":" + std::to_string(codec) +
           ",\"values\":" + std::to_string(values) + ",\"data_pages\":" + std::to_string(data_pages) + ",\"dict_pages\":" + std::to_string(dict_pages) +
           ",\"dict_encoded_pages\":" + std::to_string(dict_encoded) + "}";
    }
    j += "]}";
    if (j.size() + 1 > cap) throw EngineError(B200_ERR_INVALID, "description buffer too small");
    memcpy(out, j.c_str(), j.size() + 1);
  });
}

int b200_engine_register_parquet(b200_engine* e, const char* table, int partition, const char* path, const char* columns_csv) {
  return guard([&] {
    if (!e || !table || !path) throw EngineError(B200_ERR_INVALID, "null argument");
    CUDA_CHECK(cudaSetDevice(e->device));
    std::vector<std::string> cols;
    if (columns_csv && *columns_csv) {
      std::string sct(columns_csv);
      size_t p = 0;
      while (p <= sct.size()) {
        size_t q = sct.find(',', p);
        if (q == std::string::npos) q = sct.size();
        if (q > p) cols.push_back(sct.substr(p, q - p));
        p = q + 1;
      }
    }
    Exec x{e, nullptr, nullptr};
    DevBatchPtr b;
    try {
      b = scan_parquet(x, path, cols);
    } catch (...) {
      cudaStreamSynchronize(e->stream);
      Exec::abandon();
      throw;
    }
    std::lock_guard<std::mutex> g(e->mu);
    e->tables[table][partition] = b;
  });
}

int64_t b200_tpch_table_rows(const char* table, int64_t msf) {
  const int t = table ? table_id(table) : -1;
  return t < 0 ? -1 : tpch::table_rows(t, msf);
}

int b200_engine_export_table(b200_engine* e, const char* table, int partition, struct ArrowArray* out, struct ArrowSchema* out_schema) {
  return guard([&] {
    CUDA_CHECK(cudaSetDevice(e->device));
    DevBatchPtr b;
    {
      std::lock_guard<std::mutex> g(e->mu);
      auto it = e->tables.find(table);
      if (it == e->tables.end() || !it->second.count(partition)) throw EngineError(B200_ERR_NOT_FOUND, "no such table partition");
      b = it->second[partition];
    }
    Exec x{e, nullptr, nullptr};
    export_batch(x, *b, 0, b->n, out, out_schema);
  });
}

int b200_stage_prepare(b200_engine* e, const char* job_id, int64_t stage_id, const char* plan_json, uint64_t plan_len, b200_stage** out) {
  ScopeTimer tm("stage_prepare");
  return guard([&] {
    if (!e || !plan_json || !out) throw EngineError(B200_ERR_INVALID, "null argument");
    const size_t len = plan_len ? (size_t)plan_len : strlen(plan_json);
    // strategy hints (which aggregate sink / table size worked) are remembered per plan SHAPE: the job id is taken out
    // of the hashed text so that the next job that runs the same stage plan starts from what the last one learnt
    std::string shape(plan_json, len);
    const std::string tag = "\"job_id\":\"";
    size_t at = shape.find(tag);
    if (at != std::string::npos) {
      size_t end = shape.find('"', at + tag.size());
      if (end != std::string::npos) shape.erase(at + tag.size(), end - at - tag.size());
    }
    const std::string stage_tag = std::to_string(stage_id) + ":";
    // without a job id from the caller the stage takes the plan's own, so the whole text is the key
    const std::string key = stage_tag + (job_id ? shape : std::string(plan_json, len));
    std::shared_ptr<const PlanNode> plan;
    {
      std::lock_guard<std::mutex> g(e->mu);
      auto it = e->plan_cache.find(key);
      if (it != e->plan_cache.end()) {
        it->second.used = ++e->plan_cache_tick;
        plan = it->second.plan;
      }
    }
    if (!plan) {
      PlanPtr parsed = parse_plan(parse_json(plan_json, len));
      if (parsed->op != PlanNode::ShuffleWriter)
        throw EngineError(B200_ERR_INVALID, "Plan passed to new_query_stage_exec is not a ShuffleWriterExec");  // execution_engine.rs:164-167
      parsed->stage_id = stage_id;
      plan = std::shared_ptr<const PlanNode>(std::move(parsed));
      std::lock_guard<std::mutex> g(e->mu);
      if (e->plan_cache.size() >= PLAN_CACHE_ENTRIES) {
        auto lru = e->plan_cache.begin();
        for (auto it = e->plan_cache.begin(); it != e->plan_cache.end(); ++it)
          if (it->second.used < lru->second.used) lru = it;
        e->plan_cache.erase(lru);
      }
      e->plan_cache[key] = b200_engine::CachedPlan{plan, ++e->plan_cache_tick};
    }
    auto* s = new b200_stage();
    s->eng = e;
    s->job_id = job_id ? job_id : plan->job_id;
    s->stage_id = stage_id;
    s->fingerprint = stage_tag + std::to_string(mix64(hash_bytes((const uint8_t*)shape.data(), (uint32_t)shape.size())));
    collect_nodes(*plan, s);
    s->plan = std::move(plan);
    *out = s;
  });
}

// The task's plan as the scheduler ships it (TaskDefinition.plan: protobuf datafusion.PhysicalPlanNode): decoded to the IR
// by csrc/common/plan_proto.hpp, then prepared like any other stage plan.  Pure host code, no CUDA call.
int b200_plan_proto_to_json(const void* plan_bytes, uint64_t n_bytes, const char* job_id, char** out_json) {
  return guard([&] {
    if (!plan_bytes || !out_json) throw EngineError(B200_ERR_INVALID, "null argument");
    std::string js;
    try {
      js = pbp::plan_proto_to_json(plan_bytes, (size_t)n_bytes, job_id ? std::string(job_id) : std::string());
    } catch (const pbp::Unsupported& u) {
      throw EngineError(B200_ERR_UNSUPPORTED, u.what());
    } catch (const std::runtime_error& r) {
      throw EngineError(B200_ERR_INVALID, r.what());
    }
    char* m = (char*)malloc(js.size() + 1);
    if (!m) throw EngineError(B200_ERR_OOM, "plan JSON");
    memcpy(m, js.c_str(), js.size() + 1);
    *out_json = m;
  });
}

void b200_string_free(char* s) { free(s); }

// EXPLAIN-style diagnostic: the typed plan the engine derived from a stage-plan IR text (column references resolved to
// indices, expression / aggregate result types, every node's output schema), as canonical JSON.  Host only.
int b200_plan_typed_json(const char* plan_json, uint64_t plan_len, char** out_json) {
  return guard([&] {
    if (!plan_json || !out_json) throw EngineError(B200_ERR_INVALID, "null argument");
    Json j = parse_json(plan_json, plan_len ? (size_t)plan_len : strlen(plan_json));
    PlanPtr plan = parse_plan(j);
    const std::string js = dump_plan(*plan);
    char* m = (char*)malloc(js.size() + 1);
    if (!m) throw EngineError(B200_ERR_OOM, "plan JSON");
    memcpy(m, js.c_str(), js.size() + 1);
    *out_json = m;
  });
}

int b200_stage_prepare_proto(b200_engine* e, const char* job_id, int64_t stage_id, const void* plan_bytes, uint64_t n_bytes, b200_stage** out) {
  char* js = nullptr;
  int rc = b200_plan_proto_to_json(plan_bytes, n_bytes, job_id, &js);
  if (rc != 0) return rc;
  rc = b200_stage_prepare(e, job_id, stage_id, js, 0, out);
  free(js);
  return rc;
}

// A whole task as the executor received it (TaskDefinition / MultiTaskDefinition bytes, ballista.proto:518-542): the session
// properties are applied like b200_engine_set_config (TaskDefinition.props -> SessionConfig, executor_server.rs), the embedded
// plan is prepared, and the task identities come back as JSON ({"job_id","stage_id","tasks":[{"task_id","partition_id",..}],..}):
// the caller then runs b200_stage_execute(stage, partition_id) per task.  e == NULL: decode only (*out_stage untouched).
int b200_stage_prepare_task(b200_engine* e, const void* task_bytes, uint64_t n_bytes, int multi, b200_stage** out_stage, char** out_task_json) {
  std::string job;
  int64_t stage_id = 0;
  pbp::Slice plan;
  int rc = guard([&] {
    if (!task_bytes || !out_task_json || (e && !out_stage)) throw EngineError(B200_ERR_INVALID, "null argument");
    pbp::TaskInfo t;
    try {
      t = pbp::decode_task_definition(task_bytes, (size_t)n_bytes, multi != 0);
    } catch (const std::runtime_error& r) {
      throw EngineError(B200_ERR_INVALID, r.what());
    }
    const std::string js = pbp::task_info_json(t);
    char* m = (char*)malloc(js.size() + 1);
    if (!m) throw EngineError(B200_ERR_OOM, "task JSON");
    memcpy(m, js.c_str(), js.size() + 1);
    *out_task_json = m;
    job = t.job_id;
    stage_id = (int64_t)t.stage_id;
    plan = t.plan;
    if (e)
      for (auto& kv : t.props) b200_engine_set_config(e, kv.first.c_str(), kv.second.c_str());
  });
  if (rc != 0 || !e) return rc;
  rc = b200_stage_prepare_proto(e, job.c_str(), stage_id, plan.p, plan.n, out_stage);
  if (rc != 0) {
    free(*out_task_json);
    *out_task_json = nullptr;
  }
  return rc;
}

// TaskStatus (ballista.proto:494-509) for a finished task; rules of executor/src/lib.rs:101-152 and core/src/error.rs:205-256.
int b200_task_status_encode(const char* job_id, const char* executor_id, const b200_task_result* r, const b200_shuffle_write_partition* parts, int n_parts,
                            const b200_operator_metrics* metrics, int n_metrics, char** out_bytes, uint64_t* out_len) {
  return guard([&] {
    if (!job_id || !r || !out_bytes || !out_len || (n_parts > 0 && !parts) || (n_metrics > 0 && !metrics)) throw EngineError(B200_ERR_INVALID, "null argument");
    pbp::Writer w;
    w.u64(1, r->task_id);
    w.str(2, job_id);
    w.u64(3, r->stage_id);
    w.u64(4, r->stage_attempt_num);
    w.u64(5, r->partition_id);
    w.u64(6, r->launch_time);
    w.u64(7, r->start_exec_time);
    w.u64(8, r->end_exec_time);
    if (r->status == B200_OK) {
      pbp::Writer ok;  // SuccessfulTask { executor_id = 1, partitions = 2 } (:453-458)
      ok.str(1, executor_id ? executor_id : "");
      for (int i = 0; i < n_parts; i++) {
        pbp::Writer p;  // ShuffleWritePartition { partition_id = 1, num_batches = 3, num_rows = 4, num_bytes = 5, optional file_id = 6, is_sort_shuffle = 7 } (:481-492)
        p.u64(1, parts[i].partition_id);
        p.u64(3, parts[i].num_batches);
        p.u64(4, parts[i].num_rows);
        p.u64(5, parts[i].num_bytes);
        if (parts[i].file_id >= 0) p.u64_always(6, (uint64_t)parts[i].file_id);
        p.boolean(7, parts[i].is_sort_shuffle != 0);
        ok.msg(2, p);
      }
      w.msg(11, ok);
    } else {
      pbp::Writer f;  // FailedTask { error = 1, retryable = 2, count_to_failures = 3, failed_reason 4..9 } (:437-451)
      const std::string msg = r->error_message ? r->error_message : "";
      if (r->status == B200_ERR_NOT_FOUND) {
        f.str(1, msg);
        pbp::Writer fe;  // FetchPartitionError { executor_id = 1, map_stage_id = 2, map_partition_id = 3 } (:463-467)
        fe.str(1, r->fetch_executor_id ? r->fetch_executor_id : "");
        fe.u64(2, r->fetch_map_stage_id);
        fe.u64(3, r->fetch_map_partition_id);
        f.msg(5, fe);
      } else if (r->status == B200_ERR_CANCELLED) {
        f.str(1, msg.empty() ? std::string("Task killed") : msg);
        f.msg(9, pbp::Writer());  // TaskKilled {}
      } else {
        f.str(1, "Task failed due to runtime execution error: " + msg);
        f.msg(4, pbp::Writer());  // ExecutionError {}
      }
      w.msg(10, f);
    }
    for (int i = 0; i < n_metrics; i++) {
      pbp::Writer set;  // OperatorMetricsSet { metrics = 1 } (:286-288); OperatorMetric oneof (:318-336)
      auto one = [&](uint32_t field, uint64_t v) {
        pbp::Writer m;
        m.u64_always(field, v);
        set.msg(1, m);
      };
      auto named = [&](const char* name, uint64_t v) {
        pbp::Writer nc;  // NamedCount { name = 1, value = 2 } (:291-294)
        nc.str(1, name);
        nc.u64(2, v);
        pbp::Writer m;
        m.msg(6, nc);
        set.msg(1, m);
      };
      one(1, metrics[i].output_rows);
      one(2, metrics[i].elapsed_compute_ns);
      one(12, metrics[i].bytes_written);
      named("input_rows", metrics[i].input_rows);
      named("bytes_read", metrics[i].bytes_read);
      named("kernel_launches", metrics[i].kernel_launches);
      w.msg(12, set);
    }
    char* m = (char*)malloc(w.out.size() + 1);
    if (!m) throw EngineError(B200_ERR_OOM, "task status");
    memcpy(m, w.out.data(), w.out.size());
    m[w.out.size()] = 0;
    *out_bytes = m;
    *out_len = w.out.size();
  });
}

int b200_stage_execute(b200_stage* s, int input_partition, const volatile int32_t* cancel_flag, b200_shuffle_write_partition* out, int cap, int* n_out) {
  ScopeTimer tm("stage_execute");
  return guard([&] {
    if (!s || !n_out) throw EngineError(B200_ERR_INVALID, "null argument");
    CUDA_CHECK(cudaSetDevice(s->eng->device));
    std::vector<b200_shuffle_write_partition> res;
    // a cancelled or failed task leaves nothing behind (Executor::cancel_task drops the future together with
    // its partial outputs, executor.rs:217-237): remove whatever this task already stored
    auto discard = [&]() {
      s->eng->stream_syncs++;
      cudaStreamSynchronize(s->eng->stream);
      Exec::abandon();
      std::lock_guard<std::mutex> g(s->eng->mu);
      for (auto it = s->eng->shuffle.begin(); it != s->eng->shuffle.end();) {
        if (it->first.job == s->job_id && it->first.stage == s->stage_id) {
          auto& v = it->second;
          v.erase(std::remove_if(v.begin(), v.end(), [&](const Piece& pc) { return (pc.file_id == input_partition || (pc.file_id < 0 && it->first.part == input_partition)) && pc.src_rank == s->eng->rank; }), v.end());
          if (v.empty()) {
            it = s->eng->shuffle.erase(it);
            continue;
          }
        }
        ++it;
      }
    };
    const std::vector<OpMetrics> metrics0 = s->metrics;
    try {
      try {
        Runner r{Exec{s->eng, s, cancel_flag, true}, s->job_id};
        res = r.execute_stage(*s->plan, input_partition);
      } catch (const SpeculationMiss&) {
        // an aggregate's groups differed from the last run of its shape: the writers store only after the task's final
        // synchronisation, so nothing of the first run is visible; run the task once more without guessing
        discard();
        s->metrics = metrics0;
        Runner r{Exec{s->eng, s, cancel_flag, false}, s->job_id};
        res = r.execute_stage(*s->plan, input_partition);
      }
    } catch (...) {
      discard();
      throw;
    }
    if ((int)res.size() > cap) throw EngineError(B200_ERR_INVALID, "output array too small");
    for (size_t i = 0; i < res.size(); i++) out[i] = res[i];
    *n_out = (int)res.size();
  });
}

int b200_stage_execute_exchange(b200_stage* s, int input_partition, const volatile int32_t* cancel_flag, b200_shuffle_write_partition* out, int cap,
                                int* n_out, b200_exchange_stats* stats) {
  ScopeTimer tm("stage_execute_exchange");
  return guard([&] {
    if (!s || !n_out) throw EngineError(B200_ERR_INVALID, "null argument");
    b200_engine* e = s->eng;
    if (s->plan->op != PlanNode::ShuffleWriter || s->plan->n_out_partitions < 1)
      throw EngineError(B200_ERR_INVALID, "b200_stage_execute_exchange needs a hash-partitioning ShuffleWriterExec");
    CUDA_CHECK(cudaSetDevice(e->device));
    Exec x{e, s, cancel_flag};
    Runner r{x, s->job_id};
    Runner::FusedExchange fx;
    std::vector<b200_shuffle_write_partition> res;
    uint64_t sent = 0, recvd = 0;
    try {
      res = r.execute_stage(*s->plan, input_partition, &fx);
      if (fx.done) {
        sent = fx.sent;
        recvd = fx.recvd;
      } else if (e->world > 1) {
        // two-step path (strings in the payload, no window, or a window too small for this exchange)
        Exchange ex{x, Runner{x, s->job_id}, e, s->job_id, s->stage_id, (int)s->plan->n_out_partitions, EXCH_HASH, 0, s->plan->schema, s->plan->schema.size()};
        ex.run(&sent, &recvd);
      }
    } catch (...) {
      e->stream_syncs++;
      cudaStreamSynchronize(e->stream);
      Exec::abandon();
      throw;
    }
    e->exch_sent_bytes += sent;
    e->exch_recv_bytes += recvd;
    if (stats) {
      stats->sent_bytes = sent;
      stats->recv_bytes = recvd;
    }
    if ((int)res.size() > cap) throw EngineError(B200_ERR_INVALID, "output array too small");
    for (size_t i = 0; i < res.size(); i++) out[i] = res[i];
    *n_out = (int)res.size();
  });
}

int b200_stage_metrics(b200_stage* s, b200_operator_metrics* out, int cap, int* n_out) {
  return guard([&] {
    int n = (int)std::min<size_t>(s->metrics.size(), (size_t)cap);
    for (int i = 0; i < n; i++) {
      memset(&out[i], 0, sizeof out[i]);
      snprintf(out[i].name, sizeof out[i].name, "%s", s->metrics[(size_t)i].name.c_str());
      out[i].output_rows = s->metrics[(size_t)i].output_rows;
      out[i].input_rows = s->metrics[(size_t)i].input_rows;
      out[i].elapsed_compute_ns = s->metrics[(size_t)i].elapsed_ns;
      out[i].bytes_read = s->metrics[(size_t)i].bytes_read;
      out[i].bytes_written = s->metrics[(size_t)i].bytes_written;
      out[i].kernel_launches = s->metrics[(size_t)i].launches;
    }
    *n_out = n;
  });
}

void b200_stage_release(b200_stage* s) { delete s; }

int b200_partition_export(b200_engine* e, const char* job_id, int64_t stage_id, int out_partition, struct ArrowArray* out, struct ArrowSchema* out_schema) {
  ScopeTimer tm("partition_export");
  return guard([&] {
    CUDA_CHECK(cudaSetDevice(e->device));
    std::vector<std::pair<DevBatchPtr, std::pair<int64_t, int64_t>>> pieces;
    {
      std::lock_guard<std::mutex> g(e->mu);
      auto it = e->shuffle.find(ShuffleKey{job_id, stage_id, out_partition});
      if (it == e->shuffle.end()) throw EngineError(B200_ERR_NOT_FOUND, "no such shuffle partition");  // -> FetchFailed
      for (auto& p : it->second) pieces.push_back({p.batch, {p.r0, p.r1}});
    }
    Exec x{e, nullptr, nullptr};
    if (pieces.size() == 1) {
      export_batch(x, *pieces[0].first, pieces[0].second.first, pieces[0].second.second, out, out_schema);
      return;
    }
    Runner r{x, job_id};
    Schema s;
    for (auto& c : pieces[0].first->cols) s.push_back(Field{c.name, c.type, true});
    DevBatchPtr cat = r.concat_slices(pieces, s);
    export_batch(x, *cat, 0, cat->n, out, out_schema);
  });
}

int64_t b200_partition_rows(b200_engine* e, const char* job_id, int64_t stage_id, int out_partition) {
  std::lock_guard<std::mutex> g(e->mu);
  auto it = e->shuffle.find(ShuffleKey{job_id, stage_id, out_partition});
  if (it == e->shuffle.end()) return -1;
  int64_t n = 0;
  for (auto& p : it->second) n += p.r1 - p.r0;
  return n;
}

int b200_partition_device_buffers(b200_engine* e, const char* job_id, int64_t stage_id, int out_partition, b200_device_buffer* out, int cap, int* n_out,
                                  int64_t* n_rows) {
  return guard([&] {
    CUDA_CHECK(cudaSetDevice(e->device));
    std::vector<std::pair<DevBatchPtr, std::pair<int64_t, int64_t>>> pieces;
    {
      std::lock_guard<std::mutex> g(e->mu);
      auto it = e->shuffle.find(ShuffleKey{job_id, stage_id, out_partition});
      if (it == e->shuffle.end()) throw EngineError(B200_ERR_NOT_FOUND, "no such shuffle partition");
      for (auto& p : it->second) pieces.push_back({p.batch, {p.r0, p.r1}});
    }
    Exec x{e, nullptr, nullptr};
    Runner r{x, job_id};
    Schema s;
    for (auto& c : pieces[0].first->cols) s.push_back(Field{c.name, c.type, true});
    DevBatchPtr cat = r.concat_slices(pieces, s);
    // exchange layout per column: [validity bytes (n) or empty][values | offsets(n+1, rebased)][chars]
    auto packed = std::make_shared<DevBatch>();
    packed->n = cat->n;
    int k = 0;
    // Utf8 columns that are row slices of a larger column: rebase the offsets on the device and learn
    // the chars range of every such column with ONE read-back (not a view round trip per column)
    struct Pending { size_t col; int out_chars; };
    std::vector<Pending> pending;
    DevPtr fl = dev_alloc(8 * (cat->cols.size() + 1), x.st());
    for (auto& c0 : cat->cols) {
      DevColumn c = c0.phys == PH_STRVIEW ? as_utf8(x, c0) : c0;
      if (k + 3 > cap) throw EngineError(B200_ERR_INVALID, "buffer array too small");
      out[k++] = b200_device_buffer{(void*)c.valid, c.valid ? (uint64_t)c.n : 0};
      if (c.phys == PH_UTF8) {
        if (c.n == 0) {
          DevColumn v = as_views(x, c);
          c = as_utf8(x, v);
        } else if (c0.phys != PH_STRVIEW) {  // as_utf8 output already starts at 0 and knows its length
          DevPtr ro = dev_alloc((size_t)(c.n + 1) * 4 + 64, x.st());
          launch_rebase_offsets((const int32_t*)c.data, c.n + 1, (int32_t*)ro->ptr, (int32_t*)fl->ptr + 2 * pending.size(), x.st());
          x.count();
          c.data = (const uint8_t*)ro->ptr;
          c.keep.push_back(ro);
          pending.push_back(Pending{packed->cols.size(), k + 1});
        }
        out[k++] = b200_device_buffer{(void*)c.data, (uint64_t)(c.n + 1) * 4};
        out[k++] = b200_device_buffer{(void*)c.chars, (uint64_t)std::max<int64_t>(c.chars_bytes, 0)};
      } else {
        out[k++] = b200_device_buffer{(void*)c.data, (uint64_t)c.n * c.width()};
        out[k++] = b200_device_buffer{nullptr, 0};
      }
      packed->cols.push_back(c);
    }
    if (!pending.empty()) {
      std::vector<int32_t> h(2 * pending.size());
      CUDA_CHECK(cudaMemcpyAsync(h.data(), fl->ptr, h.size() * 4, cudaMemcpyDeviceToHost, x.st()));
      CUDA_CHECK(cudaStreamSynchronize(x.st()));
      for (size_t i = 0; i < pending.size(); i++) {
        DevColumn& c = packed->cols[pending[i].col];
        c.chars = c.chars + h[2 * i];
        c.chars_bytes = (int64_t)h[2 * i + 1] - (int64_t)h[2 * i];
        out[pending[i].out_chars] = b200_device_buffer{(void*)c.chars, (uint64_t)c.chars_bytes};
      }
    }
    CUDA_CHECK(cudaStreamSynchronize(x.st()));
    // the packed form stays alive next to the partition (until its stage / job data is removed); the stored pieces,
    // their file ids and anything a concurrent map task adds are left alone: this is a read-style call
    {
      std::lock_guard<std::mutex> g(e->mu);
      e->packed_cache[ShuffleKey{job_id, stage_id, out_partition}] = packed;
    }
    *n_out = k;
    *n_rows = packed->n;
  });
}

int b200_partition_import_device(b200_engine* e, const char* job_id, int64_t stage_id, int out_partition, int64_t file_id, const char* schema_json,
                                 const b200_device_buffer* bufs, int n_bufs, int64_t n_rows) {
  return guard([&] {
    CUDA_CHECK(cudaSetDevice(e->device));
    Json j = parse_json(schema_json, strlen(schema_json));
    Schema s = parse_schema(j);
    if ((int)s.size() * 3 != n_bufs) throw EngineError(B200_ERR_INVALID, "expected 3 buffers per column");
    cudaStream_t st = e->stream;
    auto b = std::make_shared<DevBatch>();
    b->n = n_rows;
    for (size_t c = 0; c < s.size(); c++) {
      const b200_device_buffer& bv = bufs[3 * c];
      const b200_device_buffer& bd = bufs[3 * c + 1];
      const b200_device_buffer& bc = bufs[3 * c + 2];
      DevColumn col;
      col.name = s[c].name;
      col.type = s[c].type;
      col.phys = phys_of(col.type);
      col.n = n_rows;
      auto copy_in = [&](const b200_device_buffer& src) -> const uint8_t* {
        DevPtr d = dev_alloc((size_t)src.bytes + 64, st);
        if (src.bytes) CUDA_CHECK(cudaMemcpyAsync(d->ptr, src.ptr, (size_t)src.bytes, cudaMemcpyDeviceToDevice, st));
        col.keep.push_back(d);
        return (const uint8_t*)d->ptr;
      };
      if (bv.bytes) col.valid = copy_in(bv);
      col.nullable = bv.bytes != 0;
      col.data = copy_in(bd);
      if (col.phys == PH_UTF8) {
        col.chars = copy_in(bc);
        col.chars_bytes = (int64_t)bc.bytes;
      }
      b->cols.push_back(col);
    }
    CUDA_CHECK(cudaStreamSynchronize(st));
    std::lock_guard<std::mutex> g(e->mu);
    auto& v = e->shuffle[ShuffleKey{job_id, stage_id, out_partition}];
    v.erase(std::remove_if(v.begin(), v.end(), [&](const Piece& pc) { return pc.file_id == file_id; }), v.end());
    v.push_back(Piece{file_id, b, 0, n_rows});
  });
}

int b200_remove_job_data(b200_engine* e, const char* job_id) {
  return guard([&] {
    CUDA_CHECK(cudaSetDevice(e->device));
    std::lock_guard<std::mutex> g(e->mu);
    for (auto it = e->shuffle.begin(); it != e->shuffle.end();) {
      if (it->first.job == job_id) it = e->shuffle.erase(it);
      else ++it;
    }
    for (auto it = e->packed_cache.begin(); it != e->packed_cache.end();) {
      if (it->first.job == job_id) it = e->packed_cache.erase(it);
      else ++it;
    }
    // partitions that arrived through the fused shuffle live in the exchange window: it is recycled as a whole once no
    // stored partition can refer to it any more (peers write into it only inside a collective this executor takes part in)
    if (e->shuffle.empty()) e->win_used = 0;
  });
}

int b200_device_gather(b200_engine* e, const b200_device_buffer* bufs, int n, void* dst, uint64_t dst_bytes) {
  return guard([&] {
    CUDA_CHECK(cudaSetDevice(e->device));
    uint64_t pos = 0;
    for (int i = 0; i < n; i++) {
      if (!bufs[i].bytes) continue;
      if (pos + bufs[i].bytes > dst_bytes) throw EngineError(B200_ERR_INVALID, "b200_device_gather: destination too small");
      CUDA_CHECK(cudaMemcpyAsync((uint8_t*)dst + pos, bufs[i].ptr, (size_t)bufs[i].bytes, cudaMemcpyDeviceToDevice, e->stream));
      pos += bufs[i].bytes;
    }
  });
}

int b200_remove_stage_data(b200_engine* e, const char* job_id, int64_t stage_id) {
  return guard([&] {
    CUDA_CHECK(cudaSetDevice(e->device));
    std::lock_guard<std::mutex> g(e->mu);
    for (auto it = e->shuffle.begin(); it != e->shuffle.end();) {
      if (it->first.job == job_id && it->first.stage == stage_id) it = e->shuffle.erase(it);
      else ++it;
    }
    for (auto it = e->packed_cache.begin(); it != e->packed_cache.end();) {
      if (it->first.job == job_id && it->first.stage == stage_id) it = e->packed_cache.erase(it);
      else ++it;
    }
  });
}

int b200_engine_kernel_stats(b200_engine* e, b200_kernel_stat* out, int cap, int* n_out, int reset) {
  return guard([&] {
    if (!e || !n_out) throw EngineError(B200_ERR_INVALID, "null argument");
    CUDA_CHECK(cudaSetDevice(e->device));
    CUDA_CHECK(cudaStreamSynchronize(e->stream));
    std::lock_guard<std::mutex> g(e->mu);
    for (auto& ks : e->ksamples) {
      float ms = 0;
      if (cudaEventElapsedTime(&ms, ks.e0, ks.e1) == cudaSuccess) {
        auto& st = e->kstats[ks.name];
        st.ms += ms;
        st.launches++;
        st.bytes += ks.bytes;
      }
      cudaEventDestroy(ks.e0);
      cudaEventDestroy(ks.e1);
    }
    e->ksamples.clear();
    int k = 0;
    for (auto& kv : e->kstats) {
      if (k >= cap) break;
      memset(&out[k], 0, sizeof out[k]);
      snprintf(out[k].name, sizeof out[k].name, "%s", kv.first.c_str());
      out[k].elapsed_ns = (uint64_t)(kv.second.ms * 1e6);
      out[k].launches = kv.second.launches;
      out[k].algorithmic_bytes = kv.second.bytes;
      k++;
    }
    *n_out = k;
    if (reset) e->kstats.clear();
  });
}


int b200_comm_unique_id(void* out, uint64_t cap) {
  return guard([&] {
    if (!out || cap < sizeof(ncclUniqueId)) throw EngineError(B200_ERR_INVALID, "b200_comm_unique_id needs a 128-byte buffer");
    NcclApi& N = NcclApi::get();
    if (!N.ok()) throw EngineError(B200_ERR_CUDA, "libnccl not available: " + N.error);
    ncclUniqueId id;
    NCCL_CHECK(N.GetUniqueId(&id));
    memcpy(out, &id, sizeof id);
  });
}

int b200_engine_comm_init(b200_engine* e, const void* nccl_id, uint64_t id_bytes) {
  return guard([&] {
    if (!e || !nccl_id || id_bytes < sizeof(ncclUniqueId)) throw EngineError(B200_ERR_INVALID, "b200_engine_comm_init: bad arguments");
    if (e->world <= 1) return;  // a single executor exchanges nothing
    NcclApi& N = NcclApi::get();
    if (!N.ok()) throw EngineError(B200_ERR_CUDA, "libnccl not available: " + N.error);
    CUDA_CHECK(cudaSetDevice(e->device));
    std::lock_guard<std::mutex> g(e->comm_mu);
    if (e->comm) {
      N.CommDestroy(e->comm);
      e->comm = nullptr;
    }
    ncclUniqueId id;
    memcpy(&id, nccl_id, sizeof id);
    NCCL_CHECK(N.CommInitRank(&e->comm, e->world, id, e->rank));
    release_window(e);
    if (e->win_config_bytes) setup_window(e);
  });
}

int b200_exchange_stage(b200_engine* e, const char* job_id, int64_t stage_id, int n_out_partitions, int mode, int root, const char* schema_json,
                        b200_exchange_stats* stats) {
  return guard([&] {
    if (!e || !job_id || !schema_json) throw EngineError(B200_ERR_INVALID, "null argument");
    if (mode < 0 || mode > 2 || n_out_partitions < 0 || root < 0 || root >= std::max(e->world, 1)) throw EngineError(B200_ERR_INVALID, "b200_exchange_stage: bad mode / root");
    CUDA_CHECK(cudaSetDevice(e->device));
    Json j = parse_json(schema_json, strlen(schema_json));
    Exec x{e, nullptr, nullptr};
    Exchange ex{x, Runner{x, job_id}, e, job_id, stage_id, n_out_partitions, mode, root, parse_schema(j), 0};
    ex.ncols = ex.schema.size();
    uint64_t sent = 0, recvd = 0;
    try {
      ex.run(&sent, &recvd);
    } catch (...) {
      cudaStreamSynchronize(e->stream);
      Exec::abandon();
      throw;
    }
    e->exch_sent_bytes += sent;
    e->exch_recv_bytes += recvd;
    if (stats) {
      stats->sent_bytes = sent;
      stats->recv_bytes = recvd;
    }
  });
}

// ---- the reference's shuffle file format: Arrow IPC streams with LZ4_FRAME bodies (csrc/host/arrow_ipc.hpp) ----------------
static std::vector<HostCol> host_cols_from_arrow(ArrowArray* arr, ArrowSchema* sch, int64_t* n_rows) {
  std::vector<ImportedCol> ics = import_record_batch(arr, sch, n_rows);
  const int64_t n = *n_rows;
  std::vector<HostCol> out;
  for (auto& ic : ics) {
    HostCol h;
    h.name = ic.name;
    h.type = ic.type;
    h.nullable = ic.nullable;
    h.n = n;
    if (ic.large_offsets) throw EngineError(B200_ERR_UNSUPPORTED, "LargeUtf8 columns are not supported");
    auto bit = [](const uint8_t* bm, int64_t i) { return (bm[i >> 3] >> (i & 7)) & 1; };
    if (ic.null_count > 0 && ic.validity) {
      h.validity.assign((size_t)((n + 7) / 8), 0);
      for (int64_t i = 0; i < n; i++)
        if (bit(ic.validity, i + ic.offset)) h.validity[(size_t)(i >> 3)] |= (uint8_t)(1u << (i & 7));
        else h.null_count++;
      if (h.null_count == 0) h.validity.clear();
    }
    if (ic.type.id == TypeId::Null) {
      h.null_count = n;
    } else if (ic.type.id == TypeId::Bool) {
      h.data.assign((size_t)((n + 7) / 8), 0);
      for (int64_t i = 0; i < n; i++)
        if (bit(ic.data, i + ic.offset)) h.data[(size_t)(i >> 3)] |= (uint8_t)(1u << (i & 7));
    } else if (ic.type.id == TypeId::Utf8) {
      const int32_t* off = (const int32_t*)ic.data + ic.offset;
      h.data.resize((size_t)(n + 1) * 4);
      int32_t* po = (int32_t*)h.data.data();
      for (int64_t i = 0; i <= n; i++) po[i] = off[i] - off[0];
      if (n) h.extra.assign(ic.extra + off[0], ic.extra + off[n]);
    } else {
      const size_t w = (size_t)ic.type.width();
      h.data.assign(ic.data + (size_t)ic.offset * w, ic.data + (size_t)(ic.offset + n) * w);
    }
    out.push_back(std::move(h));
  }
  return out;
}

static std::vector<uint8_t> read_whole_file(const std::string& path, uint64_t offset, uint64_t length) {
  FILE* f = fopen(path.c_str(), "rb");
  if (!f) throw EngineError(B200_ERR_NOT_FOUND, "cannot open " + path);  // -> FetchFailed
  fseek(f, 0, SEEK_END);
  const uint64_t fsize = (uint64_t)ftell(f);
  if (length == 0 && offset == 0) length = fsize;
  if (offset + length > fsize) {
    fclose(f);
    throw EngineError(B200_ERR_INVALID, "byte range outside " + path);
  }
  fseek(f, (long)offset, SEEK_SET);
  std::vector<uint8_t> buf((size_t)length);
  const size_t got = length ? fread(buf.data(), 1, (size_t)length, f) : 0;
  fclose(f);
  if (got != length) throw EngineError(B200_ERR_INVALID, "short read on " + path);
  return buf;
}

static void write_whole_file(const std::string& path, const std::vector<uint8_t>& bytes) {
  FILE* f = fopen(path.c_str(), "wb");
  if (!f) throw EngineError(B200_ERR_INVALID, "cannot create " + path);
  const size_t put = bytes.empty() ? 0 : fwrite(bytes.data(), 1, bytes.size(), f);
  fclose(f);
  if (put != bytes.size()) throw EngineError(B200_ERR_INVALID, "short write on " + path);
}

static void make_dirs(const std::string& path) {
  std::string cur;
  for (size_t i = 0; i <= path.size(); i++) {
    if (i == path.size() || path[i] == '/') {
      if (!cur.empty() && cur != "/") mkdir(cur.c_str(), 0777);
    }
    if (i < path.size()) cur.push_back(path[i]);
  }
}

int b200_ipc_encode(struct ArrowArray* batch, struct ArrowSchema* schema, int compress, int64_t max_rows_per_message, uint8_t** out, uint64_t* out_len) {
  return guard([&] {
    if (!batch || !schema || !out || !out_len) throw EngineError(B200_ERR_INVALID, "null argument");
    int64_t n = 0;
    std::vector<HostCol> cols;
    try {
      cols = host_cols_from_arrow(batch, schema, &n);
    } catch (const std::runtime_error& ex) {
      throw EngineError(B200_ERR_INVALID, ex.what());
    }
    if (batch->release) batch->release(batch);
    if (schema->release) schema->release(schema);
    std::vector<uint8_t> bytes;
    ipc::write_stream(bytes, cols, n, compress != 0, max_rows_per_message);
    uint8_t* p = (uint8_t*)malloc(bytes.size() ? bytes.size() : 1);
    if (!p) throw EngineError(B200_ERR_OOM, "host out of memory");
    memcpy(p, bytes.data(), bytes.size());
    *out = p;
    *out_len = bytes.size();
  });
}

void b200_ipc_free(uint8_t* p) { free(p); }

int b200_ipc_decode(const uint8_t* buf, uint64_t len, struct ArrowArray* out, struct ArrowSchema* out_schema) {
  return guard([&] {
    if (!buf || !out || !out_schema) throw EngineError(B200_ERR_INVALID, "null argument");
    std::vector<HostCol> cols;
    int64_t n = 0;
    try {
      n = ipc::read_streams(buf, (size_t)len, cols);
    } catch (const std::runtime_error& ex) {
      throw EngineError(B200_ERR_INVALID, ex.what());
    }
    export_record_batch(std::move(cols), n, out, out_schema);
  });
}

// Every piece this executor's map tasks produced for (job, stage), as files in the reference's layout below work_dir
// (create_shuffle_path, execution_plans/mod.rs:66-99): what makes HBM-resident shuffle output survive the executor and
// readable by the reference's own readers (a CPU executor's ShuffleReaderExec, the Flight service).
int b200_shuffle_write_files(b200_engine* e, const char* job_id, int64_t stage_id, const char* work_dir, int n_out_partitions, int sort_layout,
                             uint64_t* files_written, uint64_t* bytes_written) {
  return guard([&] {
    if (!e || !job_id || !work_dir) throw EngineError(B200_ERR_INVALID, "null argument");
    CUDA_CHECK(cudaSetDevice(e->device));
    Exec x{e, nullptr, nullptr};
    struct Item { int64_t part; Piece piece; };
    std::vector<Item> items;
    {
      std::lock_guard<std::mutex> g(e->mu);
      for (auto& kv : e->shuffle)
        if (kv.first.job == job_id && kv.first.stage == stage_id)
          for (auto& pc : kv.second)
            if (pc.src_rank == e->rank) items.push_back(Item{kv.first.part, pc});
    }
    const std::string base = std::string(work_dir) + "/" + job_id + "/" + std::to_string(stage_id);
    uint64_t nfiles = 0, nbytes = 0;
    const int64_t bs = e->batch_size;
    if (!sort_layout) {
      for (auto& it : items) {
        std::vector<HostCol> cols = download_batch(x, *it.piece.batch, it.piece.r0, it.piece.r1);
        std::vector<uint8_t> bytes;
        ipc::write_stream(bytes, cols, it.piece.r1 - it.piece.r0, true, bs);
        const std::string dir = base + "/" + std::to_string(it.part);
        make_dirs(dir);
        const std::string path = dir + (it.piece.file_id >= 0 ? "/data-" + std::to_string(it.piece.file_id) + ".arrow" : "/data.arrow");
        write_whole_file(path, bytes);
        nfiles++;
        nbytes += bytes.size();
      }
    } else {
      // one consolidated file per map task: [schema-only stream][partition 0 streams][partition 1 streams]... + index
      std::map<int64_t, std::vector<Item*>> by_task;
      for (auto& it : items) by_task[it.piece.file_id].push_back(&it);
      for (auto& kv : by_task) {
        if (kv.first < 0) throw EngineError(B200_ERR_INVALID, "sort-shuffle layout needs a file id (un-partitioned stage output)");
        std::vector<uint8_t> bytes;
        std::vector<int64_t> offsets((size_t)n_out_partitions + 1, 0);
        bool header = false;
        std::vector<std::vector<HostCol>> parts((size_t)n_out_partitions);
        std::vector<int64_t> rows((size_t)n_out_partitions, 0);
        for (Item* it : kv.second) {
          if (it->part >= n_out_partitions) throw EngineError(B200_ERR_INVALID, "stored partition id beyond n_out_partitions");
          parts[(size_t)it->part] = download_batch(x, *it->piece.batch, it->piece.r0, it->piece.r1);
          rows[(size_t)it->part] = it->piece.r1 - it->piece.r0;
          if (!header) {
            ipc::write_schema(bytes, parts[(size_t)it->part]);
            ipc::write_eos(bytes);
            header = true;
          }
        }
        for (int p = 0; p < n_out_partitions; p++) {
          offsets[(size_t)p] = (int64_t)bytes.size();
          if (rows[(size_t)p] > 0) ipc::write_stream(bytes, parts[(size_t)p], rows[(size_t)p], true, bs);
        }
        offsets[(size_t)n_out_partitions] = (int64_t)bytes.size();
        const std::string dir = base + "/" + std::to_string(kv.first);
        make_dirs(dir);
        write_whole_file(dir + "/data.arrow", bytes);
        std::vector<uint8_t> idx((size_t)(n_out_partitions + 1) * 8);
        memcpy(idx.data(), offsets.data(), idx.size());
        write_whole_file(dir + "/data.arrow.index", idx);
        nfiles += 2;
        nbytes += bytes.size() + idx.size();
      }
    }
    if (files_written) *files_written = nfiles;
    if (bytes_written) *bytes_written = nbytes;
  });
}

// One reference-format shuffle file (or a byte range of it: a partition of a sort-shuffle data file) into the shuffle
// store as a piece of (job, stage, out_partition) -- the local-read path of ShuffleReaderExec (shuffle_reader.rs:698-771,
// sort_shuffle/reader.rs:51-84) with the decoded batches landing in HBM.  byte_length 0 with byte_offset 0 = whole file;
// use_index != 0: `path` is a sort-shuffle data file, the range of `out_partition` is taken from `path` + ".index".
int b200_shuffle_read_file(b200_engine* e, const char* job_id, int64_t stage_id, int out_partition, int64_t file_id, const char* path, uint64_t byte_offset,
                           uint64_t byte_length, int use_index) {
  return guard([&] {
    if (!e || !job_id || !path) throw EngineError(B200_ERR_INVALID, "null argument");
    CUDA_CHECK(cudaSetDevice(e->device));
    std::vector<HostCol> cols;
    int64_t n = 0;
    try {
      if (use_index) {
        std::vector<uint8_t> idx = read_whole_file(std::string(path) + ".index", 0, 0);
        if (idx.size() % 8 || idx.size() < 16) throw EngineError(B200_ERR_INVALID, "invalid shuffle index file");
        const size_t entries = idx.size() / 8;
        if ((size_t)out_partition + 1 >= entries) throw EngineError(B200_ERR_NOT_FOUND, "partition not found in the shuffle index");
        int64_t o0, o1, first;
        memcpy(&first, idx.data(), 8);
        memcpy(&o0, idx.data() + 8 * (size_t)out_partition, 8);
        memcpy(&o1, idx.data() + 8 * (size_t)out_partition + 8, 8);
        if (o0 < 0 || o1 < o0 || first < 0) throw EngineError(B200_ERR_INVALID, "invalid partition byte range in the shuffle index");
        // the leading schema-only stream, then the partition's own streams
        if (first > 0) {
          std::vector<uint8_t> head = read_whole_file(path, 0, (uint64_t)first);
          ipc::read_streams(head.data(), head.size(), cols);
        }
        if (o1 > o0) {
          std::vector<uint8_t> body = read_whole_file(path, (uint64_t)o0, (uint64_t)(o1 - o0));
          n = ipc::read_streams(body.data(), body.size(), cols);
        }
      } else {
        std::vector<uint8_t> body = read_whole_file(path, byte_offset, byte_length);
        n = ipc::read_streams(body.data(), body.size(), cols);
      }
    } catch (const std::runtime_error& ex) {
      throw EngineError(B200_ERR_INVALID, ex.what());
    }
    // host columns -> Arrow C structs -> the ordinary ingest path
    ArrowArray arr;
    ArrowSchema sch;
    export_record_batch(std::move(cols), n, &arr, &sch);
    DevBatchPtr b = import_batch(e, &arr, &sch);
    std::vector<int64_t> sb;
    for (auto& c : b->cols)
      if (c.type.id == TypeId::Utf8) sb.push_back(c.chars_bytes);
    std::lock_guard<std::mutex> g(e->mu);
    auto& v = e->shuffle[ShuffleKey{job_id, stage_id, out_partition}];
    v.erase(std::remove_if(v.begin(), v.end(), [&](const Piece& pc) { return pc.file_id == file_id && pc.src_rank == -1; }), v.end());
    Piece pc;
    pc.file_id = file_id;
    pc.batch = b;
    pc.r0 = 0;
    pc.r1 = n;
    pc.src_rank = -1;  // came from a file, not from one of the box's GPU executors
    pc.str_bytes = sb;
    v.push_back(pc);
  });
}

void* b200_host_alloc_pinned(uint64_t bytes) {
  void* p = nullptr;
  if (cudaHostAlloc(&p, (size_t)bytes, cudaHostAllocDefault) != cudaSuccess) return nullptr;
  return p;
}
void b200_host_free_pinned(void* p) {
  if (p) cudaFreeHost(p);
}

}  // extern "C"
