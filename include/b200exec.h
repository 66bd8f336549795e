/* libb200exec -- C ABI of the B200-native Ballista execution engine.
 *
 * The reference defines NO C ABI: its plug-in point is the Rust trait pair
 *   ExecutionEngine::create_query_stage_exec   ballista/executor/src/execution_engine.rs:45-59
 *   QueryStageExecutor::execute_query_stage /
 *   QueryStageExecutor::collect_plan_metrics   ballista/executor/src/execution_engine.rs:67-81
 * installed through ExecutorProcessConfig.override_execution_engine
 *   (ballista/executor/src/executor_process.rs:158-160, consumed :341-351).
 * Every entry point below names the reference interface it stands behind; INTEGRATION.md shows the
 * Rust shim (`GpuExecutionEngine: ExecutionEngine`) that binds them with `extern "C"`.
 *
 * Conventions: opaque handles; every call returns 0 on success or a negative b200_status and
 * records a message retrievable with b200_last_error() (thread-local); no exceptions, no
 * callbacks, nothing unwinds across the boundary (reference rule: "the engine must never
 * panic/abort", SURVEY.md 8(b) "Error convention").  Column data crosses as Arrow C Data
 * Interface structs (include/b200_arrow_abi.h); the consumer releases what it receives.
 */
#ifndef B200EXEC_H
#define B200EXEC_H
#include <stdint.h>

#include "b200_arrow_abi.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef enum b200_status {
  B200_OK = 0,
  B200_ERR_INVALID = -1,       /* bad argument / malformed plan  -> DataFusionError::Plan           */
  B200_ERR_UNSUPPORTED = -2,   /* operator/expr not lowered yet  -> DataFusionError::NotImplemented */
  B200_ERR_EXECUTION = -3,     /* arithmetic overflow, div by 0  -> DataFusionError::Execution      */
  B200_ERR_CUDA = -4,          /* CUDA runtime failure           -> DataFusionError::External       */
  B200_ERR_NOT_FOUND = -5,     /* missing shuffle partition      -> BallistaError::FetchFailed      */
  B200_ERR_CANCELLED = -6,     /* cancel flag observed           -> task aborted (executor.rs:217)  */
  B200_ERR_OOM = -7            /* device pool exhausted          -> DataFusionError::ResourcesExhausted */
} b200_status;

typedef struct b200_engine b200_engine;  /* one per executor process == one per GPU */
typedef struct b200_stage b200_stage;    /* one per task: Arc<dyn QueryStageExecutor> */

/* Mirror of message ShuffleWritePartition, ballista/core/proto/ballista.proto:481-492.
 * file_id < 0 encodes `None` (un-partitioned writer branch, shuffle_writer.rs:260-267). */
typedef struct b200_shuffle_write_partition {
  uint64_t partition_id;
  uint64_t num_batches;
  uint64_t num_rows;
  uint64_t num_bytes;
  int64_t file_id;
  int32_t is_sort_shuffle;
  int32_t _pad;
} b200_shuffle_write_partition;

/* One entry per operator of the stage plan (pre-order), the payload of
 * QueryStageExecutor::collect_plan_metrics (execution_engine.rs:80; utils.rs:328-339). */
typedef struct b200_operator_metrics {
  char name[48];
  uint64_t output_rows;
  uint64_t input_rows;
  uint64_t elapsed_compute_ns; /* device time, CUDA events */
  uint64_t bytes_read;         /* algorithmic bytes (SURVEY.md 8(d)) */
  uint64_t bytes_written;
  uint64_t kernel_launches;
} b200_operator_metrics;

/* ---- engine lifecycle (Executor::new, ballista/executor/src/executor.rs:67-95) ------------- */
/* device: CUDA ordinal; pool_bytes: device pool release threshold (0 = keep everything);
 * rank/world: position of this executor among the box's GPU executors (exchange step). */
int b200_engine_create(int device, uint64_t pool_bytes, int rank, int world, b200_engine** out);
void b200_engine_destroy(b200_engine* e);
const char* b200_last_error(void);
/* Launch all kernels of this engine on `cuda_stream` (a cudaStream_t); NULL = engine-owned stream. */
int b200_engine_set_stream(b200_engine* e, void* cuda_stream);
int b200_engine_synchronize(b200_engine* e);
/* Number of kernels this engine has launched since creation (bench.py "gpu_launches"). */
uint64_t b200_engine_kernel_launches(b200_engine* e);
/* Introspection for tests and bench.py: how many pipelines ran on which kernel family so far.
 * name: "fused" (fused.cuh kernel, any variant), "fused_static" (an ahead-of-time shape),
 * "vm" (tile VM pipeline_kernel); "ingest_bytes_saved": host->device bytes NOT sent because
 * Decimal128 values were narrowed on the host and widened on the device; "stream_syncs": host waits on the
 * engine's stream inside stage tasks and partition exports.  Unknown names return 0. */
uint64_t b200_engine_counter(b200_engine* e, const char* name);
/* Per-kernel-family device time (CUDA events on the launching stream) and algorithmic bytes, accumulated since the
 * last reset while the config key "b200.metrics.kernel_timing" is "on" (radix partition, join build / probe,
 * group-by, sort passes, ...): the measurement behind the per-operator roofline figures. */
typedef struct b200_kernel_stat {
  char name[48];
  uint64_t elapsed_ns;
  uint64_t launches;
  uint64_t algorithmic_bytes;
} b200_kernel_stat;
int b200_engine_kernel_stats(b200_engine* e, b200_kernel_stat* out, int cap, int* n_out, int reset);
/* session config (TaskDefinition.props; SURVEY.md Appendix C), e.g. "datafusion.execution.batch_size" */
int b200_engine_set_config(b200_engine* e, const char* key, const char* value);

/* ---- leaf inputs ---------------------------------------------------------------------------- */
/* DataSourceExec leaf: host RecordBatch (struct array) for `table`, input partition `partition`.
 * Copies host->device on the engine stream (pinned staging); appends if called repeatedly.
 * The engine releases `batch` / `schema` when the copy has been issued. */
int b200_engine_register_batch(b200_engine* e, const char* table, int partition,
                               struct ArrowArray* batch, struct ArrowSchema* schema);
/* DataSourceExec + ParquetSource leaf (datafusion.proto:1058-1077; tpch.rs:684-693 registers TPC-H tables this way): the
 * file's requested column chunks cross the bus ENCODED and are decoded on the device (PLAIN / RLE_DICTIONARY pages V1+V2,
 * definition levels, INT32 / INT64 / DOUBLE / BOOLEAN / BYTE_ARRAY / FIXED_LEN_BYTE_ARRAY with DECIMAL / DATE / STRING
 * annotations, flat schemas, UNCOMPRESSED codec).  columns_csv = NULL: every column.  Replaces the table partition. */
int b200_engine_register_parquet(b200_engine* e, const char* table, int partition, const char* path, const char* columns_csv);
/* Host-only: JSON description (schema, rows, page inventory per column) of a Parquet file as the scan's metadata reader
 * sees it.  No CUDA call. */
int b200_parquet_describe(const char* path, char* out, uint64_t cap);
int b200_engine_drop_table(b200_engine* e, const char* table);
/* Synthetic TPC-H-shaped table generated directly in HBM (bench/test input; columns = NULL: all).
 * Rows [row_begin,row_end) of the table at milli-scale-factor `msf` become partition `partition`. */
int b200_engine_tpch_generate(b200_engine* e, const char* table, int64_t msf, int partition,
                              int64_t row_begin, int64_t row_end, const char* columns_csv);
/* Rows of a synthetic TPC-H table at milli-scale-factor `msf` (-1: unknown table). */
int64_t b200_tpch_table_rows(const char* table, int64_t msf);
/* Read a registered table partition back to the host (test/diagnostic). */
int b200_engine_export_table(b200_engine* e, const char* table, int partition,
                             struct ArrowArray* out, struct ArrowSchema* out_schema);

/* ---- ExecutionEngine::create_query_stage_exec (execution_engine.rs:50-58) ------------------ */
/* plan_json: stage plan IR rooted at ShuffleWriterExec / SortShuffleWriterExec (JSON rendering of
 * the DataFusion physical plan; schema in DESIGN.md).  Errors if the root is not a shuffle
 * writer, like DefaultExecutionEngine (execution_engine.rs:164-167). */
int b200_stage_prepare(b200_engine* e, const char* job_id, int64_t stage_id, const char* plan_json,
                       uint64_t plan_len, b200_stage** out);
/* The same from the bytes the scheduler ships: `TaskDefinition.plan` / `MultiTaskDefinition.plan`
 * (ballista/core/proto/ballista.proto:518-529,551-560) = a protobuf datafusion.PhysicalPlanNode
 * (ballista/core/proto/datafusion.proto:716-757) whose shuffle writer / reader nodes travel as PhysicalExtensionNode
 * (BallistaPhysicalExtensionCodec, ballista/core/src/serde/mod.rs:322-640).  The executor can pass `task.plan` through as it
 * arrived (execution_engine.rs:106-169 decodes the same bytes into an ExecutionPlan first).  Nodes, expressions or types the
 * device engine does not implement return B200_ERR_UNSUPPORTED with the offending variant named, malformed bytes
 * B200_ERR_INVALID.  `job_id` (may be NULL) replaces the job id stored inside the shuffle writer node.
 * b200_plan_proto_to_json is the decoder alone (host only, no GPU needed): *out_json is a NUL-terminated malloc'd string,
 * release it with b200_string_free. */
int b200_stage_prepare_proto(b200_engine* e, const char* job_id, int64_t stage_id, const void* plan_bytes,
                             uint64_t n_bytes, b200_stage** out);
/* ... and the way back: the `TaskStatus` message (ballista.proto:494-509) an executor reports for a finished task, built the
 * way ballista/executor/src/lib.rs:101-152 (`as_task_status`) and ballista/core/src/error.rs:205-256 (`FailedTask::from`)
 * build it.  status == B200_OK: `successful { executor_id, partitions }` from b200_stage_execute's output.  B200_ERR_NOT_FOUND:
 * `failed { error, retryable = false, count_to_failures = false, fetch_partition_error { fetch_* } }` (the scheduler re-runs the
 * map stage).  B200_ERR_CANCELLED: `failed { task_killed }`.  Anything else: `failed { error = "Task failed due to runtime
 * execution error: <message>", execution_error }`.  `metrics`: one OperatorMetricsSet per operator (b200_stage_metrics order)
 * with output_rows, elapse_time (device ns), output_bytes and the named counts input_rows / bytes_read / kernel_launches.
 * *out_bytes is malloc'd (b200_string_free releases it).  Host only. */
typedef struct b200_task_result {
  uint32_t task_id, stage_id, stage_attempt_num, partition_id;
  uint64_t launch_time, start_exec_time, end_exec_time; /* ms since the epoch, as TaskExecutionTimes */
  int32_t status;                                        /* what b200_stage_execute returned */
  uint32_t fetch_map_stage_id, fetch_map_partition_id;   /* B200_ERR_NOT_FOUND only */
  const char* fetch_executor_id;                         /* B200_ERR_NOT_FOUND only (may be NULL) */
  const char* error_message;                             /* failed tasks: b200_last_error() (may be NULL) */
} b200_task_result;
int b200_task_status_encode(const char* job_id, const char* executor_id, const b200_task_result* r,
                            const b200_shuffle_write_partition* parts, int n_parts, const b200_operator_metrics* metrics,
                            int n_metrics, char** out_bytes, uint64_t* out_len);
int b200_plan_proto_to_json(const void* plan_bytes, uint64_t n_bytes, const char* job_id, char** out_json);
/* A whole task as the executor received it: `TaskDefinition` (multi == 0; LaunchTask / PollWorkResult.tasks) or
 * `MultiTaskDefinition` (multi != 0; LaunchMultiTask) bytes, ballista.proto:518-542.  Applies `props` as
 * b200_engine_set_config does (TaskDefinition.props is how session settings reach an executor), prepares the embedded plan
 * (as b200_stage_prepare_proto, job and stage id taken from the task) and returns the task identities as JSON in
 * *out_task_json (release with b200_string_free): {"job_id","stage_id","stage_attempt_num","session_id","launch_time",
 * "tasks":[{"task_id","task_attempt_num","partition_id"}],"props":{...}} -- run b200_stage_execute(stage, partition_id) per
 * task.  With e == NULL only the decoding happens (host only). */
int b200_stage_prepare_task(b200_engine* e, const void* task_bytes, uint64_t n_bytes, int multi, b200_stage** out_stage,
                            char** out_task_json);
void b200_string_free(char* s);
/* EXPLAIN-style diagnostic (host only): the typed plan derived from a stage-plan IR text -- column references resolved to
 * indices, expression and aggregate types, every node's output schema (what ExecutionPlan::schema() reports per node) -- as
 * canonical JSON; two IR texts describe the same plan exactly when these texts are equal. */
int b200_plan_typed_json(const char* plan_json, uint64_t plan_len, char** out_json);
/* ---- QueryStageExecutor::execute_query_stage (execution_engine.rs:73-77) ------------------- */
/* Runs input partition `input_partition`; writes up to `cap` entries to `out`, count to *n_out.
 * `cancel_flag` (may be NULL) is polled between kernels: non-zero => B200_ERR_CANCELLED and all
 * partial outputs of this task are dropped (Executor::cancel_task, executor.rs:217-237). */
int b200_stage_execute(b200_stage* s, int input_partition, const volatile int32_t* cancel_flag,
                       b200_shuffle_write_partition* out, int cap, int* n_out);
/* ---- QueryStageExecutor::collect_plan_metrics (execution_engine.rs:80) ---------------------- */
int b200_stage_metrics(b200_stage* s, b200_operator_metrics* out, int cap, int* n_out);
void b200_stage_release(b200_stage* s);

/* ---- shuffle partitions (ShuffleReaderExec / Flight service side) --------------------------- */
/* Identity of stored bytes == (job_id, stage_id, out_partition, file_id, is_sort_shuffle), the
 * tuple create_shuffle_path resolves (ballista/core/src/execution_plans/mod.rs:66-99). */
/* Host-visible export of ONE output partition (all map tasks' pieces concatenated): what
 * BallistaFlightService::do_get / fetch_partition_local serve (flight_service.rs:88-184,
 * shuffle_reader.rs:698-771). */
int b200_partition_export(b200_engine* e, const char* job_id, int64_t stage_id, int out_partition,
                          struct ArrowArray* out, struct ArrowSchema* out_schema);
/* Rows currently stored for (job, stage, out_partition); -1 if absent. */
int64_t b200_partition_rows(b200_engine* e, const char* job_id, int64_t stage_id, int out_partition);
/* Device-resident exchange descriptor for peer pulls / NCCL all-to-all: fills device pointers and
 * byte sizes of the partition's column buffers (see DESIGN.md "Exchange"). */
typedef struct b200_device_buffer {
  void* ptr;
  uint64_t bytes;
} b200_device_buffer;
int b200_partition_device_buffers(b200_engine* e, const char* job_id, int64_t stage_id, int out_partition,
                                  b200_device_buffer* out, int cap, int* n_out, int64_t* n_rows);
/* Install a partition received from a peer GPU (buffers already in this GPU's HBM, laid out as
 * b200_partition_device_buffers describes; the engine takes ownership via copy on its stream). */
int b200_partition_import_device(b200_engine* e, const char* job_id, int64_t stage_id, int out_partition,
                                 int64_t file_id, const char* schema_json, const b200_device_buffer* bufs,
                                 int n_bufs, int64_t n_rows);
/* Pack `n` device buffers back to back into `dst` (device memory of this GPU, >= the sum of their
 * sizes) on the engine's stream: the send side of the exchange builds one contiguous message per
 * peer this way (the reference's counterpart is the IPC writer appending batches to one shuffle file,
 * ballista/core/src/execution_plans/shuffle_writer.rs:262-330).  Returns after the copies are
 * enqueued; call b200_engine_synchronize (or use the same stream) before reading `dst`. */
int b200_device_gather(b200_engine* e, const b200_device_buffer* bufs, int n, void* dst, uint64_t dst_bytes);
/* RemoveJobData RPC (ballista/executor/src/executor_server.rs:921-932). */
int b200_remove_job_data(b200_engine* e, const char* job_id);
/* Drop every stored partition of one stage (used by the exchange step once the pieces have been
 * handed to their owning GPUs; the reference deletes map outputs the same way on stage rollback). */
int b200_remove_stage_data(b200_engine* e, const char* job_id, int64_t stage_id);

/* ---- exchange between the box's GPU executors ------------------------------------------------
 * Stands behind ShuffleReaderExec's remote fetch (shuffle_reader.rs:522-602 -> BallistaClient::fetch_partition,
 * client.rs:143-220 -> BallistaFlightService::do_get / do_action, flight_service.rs:88-306): with one executor per GPU
 * of one box the same bytes move as an all-to-all-v over NVLink (grouped ncclSend / ncclRecv issued by this
 * library on the engine's stream).  NCCL is bound with dlopen; an engine with world == 1 never loads it.
 *   b200_comm_unique_id: 128 bytes (ncclUniqueId) generated by ONE executor; the host side distributes them to the
 *     others (in Ballista: a task property set by the scheduler; in the harness: any broadcast).
 *   b200_engine_comm_init: collective over the `world` engines created with ranks 0..world-1.
 *   b200_exchange_stage: collective, after every executor finished its map tasks of (job, stage).  Afterwards each
 *     output partition's pieces live in the HBM of the executor(s) that will run its reduce task:
 *       B200_EXCHANGE_HASH       partition p -> executor p % world        (hash repartition, planner.rs:194-256)
 *       B200_EXCHANGE_GATHER     every partition -> executor `root`       (CoalescePartitions / SortPreservingMerge)
 *       B200_EXCHANGE_BROADCAST  every partition -> every executor        (broadcast join build side,
 *                                                                          planner.rs:142-183, shuffle_reader.rs:121-144)
 *     schema_json: the stage's output schema (same JSON as b200_partition_import_device). */
#define B200_NCCL_ID_BYTES 128
enum { B200_EXCHANGE_HASH = 0, B200_EXCHANGE_GATHER = 1, B200_EXCHANGE_BROADCAST = 2 };
typedef struct b200_exchange_stats {
  uint64_t sent_bytes;   /* payload bytes this executor sent to peers */
  uint64_t recv_bytes;   /* payload bytes it received */
} b200_exchange_stats;
int b200_comm_unique_id(void* out, uint64_t cap);
int b200_engine_comm_init(b200_engine* e, const void* nccl_id, uint64_t id_bytes);
int b200_exchange_stage(b200_engine* e, const char* job_id, int64_t stage_id, int n_out_partitions, int mode, int root,
                        const char* schema_json, b200_exchange_stats* stats);
/* Fused shuffle writer + exchange: b200_stage_execute and the B200_EXCHANGE_HASH exchange of its output as ONE collective
 * (ShuffleWriterExec::execute_shuffle_write, shuffle_writer.rs:214-330, together with the readers' fetch,
 * shuffle_reader.rs:522-602).  Every executor of the communicator calls it for its map task of the same stage (executors
 * that run several map tasks of the stage call it once per task, all in the same order).  When the engines were given an
 * exchange window (configuration key "b200.exchange.window_bytes" set before b200_engine_comm_init: that many bytes of HBM
 * per executor, published to the peers through CUDA IPC) and the stage's output holds no string column, the partition
 * scatter kernel stores every row directly at its final place in the HBM of the executor that owns its output partition
 * (partition p -> executor p % world; peer stores over NVLink), after one small all-gather of the per-partition row
 * counts; nothing is staged and no separate transfer follows.  Otherwise (strings, no window, window too small for this
 * exchange -- decided identically on every executor) it runs the two steps one after the other.  Either way the stored
 * partitions afterwards are what b200_stage_execute + b200_exchange_stage leave.  `out` / `n_out` describe this map
 * task's output as b200_stage_execute does; `stats` may be NULL.  Window memory is recycled when b200_remove_job_data
 * leaves the engine without stored partitions.  Counters: "fused_exchanges", "exchange_window_bytes". */
int b200_stage_execute_exchange(b200_stage* s, int input_partition, const volatile int32_t* cancel_flag,
                                b200_shuffle_write_partition* out, int cap, int* n_out, b200_exchange_stats* stats);

/* ---- the reference's shuffle file format (SURVEY.md 8(f) rank 2) -----------------------------------
 * Arrow IPC streams with LZ4_FRAME body compression, written the way ShuffleWriterExec / SortShuffleWriterExec write
 * them (shuffle_writer.rs:317-328, sort_shuffle/writer.rs:419-513, index format sort_shuffle/index.rs:18-33) and read the
 * way ShuffleReaderExec reads them (shuffle_reader.rs:698-771, sort_shuffle/reader.rs:51-84): GPU and CPU executors can
 * consume each other's stage output, and HBM-resident partitions can be persisted under `work_dir` so that they survive
 * the executor.  b200_ipc_encode / b200_ipc_decode are the host-only codec (no CUDA call). */
int b200_ipc_encode(struct ArrowArray* batch, struct ArrowSchema* schema, int compress, int64_t max_rows_per_message,
                    uint8_t** out, uint64_t* out_len);           /* releases batch / schema; free *out with b200_ipc_free */
void b200_ipc_free(uint8_t* p);
int b200_ipc_decode(const uint8_t* buf, uint64_t len, struct ArrowArray* out, struct ArrowSchema* out_schema);  /* one or several back-to-back streams */
/* sort_layout 0: work_dir/job/stage/{out_part}/data-{file_id}.arrow (or data.arrow when the stage was un-partitioned);
 * sort_layout 1: work_dir/job/stage/{file_id}/data.arrow + data.arrow.index with n_out_partitions + 1 offsets */
int b200_shuffle_write_files(b200_engine* e, const char* job_id, int64_t stage_id, const char* work_dir, int n_out_partitions,
                             int sort_layout, uint64_t* files_written, uint64_t* bytes_written);
int b200_shuffle_read_file(b200_engine* e, const char* job_id, int64_t stage_id, int out_partition, int64_t file_id,
                           const char* path, uint64_t byte_offset, uint64_t byte_length, int use_index);

/* ---- pinned host staging (harness side of "RecordBatches are pinned and DMA'd") ------------- */
void* b200_host_alloc_pinned(uint64_t bytes);
void b200_host_free_pinned(void* p);

/* Version / build info: "b200exec <ver> sm_100a" */
const char* b200_version(void);

#ifdef __cplusplus
}
#endif
#endif /* B200EXEC_H */
