/*
 * include/dfd_b200.h — C ABI of the B200-native hash-repartition shuffle.
 *
 * This is the drop-in boundary for ONE path of datafusion-distributed: the
 * hash-repartition shuffle (producer `RepartitionExec(Hash(keys, P*T))` ->
 * exchange -> consumer `NetworkShuffleExec`).  Plain C types only (pointers,
 * sizes, Arrow C Data Interface structs); no torch / C++ types cross it.  A
 * Rust `ExecutionPlan` shim binds these symbols with `extern "C"` (see
 * INTEGRATION.md); tests and bench.py bind them with ctypes.
 *
 * Each entry point cites the reference interface it replaces
 * (paths relative to the datafusion-distributed checkout @ f032463).
 *
 * Threading: every call may come from any thread.  A dfd_ctx owns one GPU's
 * streams and scratch; calls on the same ctx are serialised internally.
 * Errors: 0 == DFD_OK; otherwise a dfd_status code, with a human-readable
 * message retrievable (per thread) through dfd_last_error().  Nothing aborts
 * the process.  There is NO CPU fallback anywhere behind this ABI: if CUDA is
 * unavailable every compute entry point returns DFD_ERR_CUDA.
 */
#ifndef DFD_B200_H
#define DFD_B200_H

#include <stddef.h>
#include <stdint.h>

#include "arrow_c_abi.h"

#ifdef __cplusplus
extern "C" {
#endif

#define DFD_ABI_VERSION 1

/* Maps onto DataFusionError in the Rust shim:
 * INVALID_ARGUMENT/UNSUPPORTED -> Plan/NotImplemented, OOM/CAPACITY ->
 * ResourcesExhausted, CUDA/NCCL -> Execution, INTERNAL -> Internal
 * (reference error transport: src/protobuf/errors/mod.rs:22-69). */
typedef enum {
    DFD_OK = 0,
    DFD_ERR_INVALID_ARGUMENT = 1,
    DFD_ERR_OOM = 2,
    DFD_ERR_CUDA = 3,
    DFD_ERR_NCCL = 4,
    DFD_ERR_INTERNAL = 5,
    DFD_ERR_UNSUPPORTED = 6,
    DFD_ERR_CAPACITY = 7
} dfd_status;

typedef struct dfd_ctx dfd_ctx;                 /* one per GPU / worker            */
typedef struct dfd_partitioner dfd_partitioner; /* ≙ BatchPartitioner::Hash        */

/* Physical layout of one column, device- or host-resident: the buffers of an
 * Arrow array flattened (what ArrowArray.buffers[] holds for these types). */
typedef enum {
    DFD_COL_FIXED = 0,     /* primitive values, `width` bytes each (1,2,4,8,16)     */
    DFD_COL_BOOL = 1,      /* bit-packed values                                     */
    DFD_COL_UTF8 = 2,      /* int32 offsets + bytes; hashed as Rust `str`           */
    DFD_COL_LARGE_UTF8 = 3,/* int64 offsets + bytes                                 */
    DFD_COL_BINARY = 4     /* int32 offsets + bytes; hashed as Rust `[u8]`          */
} dfd_col_kind;

typedef struct {
    int32_t kind;            /* dfd_col_kind                                         */
    int32_t width;           /* DFD_COL_FIXED: bytes per value                       */
    void* values;            /* values / bitmap / string bytes                       */
    void* offsets;           /* var-width kinds only                                 */
    uint8_t* validity;       /* Arrow validity bitmap (LSB first) or NULL = no nulls */
    int64_t offset;          /* Arrow logical offset (rows) into the buffers         */
    int64_t values_bytes;    /* var-width kinds: size of `values` in bytes (for an OUTPUT
                                column: its capacity); ignored for fixed / bool       */
} dfd_column;

/* Counters of the shuffle path; the reference exposes the same quantities as
 * DataFusion metrics on NetworkShuffleExec (`bytes_transferred`,
 * `elapsed_compute`, output_rows; src/worker/worker_connection_pool.rs:160-181). */
typedef struct {
    uint64_t calls;          /* partition calls since creation / last reset          */
    uint64_t rows;           /* rows partitioned                                      */
    uint64_t bytes_in;       /* payload bytes read (algorithmic)                      */
    uint64_t bytes_out;      /* payload bytes written (algorithmic)                   */
    uint64_t kernel_launches;/* CUDA kernels launched by this library                 */
    double hist_ms;          /* sums of CUDA-event durations (profiling mode only)    */
    double scan_ms;
    double scatter_ms;
    double h2d_ms;
    double d2h_ms;
    uint64_t scatter_launches;
    uint64_t onepass_reruns; /* single-pass calls that overflowed a region and re-ran exactly */
} dfd_metrics;

/* ---- library / context ------------------------------------------------ */

int dfd_abi_version(void);
/* Thread-local message of the last failing call on this thread ("" if none). */
const char* dfd_last_error(void);
const char* dfd_status_name(int status);
int dfd_device_count(int* out_count);

/* One context per GPU == one worker (reference: `Worker`,
 * src/worker/worker_service.rs:39-49; one process per GPU in this build). */
int dfd_ctx_create(int device, dfd_ctx** out);
void dfd_ctx_destroy(dfd_ctx* ctx);
/* cudaStream_t the compute kernels are launched on (for external event timing). */
void* dfd_ctx_stream(dfd_ctx* ctx);
int dfd_ctx_synchronize(dfd_ctx* ctx);
/* When on, every kernel is bracketed by CUDA events on its launch stream and
 * the durations are accumulated into dfd_metrics (costs one sync per call). */
int dfd_ctx_set_profiling(dfd_ctx* ctx, int on);

/* Buffer helpers so a host language without CUDA bindings can own memory.
 * Host allocations are pinned (page-locked). */
int dfd_device_alloc(dfd_ctx* ctx, size_t bytes, void** out);
int dfd_device_free(dfd_ctx* ctx, void* ptr);
int dfd_host_alloc(dfd_ctx* ctx, size_t bytes, void** out);
int dfd_host_free(dfd_ctx* ctx, void* ptr);
int dfd_memcpy_h2d(dfd_ctx* ctx, void* dst_device, const void* src_host, size_t bytes);
int dfd_memcpy_d2h(dfd_ctx* ctx, void* dst_host, const void* src_device, size_t bytes);
int dfd_memset_device(dfd_ctx* ctx, void* dst_device, int value, size_t bytes);
/* Writes >L2-size scratch so the next timed launch starts with a cold L2. */
int dfd_flush_l2(dfd_ctx* ctx);

/* CUDA-event stopwatch on the compute stream (bench.py's timed region). */
int dfd_timer_start(dfd_ctx* ctx);
int dfd_timer_stop(dfd_ctx* ctx, float* out_ms);

/* ---- hash partitioner --------------------------------------------------
 * Replaces DataFusion's `BatchPartitioner::try_new(Partitioning::Hash(exprs,
 * n), ..)` + `partition()` as configured by the reference at
 * src/execution_plans/network_shuffle.rs:126-134 (Hash(keys, P * task_count))
 * and executed at src/worker/impl_execute_task.rs:77-86.
 *   key_cols : indices of the key columns (`Column` exprs) in hashing order
 *   seeds    : ahash RandomState::with_seeds arguments; NULL selects
 *              DataFusion's REPARTITION_RANDOM_STATE = (0,0,0,0)
 * num_partitions must be in [1, 4096] (DFD_MAX_PARTITIONS; DataFusion stages use target_partitions x tasks,
 * typically tens to hundreds); the per-CTA shared-memory need of the scatter kernels is checked at create time.
 * The peer-store exchange transports keep an extra per-destination table in shared memory and accept up to
 * ~3 400 partitions (DFD_ERR_UNSUPPORTED above; the push and NCCL transports have no such limit). */
#define DFD_MAX_PARTITIONS 4096
int dfd_partitioner_create(dfd_ctx* ctx, uint32_t num_partitions, const int32_t* key_cols,
                           int n_keys, const uint64_t* seeds, dfd_partitioner** out);
void dfd_partitioner_destroy(dfd_partitioner* p);
uint32_t dfd_partitioner_num_partitions(const dfd_partitioner* p);
/* How a FIXED key column is fed to the hasher.  Primitive values are one `write_u{8,16,32,64,128}` (PLAIN).
 * Arrow's interval structs `#[derive(Hash)]`, i.e. one write per field, and DataFusion hashes them through that
 * impl (datafusion-common hash_utils `hash_value!(.., IntervalDayTime, IntervalMonthDayNano)`), so an
 * Interval(DayTime) key (format "tiD", 8 bytes {days: i32, milliseconds: i32}) and an Interval(MonthDayNano)
 * key ("tin", 16 bytes {months: i32, days: i32, nanoseconds: i64}) must be declared here; as PAYLOAD they are
 * plain 8 / 16-byte values.  dfd_repartition_exec_create does this from the schema's format strings. */
typedef enum { DFD_KEY_HASH_PLAIN = 0, DFD_KEY_HASH_INTERVAL_DAY_TIME = 1, DFD_KEY_HASH_INTERVAL_MONTH_DAY_NANO = 2 } dfd_key_hash_mode;
int dfd_partitioner_set_key_hash_mode(dfd_partitioner* p, int key_index, int mode);
/* Dictionary-encoded key columns (Arrow Dictionary<K, V>; the reference's bench schema has Dictionary<Int32, Utf8>,
 * src/execution_plans/benchmarks/fixture.rs:13-33).  DataFusion's hash_dictionary hashes the dictionary VALUES once
 * (create_hashes over the values array) and every row takes dict_hashes[index]; a null index or a null dictionary value
 * leaves the running hash untouched.  Pass the INDICES as the (fixed-width, signed) key column and declare its dictionary
 * here: dict_hashes_device = the values' hashes (dfd_hash_columns_device over the values column, asynchronous on the
 * context's stream), dict_validity_device = the values' validity bitmap or NULL.  The pointers must stay valid while
 * partition calls use them; NULL hashes turn the key back into a plain one.  As PAYLOAD the indices are a plain
 * fixed-width column and the dictionary travels by reference (host operator) — see dfd_repartition_exec. */
int dfd_partitioner_set_key_dictionary(dfd_partitioner* p, int key_index, const uint64_t* dict_hashes_device,
                                       const uint8_t* dict_validity_device);
/* hashes_device[i] = create_hashes(cols, RandomState::with_seeds(seeds or 0,0,0,0))[i] — raw 64-bit row hashes
 * (null rows of a single column hash to 0).  Asynchronous on dfd_ctx_stream(). */
int dfd_hash_columns_device(dfd_ctx* ctx, const dfd_column* cols, int n_cols, int64_t n_rows, const uint64_t* seeds,
                            uint64_t* hashes_device);

/* dest[i] = create_hashes(key columns)[i] % num_partitions, for device
 * columns; `dest_device` holds n_rows uint32.  (Debug/parity entry point for
 * `create_hashes` + `hash % partitions`.) */
int dfd_partition_ids_device(dfd_partitioner* p, const dfd_column* cols, int n_cols,
                             int64_t n_rows, uint32_t* dest_device);

/* The hot path, device-resident: partition `n_rows` rows of `n_cols` columns
 * into num_partitions destinations.  Output column c is ONE buffer
 * (out_cols[c].values, capacity n_rows) in which destination p occupies rows
 * [part_starts[p], part_starts[p+1]) — N contiguous per-destination Arrow
 * buffers, zero-copy sliceable.  Within a destination, rows keep input order
 * (SURVEY.md §8a invariant iii; DataFusion pushes indices in row order).
 * part_starts_host (N+1 int64, may be NULL) is filled after a stream sync;
 * with NULL the call is fully asynchronous on dfd_ctx_stream() and the device
 * copy is available through dfd_partitioner_part_starts_device().
 * Bit-packed outputs — out_cols[c].validity of a nullable column and the `values` of a
 * DFD_COL_BOOL column — are written with 32-bit atomic ORs: each must be 4-byte aligned and
 * hold ceil(n_rows / 32) * 4 bytes (whole words; output offset is 0).  The library zeroes
 * them itself at the start of the call.
 * Variable-width payload columns (Utf8 / LargeUtf8 / Binary; K4): out_cols[c]
 * carries `offsets` (n_rows + 1 entries of the input's offset width) and
 * `values` with `values_bytes` >= the input's byte count; the output is one
 * offsets buffer + one byte buffer in destination order, so destination p is
 * again the zero-copy slice [part_starts[p], part_starts[p+1]). */
int dfd_partition_device(dfd_partitioner* p, const dfd_column* in_cols, int n_cols,
                         int64_t n_rows, const dfd_column* out_cols, int64_t* part_starts_host);
const int64_t* dfd_partitioner_part_starts_device(const dfd_partitioner* p);

/* Single-pass form of the hot path (same reference interface as dfd_partition_device:
 * BatchPartitioner::partition, src/worker/impl_execute_task.rs:77-86).  ONE kernel hashes every
 * row once, ranks it, resolves the per-tile write cursors by decoupled look-back and scatters —
 * there is no histogram pass, so destination totals are not known before the first store.
 * Destination p therefore owns a fixed REGION of every output column: rows
 * [part_starts[p], part_starts[p] + part_counts[p]) with part_starts[p] = p * region_rows — still
 * N contiguous, zero-copy sliceable per-destination buffers, in input order.
 *   out_cols[c] must hold N * region_rows rows, and N * region_rows >= n_rows.
 *   If a destination outgrows its region (skewed keys) nothing is lost: collection re-runs
 *   the kernel with exact regions (part_starts = prefix sums of the now-known counts, dense).
 *   Variable-width payload columns, boolean-only schemas and N > 256 take the two-pass
 *   path internally and return the dense layout through the same (start, count) contract.
 * part_starts_host / part_counts_host (N int64 each): both NULL = asynchronous on
 * dfd_ctx_stream(); fetch the result later with dfd_partitioner_collect (which synchronises
 * and performs the exact re-run if needed).  Bit-packed outputs follow the rules of
 * dfd_partition_device with n_rows replaced by N * region_rows. */
int dfd_partition_device_onepass(dfd_partitioner* p, const dfd_column* in_cols, int n_cols, int64_t n_rows,
                                 const dfd_column* out_cols, int64_t region_rows, int64_t* part_starts_host,
                                 int64_t* part_counts_host);
int dfd_partitioner_collect(dfd_partitioner* p, int64_t* part_starts_host, int64_t* part_counts_host);

/* ---- host operator: RepartitionExec(Hash) over Arrow C Data / C Stream ----
 * Replaces, on one worker, `RepartitionExec::try_new(input,
 * Partitioning::Hash(exprs, n))` (built by the reference at
 * src/execution_plans/network_shuffle.rs:126-134) and
 * `ExecutionPlan::execute(partition, ctx) -> SendableRecordBatchStream`
 * (called at src/worker/impl_execute_task.rs:77-86).  Input and output are
 * HOST record batches; host<->device copies happen inside.
 *   schema    : struct ("+s") schema of the input batches (borrowed)
 *   push      : feed one input RecordBatch (struct ArrowArray); ownership of
 *               `batch` moves to the operator (released after its H2D copy).
 *               Single producer thread; blocks on the pipeline depth, and — with
 *               dfd_exec_options.max_pinned_chunks — on consumers that have not
 *               released their batches yet (back-pressure).
 *   finish    : end of input; drains the pipeline.
 *   run       : pull `input` (≙ child.execute()) to exhaustion, then finish.
 *   execute   : stream of destination `partition`'s batches; get_next blocks
 *               until a batch is ready or the input is finished.  Batches are
 *               zero-copy slices of pooled pinned buffers; only non-empty
 *               batches are emitted; an operator error is delivered to every
 *               partition stream (EIO + get_last_error), like the reference
 *               (src/worker/worker_connection_pool.rs:393-397).
 * Rows inside (one input chunk, one destination) keep input order.  Input
 * batches of every shape (validity bitmaps, booleans, strings, views, lists)
 * are appended to the open chunk until it holds chunk_rows rows — bitmaps are
 * concatenated at bit granularity, string offsets re-based — so small batches
 * cost no extra kernel launches; only a batch with a DIFFERENT dictionary
 * (or > 2 GiB of string bytes under 32-bit offsets) starts a new chunk early.
 * Supported columns: fixed-width primitives (incl. Decimal128, timestamps,
 * dates, intervals), Boolean, Utf8 / LargeUtf8 / Binary, Utf8View / BinaryView
 * (converted to offsets + bytes on the way in; the output batches carry
 * compact views over one data buffer per chunk — the effect of the reference's
 * `gc()` before its network hop, src/worker/impl_execute_task.rs:248-271) and
 * Dictionary<integer, flat values> (the indices are scattered, every output
 * batch references the input batch's dictionary; dictionary KEYS are hashed
 * through their values on the device), all nullable.  List<Utf8> and
 * List<Binary> (int32 offsets; the `tags` column of the reference's bench
 * schema, src/execution_plans/benchmarks/fixture.rs:13-33) move as PAYLOAD:
 * the operator splits a list column into three hidden variable-width device
 * columns (element lengths + the list's validity, element bytes, element
 * validity), scatters them with the ordinary variable-width kernels, rebuilds
 * the child offsets with a device scan and exports nested Arrow arrays; as a
 * hash KEY a list is refused at create time.  List<fixed-width primitive> (the
 * partial states of array_agg / median) moves the same way, without child offsets.
 * LargeBinary and FixedSizeBinary of
 * 1 / 2 / 4 / 8 / 16 bytes (UUIDs) also move as payload only (DataFusion hashes
 * them as byte slices).  Other nested types (Struct, Map,
 * List of lists / booleans / dictionaries): DFD_ERR_UNSUPPORTED. */
typedef struct dfd_repartition_exec dfd_repartition_exec;

/* Pure host helpers (no GPU needed) for the plan hook that decides whether a stage-head
 * `RepartitionExec(Hash)` can be swapped for the GPU operator
 * (`Worker::add_on_plan_hook`, src/worker/worker_service.rs:91-96):
 *   dfd_arrow_format_layout : Arrow C format string -> (dfd_col_kind, value width);
 *                             DFD_ERR_UNSUPPORTED for formats with no flat layout
 *                             (nested types, 256-bit decimals, FixedSizeBinary of other than 1/2/4/8/16 bytes ...).
 *                             LargeBinary reports the LargeUtf8 layout (int64 offsets + bytes: how it MOVES).
 *   dfd_schema_supported    : DFD_OK iff every column of the record-batch schema is
 *                             supported — flat columns, views, Dictionary<integer, flat>
 *                             and List<Utf8 / Binary>; otherwise DFD_ERR_UNSUPPORTED with
 *                             the reason in dfd_last_error().
 *   dfd_repartition_supported : the same with the hash KEY columns taken into account — what the hook should ask before
 *                             swapping a RepartitionExec(Hash(keys, n)): lists, LargeBinary and FixedSizeBinary(1/2/4/8/16)
 *                             columns travel as payload but cannot be hash keys (DataFusion hashes them as byte slices),
 *                             nor can dictionaries with view-typed values.  dfd_repartition_exec_create applies the same checks. */
int dfd_arrow_format_layout(const char* format, int32_t* kind, int32_t* width);
int dfd_schema_supported(const struct ArrowSchema* schema);
int dfd_repartition_supported(const struct ArrowSchema* schema, const int32_t* key_cols, int n_keys);

typedef struct {
    int64_t chunk_rows;         /* rows per device chunk; 0 = 4Mi                   */
    int32_t pipeline_depth;     /* chunks in flight (H2D | kernels | D2H); 0 = 3    */
    int32_t pinned_pool_chunks; /* pinned output chunks preallocated; 0 = depth + 1 */
    int32_t max_pinned_chunks;  /* 0 = the pool grows on demand (a slow consumer costs pinned memory, nothing blocks);
                                   > 0 = hard bound: push()/finish() BLOCK until a consumer releases a chunk — the
                                   operator's back-pressure (needs concurrent consumers, like the reference's bounded
                                   hand-off, src/worker/worker_connection_pool.rs:151-153) */
    int32_t reserved;
} dfd_exec_options;

typedef struct {
    uint64_t rows_in, rows_out, bytes_h2d, bytes_d2h;
    /* pinned output chunks: held by this operator now / pinned by it (cudaHostAlloc) / taken over from the worker
     * context's cache of chunks that finished operators of the same column layout left behind (the role of the
     * reference workers' caching allocator, benchmarks/cdk/bin/worker.rs:32; bound: env DFD_PINNED_CACHE_BYTES, 4 GiB) */
    uint64_t pinned_chunks, pinned_chunks_allocated, pinned_chunks_reused;
    /* producer-thread wall time inside push()/finish(), and the parts of it spent blocked on a D2H copy of a slot
     * being recycled and on the pinned pool (allocation, or back-pressure when max_pinned_chunks is set) */
    uint64_t ns_push, ns_wait_d2h, ns_wait_pool;
} dfd_exec_stats;

int dfd_repartition_exec_create(dfd_ctx* ctx, const struct ArrowSchema* schema, const int32_t* key_cols,
                                int n_keys, uint32_t num_partitions, const dfd_exec_options* opts,
                                dfd_repartition_exec** out);
void dfd_repartition_exec_destroy(dfd_repartition_exec* x);
int dfd_repartition_exec_push(dfd_repartition_exec* x, struct ArrowArray* batch);
int dfd_repartition_exec_finish(dfd_repartition_exec* x);
/* The producer's INPUT failed: instead of finish(), fail the operator — every partition stream's get_next returns EIO
 * with `message` (rows already queued are still delivered first), exactly as RepartitionExec forwards an input error
 * to all of its output partitions and as the reference fans a task failure out (worker_connection_pool.rs:393-397).
 * Call from the producer thread (in place of push/finish).  No effect after finish() or an earlier error. */
int dfd_repartition_exec_abort(dfd_repartition_exec* x, const char* message);
int dfd_repartition_exec_run(dfd_repartition_exec* x, struct ArrowArrayStream* input);
int dfd_repartition_exec_execute(dfd_repartition_exec* x, uint32_t partition, struct ArrowArrayStream* out);
int dfd_repartition_exec_stats(dfd_repartition_exec* x, dfd_exec_stats* out);

/* ---- inter-worker exchange (one worker per GPU, single NVSwitch box) -------
 * Replaces the reference's shuffle data plane: the per-(consumer, producer)
 * gRPC/Arrow-Flight streams served by `impl_execute_task`
 * (src/worker/impl_execute_task.rs:36-169), demultiplexed by `WorkerConnection`
 * (src/worker/worker_connection_pool.rs:143-390) and merged by
 * `NetworkShuffleExec::execute` (src/execution_plans/network_shuffle.rs:213-238).
 * Addressing follows the reference exactly: with N = P * T global partitions,
 * global partition g belongs to consumer task g / P as its local partition
 * g % P (off = P * task_index, network_shuffle.rs:219).
 *
 *   DFD_EXCHANGE_NCCL  : local K1/K1b/K2 into a staging buffer, ncclAllGather of
 *                        the T x N count matrix, grouped ncclSend/ncclRecv.
 *   DFD_EXCHANGE_FUSED : K2 stores each destination's runs directly into the
 *                        owner's receive window over NVLink (CUDA-IPC peer
 *                        memory); counts all-gather before, one barrier after.
 *                        Fixed-width non-null columns only.
 * Control plane (who is rank r, the 128-byte NCCL id) stays with the caller —
 * in the reference that is the gRPC coordinator channel / TaskKey plumbing. */
typedef struct dfd_exchange dfd_exchange;
enum { DFD_EXCHANGE_NCCL = 0, DFD_EXCHANGE_FUSED = 1 };

/* ncclGetUniqueId: call on one worker, ship the 128 bytes to the others. */
int dfd_nccl_unique_id(void* out_128_bytes);
/* Collective over all `world` workers (≙ the T tasks of the stage pair). */
int dfd_exchange_create(dfd_ctx* ctx, int rank, int world, const void* nccl_unique_id, dfd_exchange** out);
void dfd_exchange_destroy(dfd_exchange* x);
int dfd_exchange_rank(const dfd_exchange* x);
int dfd_exchange_world(const dfd_exchange* x);
/* Collective: allocate this worker's receive window (fused mode) and map every
 * peer's window through CUDA IPC.  window_bytes must be the SAME on every worker (slot sizes, column
 * offsets and capacity checks are derived from it on each producer); a mismatch fails with
 * DFD_ERR_INVALID_ARGUMENT on every worker. */
int dfd_exchange_setup_window(dfd_exchange* x, size_t window_bytes);

/* Pure host arithmetic of the exchange (no GPU needed; also what the Rust shim
 * or a CPU test harness would call): from counts[world][N] (rows producer r
 * holds for global partition g, N = partitions_per_task * world) compute, for
 * worker `rank` (any output pointer may be NULL):
 *   send_start[N]      start row of destination g in rank's partitioned buffer
 *   recv_start[P*world] start row, in rank's receive buffer, of (local
 *                      partition q, producer r) at index q*world + r
 *   part_starts[P+1]   rank's output partition boundaries
 *   dest_base[N]       start row of rank's rows inside the OWNER's receive
 *                      buffer for destination g (fused mode)
 *   recv_rows          total rows rank receives                              */
int dfd_exchange_plan(int world, uint32_t partitions_per_task, int rank, const int64_t* counts,
                      int64_t* send_start, int64_t* recv_start, int64_t* part_starts,
                      int64_t* dest_base, int64_t* recv_rows);

/* Collective shuffle of device-resident columns.  On return (stream
 * synchronised) this worker holds its P = partitions_per_task destinations:
 * out column c, rows [part_starts_host[q], part_starts_host[q+1]) = local
 * partition q = global partition rank*P + q, producers' rows in task order,
 * each producer's rows in its input order.
 *   NCCL mode : out_cols[c].values (/offsets/validity) are caller buffers of
 *               out_capacity_rows; every column kind of dfd_partition_device
 *               is supported.  A column travels with a validity lane iff
 *               out_cols[c].validity != NULL — set it from the SCHEMA's
 *               nullable flag so that every worker agrees, whether or not its
 *               own rows contain nulls; string outputs need values_bytes.
 *   FUSED mode: out_cols[c].values are SET to point into the receive window
 *               (valid until the next shuffle); out_capacity_rows is ignored.
 * DFD_ERR_CAPACITY if a receive buffer / window is too small (nothing is
 * written in that case). */
int dfd_shuffle_device(dfd_exchange* x, dfd_partitioner* p, int mode, const dfd_column* in_cols, int n_cols,
                       int64_t n_rows, uint32_t partitions_per_task, dfd_column* out_cols,
                       int64_t out_capacity_rows, int64_t* part_starts_host);
/* DFD_EXCHANGE_FUSED without the final host synchronisation: the whole shuffle is enqueued on
 * dfd_ctx_stream() and the call returns (out_cols already point into the receive window).
 * dfd_exchange_wait() synchronises, reports DFD_ERR_CAPACITY if a window overflowed and fills
 * part_starts_host[P+1] (may be NULL).  Lets consecutive collectives pipeline on the stream. */
int dfd_shuffle_device_async(dfd_exchange* x, dfd_partitioner* p, const dfd_column* in_cols, int n_cols,
                             int64_t n_rows, uint32_t partitions_per_task, dfd_column* out_cols);
int dfd_exchange_wait(dfd_exchange* x, int64_t* part_starts_host);

/* Single-pass fused shuffle (the fast path; collective, asynchronous on dfd_ctx_stream()).  Every (consumer partition
 * q, producer r) pair owns a FIXED sub-window of the consumer's receive window, so producers need no global counts
 * before their first store: one k_scatter_onepass launch per worker hashes every row once and stores straight into
 * the owners' windows over NVLink; counts, overflow and completion are peer-memory flags in the window headers —
 * no NCCL call on the critical path.  This is the reference's own contract: a consumer partition is the merge of
 * one stream per producer, unordered across producers (src/execution_plans/network_shuffle.rs:230-237 `select_all`);
 * within a segment rows keep the producer's input order.
 *   out_cols[c].values are SET to point into this worker's receive window (valid until the next shuffle).
 *   dfd_exchange_collect synchronises and returns, for local partition q and producer r, the segment
 *   rows [seg_starts[q*T + r], +seg_counts[q*T + r]) of every out column (T = workers).  If any sub-window
 *   overflowed on any worker (skew), collect re-runs the shuffle through the exact two-pass fused path on every
 *   worker (all see the same flags) and rewrites out_cols (may be NULL if the caller keeps the originals) — the
 *   segments then describe that dense layout.
 * Column kinds: fixed-width non-null columns with <= 256 partitions take the single-pass kernel.  Nullable, boolean and
 * Utf8 / LargeUtf8 / Binary columns (every kind dfd_partition_device moves) take the PUSH transport, also NCCL-free:
 * local partition -> flag-based all-gather of the row / byte counts -> each destination's contiguous runs (values,
 * shifted bitmaps, re-based string offsets, string bytes) are stored into the owner's window by k_push_runs.  There a
 * segment starts on a 32-row boundary; out_cols[c].offsets / .validity are set like .values, and the string offsets
 * of a segment index the column's single `values` byte buffer directly (Arrow layout, zero-copy sliceable).  ON
 * ENTRY out_cols[c].validity != NULL marks column c as nullable in the SCHEMA (all workers must agree), whether or
 * not this worker's rows contain nulls; in_cols[c].values_bytes must hold the byte size of a string column's data. */
int dfd_shuffle_device_onepass(dfd_exchange* x, dfd_partitioner* p, const dfd_column* in_cols, int n_cols, int64_t n_rows,
                               uint32_t partitions_per_task, dfd_column* out_cols);
int dfd_exchange_collect(dfd_exchange* x, dfd_column* out_cols, int64_t* seg_starts, int64_t* seg_counts);
uint64_t dfd_exchange_onepass_fallbacks(const dfd_exchange* x);
/* Profiling (dfd_ctx_set_profiling): mean CUDA-event milliseconds of the three stream phases of the single-pass shuffles
 * since the last call: [0] k_xchg_signal_ready, [1] k_scatter_onepass<PEER> (+ follow-ups), [2] k_xchg_publish_wait. */
int dfd_exchange_phase_ms(dfd_exchange* x, double* out3, uint64_t* n_shuffles);

/* ---- device-side PartialReduce ahead of the shuffle ----------------------------------------------------------------
 * The reference inserts AggregateExec(mode = PartialReduce) above the producers' hash RepartitionExec
 * (src/distributed_planner/partial_reduce_below_network_shuffles.rs:17-100): once rows are hash-partitioned, equal group
 * keys share a destination, so merging their aggregate states there shrinks the shuffle.  Input: a DENSE partitioned
 * table on the device (the output of dfd_partition_device: partition p = rows [part_starts[p], part_starts[p+1])),
 * `key_cols` = the group-by columns, agg_ops[c] = how state column c merges (-1 for the key columns).  Output: one row
 * per distinct key, partition p = rows [out_part_starts[p], out_part_starts[p+1]) of out_cols (capacity n_rows; row order
 * inside a partition is unspecified, like a hash aggregate's).  Feed it to dfd_exchange_gather(DFD_ROUTE_SHUFFLE) — the
 * rows never leave the GPU between Partial aggregation, repartition, PartialReduce and the exchange.
 * Synchronous.
 * Columns: group keys are fixed-width (1 / 2 / 4 / 8 / 16 bytes), Boolean (bit-packed; the Arrow offset is a bit offset) or
 * Utf8 / LargeUtf8 / Binary; aggregate states are fixed-width.  Keys and states may be nullable.  out_cols[c] has the
 * kind (and offset width) of in_cols[c]; an op on a Boolean or string column, a kind / offset-width mismatch, and
 * Dictionary or view columns give DFD_ERR_UNSUPPORTED.
 * Nullability: a column is nullable iff out_cols[c].validity != NULL (the convention of dfd_shuffle_device_onepass).  A
 * nullable input needs an output validity bitmap (DFD_ERR_UNSUPPORTED otherwise); a non-null input with an output bitmap
 * gets every bit set.  Bit-packed outputs (validity, Boolean key values) follow dfd_partition_device: 4-byte aligned,
 * ceil(n_rows / 32) * 4 bytes, output offset 0; the library zeroes them itself and writes them with 32-bit atomic ORs.
 * String keys: out_cols[c].offsets gets n_out + 1 entries of the input's offset width and out_cols[c].values the
 * representatives' bytes in output-row order, so partition p is the zero-copy slice [out_part_starts[p],
 * out_part_starts[p+1]) as in dfd_partition_device.  out_cols[c].values_bytes is the byte capacity: if it is smaller than
 * the group keys' bytes the call returns DFD_ERR_CAPACITY with the needed size in the message and writes no output column.
 * n_rows == 0 writes offsets[0] = 0 of every string output.
 * Semantics (tests/test_reduce_exact_gpu.py, tests/test_reduce_nullable_gpu.py):
 *   - Groups never cross input partitions: a row joins a group only if its keys are equal AND it lies in the same
 *     input partition, so the same key in two partitions is two groups, each in its own output partition, whatever
 *     decided part_starts.  Fixed-width key equality is byte equality (float keys: to_bits equality; +0.0, -0.0 and every
 *     NaN payload are distinct groups).  String keys are equal iff their lengths and bytes are; Boolean keys by value.
 *   - NULL is a group value, as in SQL GROUP BY: the NULLs of a key column are equal to each other and differ from every
 *     non-null value (an empty string and NULL are two groups); with several keys the null pattern is part of the key.
 *     The bytes under a null key are never read.  A null key is written as zero bytes (a string: length 0, a Boolean: 0).
 *   - Null input states are skipped; an output state is null iff every input state of its group is null, and is then
 *     written as 0.  The value bytes of a null input state never reach the result.
 *   - SUM_I64 and SUM_I128 wrap (two's complement, mod 2^64 / 2^128); MIN / MAX_I64 are exact.
 *   - MIN / MAX_F64 follow IEEE-754 totalOrder (Rust's f64::total_cmp): -NaN < -inf < ... < -0.0 < +0.0 < ... < +inf
 *     < +NaN.  The result is bit-identical to a sequential fold in any row order (an all-NaN group gives a NaN; a group
 *     of +0.0 and -0.0 gives -0.0 / +0.0).
 *   - Parity unpinned: DataFusion's groups accumulators (MIN / MAX, and the null handling of every op) are not in this
 *     repository, so agreement with their float order and null semantics is not checked (DESIGN.md §2).
 *   - SUM_F64 is the only result that is not bit-exact: the additions land in an unspecified order, and for a group of
 *     k finite rows |result - exact sum| <= (k-1) * 2^-53 * sum|x|.  A NaN row, or +inf with -inf, gives NaN.
 * Kernel launches (dfd_metrics.kernel_launches) for n_rows > 0: 4 + F + 4 * S, where F = 1 if some state column is
 * MIN / MAX_F64 or a MIN / MAX column with an input validity bitmap (the finishing pass), else 0, and S = the number of
 * string key columns (a 3-launch lengths -> offsets scan and one byte gather each).  n_rows == 0 launches nothing. */
typedef enum {
    DFD_AGG_SUM_I64 = 0,  /* also COUNT states */
    DFD_AGG_SUM_F64 = 1,
    DFD_AGG_MIN_I64 = 2,
    DFD_AGG_MAX_I64 = 3,
    DFD_AGG_SUM_I128 = 4, /* Decimal128 sums */
    DFD_AGG_MIN_F64 = 5,
    DFD_AGG_MAX_F64 = 6
} dfd_agg_op;
int dfd_partial_reduce_device(dfd_ctx* ctx, const dfd_column* in_cols, int n_cols, int64_t n_rows, const int32_t* key_cols, int n_keys,
                              const int32_t* agg_ops, const int64_t* part_starts_device, uint32_t num_partitions,
                              const dfd_column* out_cols, int64_t* out_part_starts_host, int64_t* out_part_starts_device);

/* ---- back-pressure: a shuffle delivered in rounds ----------------------------------------------------------------
 * Replaces the reference's byte-budget back-pressure between WorkerConnection and its consumers
 * (src/worker/worker_connection_pool.rs:151-153, 251-257): a consumer that cannot hold more data throttles its producers,
 * it never fails the query.  Here the bounded resource is the consumer's receive window.  dfd_shuffle_stream_next
 * delivers the next ROUND of the shuffle (out_cols + P x T segments, valid until the following call — the consumer
 * drains in between).  When a round does not fit some consumer's window — skew, a window smaller than the data — every
 * worker sees the same global counts, cuts the remaining rows of every producer into finer ranges and retries with
 * less data; nothing fails unless a single row cannot fit.  Collective: every worker calls begin / next / end alike.
 * `nullable[c]` (may be NULL) is the schema's nullable flag of column c. */
typedef struct dfd_shuffle_stream dfd_shuffle_stream;
int dfd_shuffle_stream_begin(dfd_exchange* x, dfd_partitioner* p, const dfd_column* in_cols, int n_cols, int64_t n_rows,
                             uint32_t partitions_per_task, const uint8_t* nullable, dfd_shuffle_stream** out);
int dfd_shuffle_stream_next(dfd_shuffle_stream* s, dfd_column* out_cols, int64_t* seg_starts, int64_t* seg_counts, int* done);
int dfd_shuffle_stream_stats(const dfd_shuffle_stream* s, uint64_t* rounds, uint64_t* splits);
void dfd_shuffle_stream_end(dfd_shuffle_stream* s);

/* ---- sibling exchanges over the same transport (no repartition) ---------------------------------------------
 * NetworkCoalesceExec (src/execution_plans/network_coalesce.rs:75-120, execute :170-240) and NetworkBroadcastExec
 * (src/execution_plans/network_broadcast.rs:119-254) move whole partitions between stages; here they ride the push
 * transport of the shuffle (flag-based count all-gather + k_push_runs peer stores; every column kind; NCCL-free).
 * Every worker is producer task `rank` and holds P partitions = the row slices [slice_starts[j], slice_starts[j+1])
 * of in_cols; workers 0 .. consumer_tasks-1 are the consumer tasks.
 *   DFD_ROUTE_SHUFFLE  : the rows are ALREADY hash-partitioned into partitions x workers slices (global partitions, e.g. by
 *                        dfd_partition_device [+ dfd_partial_reduce_device]): slice g goes to consumer g / partitions as
 *                        segment (g % partitions) * T + r — the exchange half of the shuffle without re-partitioning.
 *                        consumer_tasks must equal the number of workers; slice_starts has partitions x workers + 1 entries.
 *   DFD_ROUTE_COALESCE : consumer c receives the P partitions of each producer in its contiguous group
 *                        (dfd_coalesce_task_group == the reference's task_group); its output partition
 *                        i = (producer - group.start) * P + j; groups shorter than the longest get empty partitions.
 *   DFD_ROUTE_BROADCAST: every consumer receives every producer's P partitions; output partition j is the merge of
 *                        segments j * T + r (r = producer task).
 * Collective and synchronous.  dfd_exchange_collect then returns dfd_exchange_pending_segments() (start, count)
 * pairs in the order above; out_cols are set like in dfd_shuffle_device_onepass (same nullable convention). */
enum { DFD_ROUTE_SHUFFLE = 0, DFD_ROUTE_COALESCE = 1, DFD_ROUTE_BROADCAST = 2 };
int dfd_coalesce_task_group(int input_task_count, int task_index, int task_count, int* start_task, int* len, int* max_len);
/* Pure host helper (no GPU): the routing table every worker derives for an exchange — which producer task and which of its
 * slices feed segment `segment` of consumer task `consumer` (`*producer` = -1: a padding segment of an uneven coalesce
 * group), and how many segments that consumer has (`*n_segments`; 0 for workers that are not consumer tasks).  Out pointers
 * may be NULL.  This is the index arithmetic of NetworkShuffleExec::execute (network_shuffle.rs:219-231: off = P x task_index,
 * partition off + p from every producer), NetworkCoalesceExec::execute (network_coalesce.rs:205-226) and
 * NetworkBroadcastExec::execute (network_broadcast.rs:230-241). */
int dfd_route_segment_source(int route, uint32_t partitions, int producer_tasks, int consumer_tasks, int consumer, uint32_t segment,
                             int* producer, uint32_t* slice, uint32_t* n_segments);
int dfd_exchange_gather(dfd_exchange* x, int route, const dfd_column* in_cols, int n_cols, const int64_t* slice_starts,
                        uint32_t partitions, int consumer_tasks, dfd_column* out_cols);
uint32_t dfd_exchange_pending_segments(const dfd_exchange* x);

/* Host-to-host collective shuffle (end-to-end path of the multi-worker exchange; replaces, per
 * worker, "execute the producer plan, Flight-encode, stream, decode" of
 * src/worker/impl_execute_task.rs:36-169 + src/worker/worker_connection_pool.rs:143-390 for
 * fixed-width non-null columns).  HOST in_cols (n_rows) -> HOST out_cols (out_capacity_rows;
 * pinned memory from dfd_host_alloc gives full PCIe rate).  The rows are cut into n_chunks
 * equal pieces — one fused collective shuffle each, so every worker must pass the same
 * n_chunks — and H2D(i+1) | shuffle(i) | D2H(i-1) overlap (needs a receive window of
 * at least 2 x the per-chunk receive size).  Output is chunk-major, like a stream of
 * per-destination batches: chunk i / local partition q = rows
 * [chunk_part_starts[i*(P+1)+q], chunk_part_starts[i*(P+1)+q+1]) of every out column. */
int dfd_shuffle_host(dfd_exchange* x, dfd_partitioner* p, const dfd_column* in_cols, int n_cols, int64_t n_rows,
                     uint32_t partitions_per_task, int n_chunks, const dfd_column* out_cols,
                     int64_t out_capacity_rows, int64_t* chunk_part_starts);
int dfd_exchange_stats(dfd_exchange* x, uint64_t* bytes_sent, uint64_t* bytes_received, uint64_t* shuffles);

/* Arrow C Device Data Interface export of ONE destination of a dfd_partition_device /
 * dfd_shuffle_device result: a struct array (record batch) of `n_cols` children whose buffers are
 * the device buffers of `cols` (no copy), sliced with `offset = first_row`, `length = n_rows`.
 * device_type = ARROW_DEVICE_CUDA, device_id = the context's GPU, sync_event = a cudaEvent_t*
 * recorded on dfd_ctx_stream() (the consumer waits on it before reading).  The export does not
 * own the column buffers: keep them alive until out->array.release has been called.
 * (≙ handing a RecordBatch of `NetworkShuffleExec::execute(partition)` to a device-side consumer.) */
int dfd_export_partition_device(dfd_ctx* ctx, const dfd_column* cols, int n_cols, int64_t first_row, int64_t n_rows,
                                struct ArrowDeviceArray* out);

int dfd_metrics_get(dfd_ctx* ctx, dfd_metrics* out);
int dfd_metrics_reset(dfd_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* DFD_B200_H */
