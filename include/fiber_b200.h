/* fiber_b200.h -- C ABI of the B200-native Pool.map engine (libfiber_b200.so).
 *
 * This is the drop-in boundary for the ONE hot path of uber/fiber this repository replaces:
 * Pool.map / starmap / apply_async task scatter + result gather.  The reference is pure Python
 * and has no FFI of its own; each entry point below therefore cites the reference *interface* it
 * stands in for (paths relative to the reference checkout, fiber @ ad6faf02).  A reference
 * maintainer binds them with ctypes exactly as fiber_b200/_abi.py does (see INTEGRATION.md).
 *
 * Conventions: plain pointers and sizes only (no torch / C++ types); every function returns
 * FBR_OK (0) or a negative fbr_status; fbr_last_error() gives the thread-local message.  Blocking
 * calls (fbr_result_wait, fbr_pool_join) do not touch Python and are called with the GIL released.
 * The library never computes a task on the CPU: without a usable CUDA device fbr_pool_create
 * fails with FBR_ENODEV.
 */
#ifndef FIBER_B200_H_
#define FIBER_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FBR_ABI_VERSION 2

typedef enum fbr_status {
    FBR_OK = 0,
    FBR_EINVAL = -1,    /* bad argument */
    FBR_ECUDA = -2,     /* CUDA runtime error (message has the cudaError string) */
    FBR_ENOMEM = -3,
    FBR_ESTATE = -4,    /* pool not in RUN state: the ABI face of ValueError("Pool is not running"),
                           fiber/pool.py:1107-1108,1166-1167,1284-1285 */
    FBR_ETIMEOUT = -5,
    FBR_ETASK = -6,     /* a device body reported a task error (see fbr_result_t.err_*) */
    FBR_ENODEV = -7,    /* no CUDA device: there is no CPU fallback */
    FBR_ENOENT = -8     /* unknown body name / seq */
} fbr_status;

typedef struct fbr_pool fbr_pool_t;

/* ---- library ------------------------------------------------------------------------------ */
int fbr_abi_version(void);
const char* fbr_last_error(void);
/* fiber/context.py:61-62 cpu_count(): the engine's unit of parallel hardware is the GPU. */
int fbr_device_count(int* n);

/* ---- device-body registry -------------------------------------------------------------------
 * The reference ships `func` to workers by pickle reference (fiber/pool.py:961) and calls it at
 * fiber/pool.py:806,809,820.  A Python callable cannot run on a GPU, so callables are bound to a
 * compiled-in device body by name; unbound callables are rejected by the host layer. */
typedef enum fbr_result_kind {
    FBR_RES_BYTES = 0,   /* opaque fixed-size record */
    FBR_RES_BOOL = 1,    /* uint8 0/1  (Python bool) */
    FBR_RES_I64 = 2,     /* int64      (Python int) */
    FBR_RES_U32 = 3,     /* uint32     (Python int) */
    FBR_RES_F64X2 = 4,   /* two float64 (Python tuple of floats) */
    FBR_RES_NONE = 5,    /* body returns None; one pad byte per task */
    FBR_RES_BITS8 = 6    /* one byte = the bool results of 8 consecutive items, bit k (LSB first) = item
                            8*task + k.  A map over N items is submitted as ceil(N/8) tasks: range() indices
                            (arg_stride 0) or 8 argument items per task record (arg_stride = 8 * item size,
                            fbr_map_desc_t.n_items = N so that items past N are never read).  For range()
                            indices the bits past N in the last byte are computed like any other index and
                            are masked by the caller (fiber_b200/pool.py does) */
} fbr_result_kind;

#define FBR_BODY_INDEX_ARG 0x1u   /* body can take the task index itself as its int64 argument */
#define FBR_BODY_NEEDS_SHARED 0x2u /* body reads a shared (broadcast) argument block */
#define FBR_BODY_SUMMABLE 0x4u    /* the dispatch kernel can fold sum(results) (bool/int64/u32; popcount for bits) */
#define FBR_BODY_INDEX_ONLY 0x8u  /* body takes range() arguments only (arg_stride must be 0) */
#define FBR_BODY_RECORD 0x10u     /* record body (FBR_EXPORT_RECORD_BODY): argument and result records of 4..256 bytes,
                                     multiples of 4 (result_kind FBR_RES_BYTES); explicit, 4-byte aligned argument
                                     records only (arg_stride % 4 == 0); not summable, no range() or shared block */

typedef struct fbr_body_info {
    int32_t func_id;
    uint32_t arg_bytes;      /* fixed-layout per-task argument record */
    uint32_t result_bytes;   /* fixed-layout per-task result record */
    uint32_t result_kind;    /* fbr_result_kind */
    uint32_t flags;          /* FBR_BODY_* */
    uint32_t unit_tasks;     /* preferred claim-unit size (tasks per ring slot) */
    char name[40];
} fbr_body_info_t;

int fbr_body_count(int* n);
int fbr_body_info(int func_id, fbr_body_info_t* info);
int fbr_body_lookup(const char* name, int* func_id);

/* Out-of-tree device bodies.  The reference pickles ANY callable into the task tuple
 * (fiber/pool.py:961) and the worker calls it (fiber/pool.py:806,809,820); here the callable's device
 * code may be compiled separately from this library: a shared object built with nvcc for sm_100a from a
 * source that includes include/fiber_b200_body.cuh, defines a ThreadBody struct and exports it with
 * FBR_EXPORT_THREAD_BODY(Body, name, entry) (integer and bool results), or with FBR_EXPORT_RECORD_BODY(Body, name,
 * entry, flags) for any float / struct argument and result records (FBR_BODY_RECORD).  fbr_register_body dlopen()s `module_path`, calls `entry`
 * to obtain the module descriptor below, checks its ABI stamp and appends the body to the table
 * (func_id >= the compiled-in count; the same name may be registered once).  The module's launch routine
 * receives the same wave parameters as the compiled-in kernels, so registered bodies run in the same
 * persistent-CTA dispatch kernels (direct placement, ring + gather_ordered, resilient re-dispatch). */
#define FBR_BODY_MODULE_ABI 1
typedef struct fbr_body_module {
    uint32_t abi;               /* FBR_BODY_MODULE_ABI */
    uint32_t wave_params_bytes; /* sizeof(fbr::WaveParams) the module was compiled against */
    const char* name;
    uint32_t arg_bytes, result_bytes, result_kind, flags, unit_tasks;
    void (*launch)(const void* wave_params, int grid, void* cuda_stream);
    int (*occupancy)(int index_mode);   /* resident CTAs per SM on the current device */
} fbr_body_module_t;
typedef const fbr_body_module_t* (*fbr_body_entry_fn)(void);
int fbr_register_body(const char* name, const char* module_path, const char* entry, int* func_id);

/* ---- pool lifecycle -------------------------------------------------------------------------
 * fbr_pool_create   <- ZPool.__init__ (fiber/pool.py:888-943) + worker start
 *                      (_maintain_workers, fiber/pool.py:1009-1057) + local_backend.create_job
 *                      (fiber/local_backend.py:37-42): one worker == one CUDA device with its
 *                      three streams and its ring set, instead of one subprocess with two sockets.
 * fbr_pool_close    <- ZPool.close      (fiber/pool.py:1337-1353)
 * fbr_pool_terminate<- ZPool.terminate  (fiber/pool.py:1355-1388)
 * fbr_pool_join     <- ZPool.join       (fiber/pool.py:1390-1403); requires close/terminate first
 * fbr_pool_destroy  frees everything (the reference relies on process exit).
 * ring_bytes: size of each device ring arena per worker (result ring, and each half of the
 * argument / ordered-output staging rings); 0 selects the default (256 MiB). */
#define FBR_POOL_TIMING 0x1u  /* bracket every dispatch/gather launch with CUDA events (stats) */
#define FBR_POOL_OVERLAP 0x2u  /* run gather(w) on a second stream concurrently with the next dispatch
                                   (device-resident results only; ring used in halves) */
int fbr_pool_create(int n_workers, const int* device_ids, uint64_t ring_bytes, uint32_t flags,
                    fbr_pool_t** pool);
int fbr_pool_close(fbr_pool_t* pool);
int fbr_pool_terminate(fbr_pool_t* pool);
int fbr_pool_join(fbr_pool_t* pool);
int fbr_pool_destroy(fbr_pool_t* pool);
int fbr_pool_n_workers(fbr_pool_t* pool, int* n);
int fbr_pool_worker_device(fbr_pool_t* pool, int worker, int* device_id);

/* ---- map submission -------------------------------------------------------------------------
 * fbr_map_submit <- ZPool.map_async / starmap_async / apply_async (fiber/pool.py:1139-1184,
 * 1258-1305, 1089-1116) + _handle_tasks (fiber/pool.py:952-963): cut [0,n_tasks) into chunks,
 * write one fixed-layout task record per claim unit into the pinned task ring, cudaMemcpyAsync
 * them (and the argument records) to the worker's device ring, launch the persistent-CTA
 * dispatch kernel and the ordered gather.  Returns immediately with the map's `seq`
 * (Inventory.add, fiber/pool.py:659-664). */
#define FBR_MAP 0x0u            /* 5th task-tuple field False (fiber/pool.py:1181) */
#define FBR_STARMAP 0x1u        /* 5th field True, item = (args,)      (fiber/pool.py:1297-1301) */
#define FBR_APPLY 0x2u          /* 5th field True, item = (args, kwds) (fiber/pool.py:1112-1113) */
#define FBR_KIND_MASK 0x3u
#define FBR_ARGS_DEVICE 0x10u   /* args/shared are device pointers on worker 0; other workers of the pool read
                                   their block through NVLink peer loads inside the dispatch kernel */
#define FBR_OUT_DEVICE 0x20u    /* out is a device pointer on worker 0; other workers' gather kernels store
                                   their units into it through NVLink peer stores */
#define FBR_WANT_SUM 0x40u      /* fold sum(results) into fbr_result_t.sum (FBR_BODY_SUMMABLE) */
#define FBR_SHUFFLE 0x80u       /* permute task records inside each wave (arrival != index order;
                                   exercises placement-by-index, fiber/pool.py:672) */
#define FBR_FULL_WINDOW 0x100u  /* keep the whole ordered output resident on the device until the
                                   map completes (needed when units may be re-dispatched) */
#define FBR_SHARED_HANDLE 0x200u /* `shared` is a handle from fbr_shared_put, not a pointer */
#define FBR_RESULTS_ON_DEVICE 0x800u /* keep the ordered results in an engine-owned device buffer (per
                                   worker block); nothing but the 24-byte control block crosses PCIe
                                   until fbr_result_fetch asks for a range */
#define FBR_VIA_RING 0x1000u    /* always go through task records + result ring + gather_ordered, even for a
                                   contiguous block whose units could be stored at their final index by
                                   the dispatch kernel (direct placement) */
#define FBR_NO_ZERO_COPY 0x2000u /* results are wanted wave by wave (imap): stage and copy them out instead of letting the kernel
                                   store small results straight into the pinned segment */
#define FBR_RESILIENT 0x400u    /* ResilientZPool semantics (fiber/pool.py:1425-1688): a claim unit whose
                                   worker dies (FBR_TASK_FAULT) is re-dispatched until it completes */

typedef struct fbr_map_desc {
    int32_t func_id;
    uint32_t flags;
    uint64_t n_tasks;
    uint32_t chunksize;      /* 0 -> 32 (fiber/pool.py:1169-1170) */
    uint32_t arg_stride;     /* bytes between argument records; 0 -> implicit index arguments */
    const void* args;        /* n_tasks records of arg_stride bytes (host, ideally pinned; or device) */
    int64_t index_start;     /* implicit argument of task i = index_start + i*index_step (range()) */
    int64_t index_step;
    const void* shared;      /* broadcast argument block (e.g. parzen samples), may be NULL */
    uint64_t shared_bytes;
    void* out;               /* NULL: engine-owned pinned result segment; else n_tasks*result_bytes */
    uint64_t task_index_base;/* global index of task 0 (sharded maps: rank's block start) */
    uint64_t shuffle_seed;
    uint64_t n_items;        /* FBR_RES_BITS8 bodies with explicit arguments: number of argument items of the
                                whole map (the last task may cover fewer than 8); 0 = 8 * n_tasks */
    uint32_t attempt;        /* how many times this block of tasks has been dispatched before (a resilient pool that
                                re-queues a dead worker's chunk, fiber/pool.py:1635-1654, passes attempt + 1); bodies
                                see it as their `attempt` argument */
    uint32_t pad;
} fbr_map_desc_t;

int fbr_map_submit(fbr_pool_t* pool, const fbr_map_desc_t* desc, uint64_t* seq);

/* Broadcast argument blocks (initargs / arguments every task shares, e.g. the parzen sample array
 * the reference pickles into each of its 102 task messages, SURVEY.md 3.2): uploaded once to every
 * worker's device, then referenced by handle (desc.shared = (void*)handle + FBR_SHARED_HANDLE). */
int fbr_shared_put(fbr_pool_t* pool, const void* host, uint64_t bytes, uint64_t* handle);
int fbr_shared_drop(fbr_pool_t* pool, uint64_t handle);

/* Host-side planning of a map, without touching a device (pure function of its arguments): the claim
 * unit fbr_map_submit would pick, the resulting ring slot stride, and worker w's task block.  Lets
 * the chunking / alignment rules be checked against the reference's chunk plan
 * (fiber/pool.py:1084-1087) on a machine without a GPU. */
typedef struct fbr_plan {
    uint32_t unit_tasks;      /* tasks per claim unit (ring slot) */
    uint32_t slot_stride;     /* bytes per ring slot (multiple of 16) */
    uint64_t n_units;         /* claim units of the whole map */
    uint64_t block_first;     /* worker's block: first task */
    uint64_t block_count;     /*                 number of tasks */
} fbr_plan_t;
int fbr_plan_query(int func_id, uint64_t n_tasks, uint32_t chunksize, uint64_t ring_bytes, int n_workers,
                   int worker, int sm_count, fbr_plan_t* plan);

/* ---- result collection ----------------------------------------------------------------------
 * fbr_result_wait    <- MapResult.get -> Inventory.get (fiber/pool.py:736-737, 666-679)
 * fbr_result_poll    <- Inventory.iget_ordered / iget_unordered progress (fiber/pool.py:681-728)
 * fbr_result_release <- `self._inventory[job_seq] = None` (fiber/pool.py:677-679) */
typedef struct fbr_result {
    uint64_t seq;
    uint64_t n_tasks;
    uint32_t result_bytes;
    uint32_t result_kind;
    void* data;              /* ordered results: pinned host (or the caller's `out`) */
    int64_t sum;             /* valid with FBR_WANT_SUM: sum(results), wrapped to int64 */
    uint32_t err_code;       /* 0, or fbr_task_error of the lowest failing task */
    uint32_t n_waves;
    uint64_t err_task;       /* index of that task */
    uint64_t sum_lo;         /* the exact sum is sum_hi * 2^32 + sum_lo (Python ints are unbounded: the device */
    int64_t sum_hi;          /* folds the two halves of int64 results separately, so nothing wraps silently) */
    uint32_t sum_overflow;   /* 1: the exact sum does not fit int64, `sum` is its low 64 bits */
    uint32_t pad;
} fbr_result_t;

typedef enum fbr_task_error {
    FBR_TASK_OK = 0,
    FBR_TASK_OVERFLOW = 1,   /* int64 result overflow (Python ints are unbounded: fail loudly) */
    FBR_TASK_BADARG = 2,
    FBR_TASK_FAULT = 3       /* injected fault (resilient-pool tests) */
} fbr_task_error;

int fbr_result_wait(fbr_pool_t* pool, uint64_t seq, int timeout_ms, fbr_result_t* res);
int fbr_result_poll(fbr_pool_t* pool, uint64_t seq, uint64_t* n_done);
/* Address of the map's ordered-result buffer without waiting: tasks [0, n_done) of it are final. */
int fbr_result_data(fbr_pool_t* pool, uint64_t seq, void** data);
/* Copy results [first, first+count) of a FBR_RESULTS_ON_DEVICE map to host memory (blocking). */
int fbr_result_fetch(fbr_pool_t* pool, uint64_t seq, uint64_t first, uint64_t count, void* host_dst);
int fbr_result_release(fbr_pool_t* pool, uint64_t seq);

/* ---- memory helpers ------------------------------------------------------------------------
 * Pinned host segments are the endpoints that replace LazyZConnection sockets
 * (fiber/queues.py:190-249): the host encodes argument records straight into them. */
int fbr_host_alloc(fbr_pool_t* pool, uint64_t bytes, void** ptr);
int fbr_host_free(fbr_pool_t* pool, void* ptr);
int fbr_device_alloc(fbr_pool_t* pool, int worker, uint64_t bytes, void** dptr);
int fbr_device_free(fbr_pool_t* pool, int worker, void* dptr);
int fbr_memcpy_h2d(fbr_pool_t* pool, int worker, void* dptr, const void* src, uint64_t bytes);
int fbr_memcpy_d2h(fbr_pool_t* pool, int worker, void* dst, const void* dptr, uint64_t bytes);
/* Fill device memory with the synthetic 4 KB payload records of tasks [t0, t0+n). */
int fbr_payload_fill_device(fbr_pool_t* pool, int worker, void* dptr, uint64_t t0, uint64_t n);

/* ---- statistics ------------------------------------------------------------------------------
 * ZPool keeps bare counters sent_tasks/recv_tasks (fiber/pool.py:902-903); these extend them. */
typedef struct fbr_stats {
    uint64_t tasks_submitted, tasks_completed;
    uint64_t units_dispatched;          /* task records claimed by persistent CTAs */
    uint64_t dispatch_launches, gather_launches, fill_launches;
    uint64_t h2d_bytes, d2h_bytes;
    double dispatch_ms, gather_ms;      /* summed CUDA-event time (FBR_POOL_TIMING only) */
    uint64_t gather_bytes;              /* algorithmic bytes moved by gather_ordered (read+write) */
    uint64_t dispatch_bytes;            /* algorithmic bytes of the dispatch kernels (args+results) */
    uint64_t units_redispatched;        /* lost units re-queued by resilient maps (pending-table resubmits) */
    uint64_t records_copied;            /* task records written to the pinned ring and copied to the device */
    uint64_t direct_waves;              /* waves whose dispatch kernel stored at the final index (no gather) */
    uint64_t peer_push_bytes;           /* argument bytes pushed from worker 0's memory into other workers' staging by
                                           worker 0's copy engine (root-resident maps over NVLink) */
    uint64_t workers_lost;              /* workers retired because their CUDA context died (sticky error); maps with
                                           FBR_RESILIENT had their blocks re-dispatched to the surviving workers */
} fbr_stats_t;
int fbr_pool_stats(fbr_pool_t* pool, fbr_stats_t* stats);
int fbr_pool_stats_reset(fbr_pool_t* pool);

/* ---- SimpleQueue / Pipe / device Process (fiber/queues.py:262-352, fiber/process.py:83-323) ---------
 * Every endpoint owns one SPSC lane of 64-byte records in pinned, device-mapped memory; a queue's
 * forwarder fair-queues its writer lanes into its reader lanes with strict round-robin (the
 * nn_device of fiber/socket.py:297-320; tests/test_queue.py:218-250 pins 600 of 2400 messages per
 * reader).  An endpoint is the host or a device process: a resident one-warp kernel that runs one
 * of the reference tests' process targets against its lanes. */
typedef struct fbr_queue fbr_queue_t;
typedef struct fbr_lane fbr_lane_t;
typedef struct fbr_process fbr_process_t;

typedef enum fbr_record_tag { FBR_REC_NONE = 0, FBR_REC_INT = 1, FBR_REC_FLOAT = 2, FBR_REC_BYTES = 3, FBR_REC_STR = 4 } fbr_record_tag;
typedef struct fbr_record {      /* fixed-layout message: what the reference pickles (queues.py:164-181) */
    uint32_t tag;                /* fbr_record_tag */
    uint32_t len;                /* payload bytes in use */
    uint8_t payload[56];
} fbr_record_t;

typedef enum fbr_process_kind {
    FBR_PROC_QUEUE_WORKER = 1,   /* worker(q_in, q_out, ident)      tests/test_queue.py:44-50 */
    FBR_PROC_PUT_QUEUE = 2,      /* put_queue(q, data)              tests/test_queue.py:23-33 */
    FBR_PROC_GET_QUEUE = 3,      /* get_queue(q_in, q_out, n)       tests/test_queue.py:36-42 */
    FBR_PROC_WRITE_PIPE = 4,     /* write_pipe(pipe, msg)           tests/test_queue.py:19-20 */
    FBR_PROC_PIPE_WORKER = 5     /* pipe_worker(conn)               tests/test_queue.py:53-57 */
} fbr_process_kind;

const char* fbr_queue_last_error(void);
int fbr_queue_create(fbr_queue_t** q);                                   /* SimpleQueuePush.__init__ / Pipe */
int fbr_queue_open_writer(fbr_queue_t* q, fbr_lane_t** lane);            /* LazyZConnection(("w", addr)) */
int fbr_queue_open_reader(fbr_queue_t* q, fbr_lane_t** lane);            /* LazyZConnection(("r", addr)) */
int fbr_lane_send(fbr_lane_t* lane, const fbr_record_t* rec, int timeout_ms);   /* ZConnection.send */
int fbr_lane_recv(fbr_lane_t* lane, fbr_record_t* rec, int timeout_ms);         /* ZConnection.recv */
int fbr_lane_poll(fbr_lane_t* lane, int* ready);                                 /* ZConnection._poll */
int fbr_queue_put(fbr_queue_t* q, const fbr_record_t* rec, int timeout_ms);     /* SimpleQueuePush.put */
int fbr_queue_get(fbr_queue_t* q, fbr_record_t* rec, int timeout_ms);           /* SimpleQueuePush.get */
int fbr_queue_stats(fbr_queue_t* q, uint64_t* forwarded, uint32_t* n_writers, uint32_t* n_readers);
int fbr_queue_destroy(fbr_queue_t* q);
/* Process.start / is_alive+exitcode / join / terminate (fiber/process.py:187-215, 217-262). */
int fbr_process_start(int device_id, int kind, fbr_lane_t* in, fbr_lane_t* out, int64_t ident,
                      const fbr_record_t* msg, const fbr_record_t* list, uint32_t list_len, int idle_timeout_ms,
                      fbr_process_t** proc);
int fbr_process_poll(fbr_process_t* proc, int* alive, int* exitcode);
int fbr_process_join(fbr_process_t* proc, int timeout_ms);
int fbr_process_terminate(fbr_process_t* proc);
int fbr_process_handled(fbr_process_t* proc, uint64_t* handled);
int fbr_process_destroy(fbr_process_t* proc);

/* ---- express lane: doorbell path for one-task submissions (apply / apply_async) --------------------
 * A resident one-warp kernel per device polls a pinned, device-mapped request lane, runs the body and
 * writes the result record into a pinned response lane the host polls: no kernel launch, copy or
 * event on the round trip (fiber/pool.py:1089-1116 pays a TCP round trip per apply).  The kernel exits
 * after `idle_timeout_us` without requests and is relaunched on demand.  Bodies whose argument and
 * result fit 48 bytes: square_i64, mul2_i64, square_scale_i64, identity_i64, pi_inside_det, sleep_f64. */
typedef struct fbr_express fbr_express_t;
const char* fbr_express_last_error(void);
int fbr_express_create(int device_id, int idle_timeout_us, fbr_express_t** x);
int fbr_express_submit(fbr_express_t* x, int func_id, const void* arg, uint32_t arg_bytes, uint64_t* ticket);
int fbr_express_wait(fbr_express_t* x, uint64_t ticket, void* result, uint32_t* result_bytes, uint32_t* err, int timeout_ms);
int fbr_express_discard(fbr_express_t* x, uint64_t ticket);   /* handle dropped without a wait: forget the response */
int fbr_express_stats(fbr_express_t* x, uint64_t* served, uint64_t* launches, int* resident);
int fbr_express_destroy(fbr_express_t* x);

/* ---- engine-level collectives: one process per GPU (SURVEY.md 8(e); fiber/experimental/ring.py:44-129) ---------
 * The map shards by contiguous task block with no data-path collective; what surrounds it does exchange data:
 * shared arguments that live on one rank (ncclBroadcast), an input array resident on one rank (scatter =
 * grouped ncclSend/ncclRecv: the fan-out of fiber/pool.py:910-914), the ordered result blocks (ncclAllGather, or
 * grouped send/recv to a root: the fan-in of fiber/pool.py:916-920), scalar folds (ncclAllReduce int64) and
 * experimental.Ring's all-reduce (examples/ring.py:81-86).  A communicator is bound to one CUDA device and owns
 * one stream; calls enqueue on it, fbr_comm_sync waits.  The 128-byte bootstrap id (ncclUniqueId) is what a ring
 * node publishes in the member table instead of the reference's ip/port.  NCCL is dlopen()ed on first use. */
typedef struct fbr_comm fbr_comm_t;
#define FBR_COMM_ID_BYTES 128
typedef enum fbr_dtype { FBR_DT_U8 = 0, FBR_DT_I32 = 1, FBR_DT_I64 = 2, FBR_DT_F32 = 3, FBR_DT_F64 = 4 } fbr_dtype;
typedef enum fbr_redop { FBR_OP_SUM = 0, FBR_OP_PROD = 1, FBR_OP_MAX = 2, FBR_OP_MIN = 3 } fbr_redop;
const char* fbr_comm_last_error(void);
int fbr_comm_load(const char* libnccl_path, int* version);          /* optional: pick the NCCL build; reports its version */
int fbr_comm_unique_id(void* id128);                                 /* rank 0: ncclGetUniqueId */
int fbr_comm_create(int device_id, int nranks, int rank, const void* id128, fbr_comm_t** comm);   /* ncclCommInitRank */
int fbr_comm_info(fbr_comm_t* comm, int* rank, int* nranks, int* device_id);
int fbr_comm_sync(fbr_comm_t* comm);
int fbr_comm_broadcast(fbr_comm_t* comm, void* dptr, uint64_t bytes, int root);
int fbr_comm_allgather(fbr_comm_t* comm, const void* send, void* recv, uint64_t bytes_per_rank);
int fbr_comm_gather(fbr_comm_t* comm, const void* send, void* recv_on_root, uint64_t bytes_per_rank, int root);
int fbr_comm_scatter(fbr_comm_t* comm, const void* send_on_root, void* recv, uint64_t bytes_per_rank, int root);
int fbr_comm_allreduce(fbr_comm_t* comm, const void* send, void* recv, uint64_t count, int dtype, int op);
int fbr_comm_allreduce_timed(fbr_comm_t* comm, void* buf, uint64_t count, int dtype, int op, int iters, float* ms_per_call);
int fbr_comm_allreduce_i64(fbr_comm_t* comm, int64_t* value);       /* host scalar in, global sum out (the pi count) */
int fbr_comm_allreduce_i64_begin(fbr_comm_t* comm, int64_t value);  /* the same, split: enqueue now ...               */
int fbr_comm_allreduce_i64_end(fbr_comm_t* comm, int64_t* sum);     /* ... collect later (overlaps the next map)      */
int fbr_comm_device_alloc(fbr_comm_t* comm, uint64_t bytes, void** dptr);
int fbr_comm_device_free(fbr_comm_t* comm, void* dptr);
int fbr_comm_memcpy_h2d(fbr_comm_t* comm, void* dptr, const void* src, uint64_t bytes);
int fbr_comm_memcpy_d2h(fbr_comm_t* comm, void* dst, const void* dptr, uint64_t bytes);
int fbr_comm_destroy(fbr_comm_t* comm);

#ifdef __cplusplus
}
#endif
#endif /* FIBER_B200_H_ */
