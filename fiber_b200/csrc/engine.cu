// engine.cu -- host side of libfiber_b200.so: pool object, per-GPU workers, rings, wave pipeline,
// and the extern "C" entry points declared in include/fiber_b200.h.
//
// One worker == one CUDA device (the GPU analogue of one job-backed worker process,
// fiber/pool.py:1009-1057 + fiber/local_backend.py:37-42) with
//   * three streams: copy-in (task records + arguments), compute (dispatch + gather), copy-out;
//   * a pinned host task ring and its device mirror (fixed-layout TaskRecord, cudaMemcpyAsync);
//   * a device result ring (payload arena + one SlotHeader per claim unit);
//   * double-buffered device staging for host-resident arguments and ordered output.
// A map is cut into waves that fit the rings; wave w+1's copy-in and wave w-1's copy-out overlap
// wave w's kernels.  No host thread is needed: ordering is carried by stream events, completion
// by events the caller waits on (fbr_result_wait / fbr_result_poll).
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/mman.h>
#include <sys/syscall.h>
#include <unistd.h>

#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <deque>
#include <memory>
#include <mutex>
#include <numeric>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "../../include/fiber_b200.h"
#include "kernels.cuh"

using namespace fbr;

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local std::string g_err;

static int fail(int code, const char* fmt, ...);
const std::string& last_error_of_this_thread();
static int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}
const std::string& last_error_of_this_thread() { return g_err; }
#define CK(call)                                                                                  \
    do {                                                                                          \
        cudaError_t e_ = (call);                                                                  \
        if (e_ != cudaSuccess)                                                                    \
            return fail(FBR_ECUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

struct SubmitThread;
void SubmitThread_loop_impl(SubmitThread* t);
// One host thread per worker for submissions: the CUDA calls of different devices (stream waits, launches,
// async copies, event records: ~50 us per part of 8 waves) run side by side instead of one after the other,
// which is what an 8-GPU in-process pool needs to keep up with 0.25 ms kernels.
struct SubmitThread {
    std::mutex mu;
    std::condition_variable cv;
    std::function<int()> job;
    bool pending = false, finished = false, quit = false;
    int rc = 0;
    std::string err;
    std::thread th;             // declared LAST: it starts running in the constructor and uses every member above
    SubmitThread() : th([this] { loop(); }) {}
    ~SubmitThread() {
        { std::lock_guard<std::mutex> g(mu); quit = true; }
        cv.notify_all();
        if (th.joinable()) th.join();
    }
    void loop() { SubmitThread_loop_impl(this); }
    void post(std::function<int()> f) {
        { std::lock_guard<std::mutex> g(mu); job = std::move(f); pending = true; finished = false; }
        cv.notify_all();
    }
    int wait(std::string* msg) {
        std::unique_lock<std::mutex> g(mu);
        cv.wait(g, [this] { return finished; });
        if (msg) *msg = err;
        return rc;
    }
};

// ------------------------------------------------------------------------------------------------
// body table: the compiled-in bodies plus bodies registered at run time from separately compiled
// modules (fbr_register_body).  The reference ships ANY callable to its workers (fiber/pool.py:961,
// executed at :806,809,820); here a callable's device body may live outside this library.
// ------------------------------------------------------------------------------------------------
typedef void (*launch_fn)(const void* wave_params, int grid, void* stream);
typedef int (*occupancy_fn)(int index_mode);

template <class B>
static void launch_thread(const void* wpv, int grid, void* sv) {
    const WaveParams& wp = *(const WaveParams*)wpv;
    cudaStream_t s = (cudaStream_t)sv;
    if constexpr (B::kIndexArg) {
        if (wp.arg_stride == 0) {
            dispatch_thread_kernel<B, true><<<grid, kThreads, 0, s>>>(wp);
            return;
        }
    }
    dispatch_thread_kernel<B, false><<<grid, kThreads, 0, s>>>(wp);
}
static int occ_of(const void* kernel) {
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, kThreads, 0) != cudaSuccess) { cudaGetLastError(); return 1; }
    return occ > 0 ? occ : 1;
}
template <class B>
static int occ_thread(int index_mode) {
    if constexpr (B::kIndexArg) {
        if (index_mode) return occ_of((const void*)dispatch_thread_kernel<B, true>);
    }
    return occ_of((const void*)dispatch_thread_kernel<B, false>);
}
static void launch_payload_map(const void* wpv, int grid, void* sv) {
    const WaveParams& wp = *(const WaveParams*)wpv;
    cudaStream_t s = (cudaStream_t)sv;
    // contiguous records: TMA-staged, warp-specialised kernel (2 CTAs of 5 warps per SM; a 6+3-stage variant at 1 CTA/SM
    // was no faster, DESIGN.md section 6); strided records (arg_stride > 4096) keep the register-streaming kernel
    if (wp.arg_stride == kPayloadBytes) {
        int sm = 148, dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, dev);
        const int g = (int)std::min<uint32_t>(wp.n_units, (uint32_t)(sm * 2));
        dispatch_payload_map_tma_kernel<3, 2><<<g, 160, tma_map::kSmemBytes, s>>>(wp);
        return;
    }
    dispatch_payload_map_kernel<<<grid, kThreads, 0, s>>>(wp);
}
static int occ_payload_map(int) {
    cudaFuncSetAttribute(dispatch_payload_map_tma_kernel<3, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tma_map::kSmemBytes);
    cudaFuncAttributes at;
    cudaFuncGetAttributes(&at, (const void*)dispatch_payload_map_tma_kernel<3, 2>);   // force-load
    return occ_of((const void*)dispatch_payload_map_kernel);
}
static void launch_payload_checksum(const void* wpv, int grid, void* sv) {
    dispatch_payload_checksum_kernel<<<grid, kThreads, 0, (cudaStream_t)sv>>>(*(const WaveParams*)wpv);
}
static int occ_payload_checksum(int) { return occ_of((const void*)dispatch_payload_checksum_kernel); }
// bit-packed twin of a bool body: range() indices through the body's own 16-index vector routine,
// explicit argument items through the generic ballot kernel
static void launch_pi_bits(const void* wpv, int grid, void* sv) {
    const WaveParams& wp = *(const WaveParams*)wpv;
    if (wp.arg_stride == 0) dispatch_pi_bits_kernel<<<grid, kThreads, 0, (cudaStream_t)sv>>>(wp);
    else dispatch_bits_items_kernel<PiInsideDet><<<grid, kThreads, 0, (cudaStream_t)sv>>>(wp);
}
static int occ_pi_bits(int index_mode) {
    return index_mode ? occ_of((const void*)dispatch_pi_bits_kernel) : occ_of((const void*)dispatch_bits_items_kernel<PiInsideDet>);
}
template <typename T>
static void launch_parzen(const void* wpv, int grid, void* sv) {
    dispatch_parzen_kernel<T><<<grid, kThreads, 0, (cudaStream_t)sv>>>(*(const WaveParams*)wpv);
}
template <typename T>
static int occ_parzen(int) { return occ_of((const void*)dispatch_parzen_kernel<T>); }

struct BodyEntry {
    std::string name;
    uint32_t arg_bytes = 0, result_bytes = 0, result_kind = 0, flags = 0, unit_tasks = 0;
    launch_fn launch = nullptr;
    occupancy_fn occupancy = nullptr;
    int max_ctas_per_sm = 0;   // 0 = as many as fit; streaming read+write bodies run best with few, fat streams
    void* module = nullptr;    // dlopen handle of a registered body (never closed: kernels may be in flight)
};

static std::mutex g_body_mu;
static std::deque<BodyEntry> g_bodies;   // append-only: references stay valid, func_id = position

static void builtin_bodies_once() {
    // caller holds g_body_mu
    if (!g_bodies.empty()) return;
    auto add = [](const char* name, uint32_t ab, uint32_t rb, uint32_t kind, uint32_t flags, uint32_t unit, launch_fn l,
                  occupancy_fn o, int max_ctas) {
        BodyEntry b;
        b.name = name; b.arg_bytes = ab; b.result_bytes = rb; b.result_kind = kind; b.flags = flags; b.unit_tasks = unit;
        b.launch = l; b.occupancy = o; b.max_ctas_per_sm = max_ctas;
        g_bodies.push_back(b);
    };
    // order == enum FuncId (bodies.cuh)
    add("square_i64", 8, 8, FBR_RES_I64, FBR_BODY_INDEX_ARG | FBR_BODY_SUMMABLE, 4096, launch_thread<SquareI64>, occ_thread<SquareI64>, 0);
    add("mul2_i64", 16, 8, FBR_RES_I64, FBR_BODY_SUMMABLE, 4096, launch_thread<Mul2I64>, occ_thread<Mul2I64>, 0);
    add("square_scale_i64", 16, 8, FBR_RES_I64, FBR_BODY_SUMMABLE, 4096, launch_thread<SquareScaleI64>, occ_thread<SquareScaleI64>, 0);
    add("identity_i64", 8, 8, FBR_RES_I64, FBR_BODY_INDEX_ARG | FBR_BODY_SUMMABLE, 4096, launch_thread<IdentityI64>, occ_thread<IdentityI64>, 0);
    add("pi_inside_det", 8, 1, FBR_RES_BOOL, FBR_BODY_INDEX_ARG | FBR_BODY_SUMMABLE, 4096, launch_thread<PiInsideDet>, occ_thread<PiInsideDet>, 0);
    add("parzen_f32", 8, 16, FBR_RES_F64X2, FBR_BODY_NEEDS_SHARED, 1, launch_parzen<float>, occ_parzen<float>, 0);
    add("parzen_f64", 8, 16, FBR_RES_F64X2, FBR_BODY_NEEDS_SHARED, 1, launch_parzen<double>, occ_parzen<double>, 0);
    add("payload_map_4k", 4096, 4096, FBR_RES_BYTES, 0, 32, launch_payload_map, occ_payload_map,
        3 /* measured: 3 CTAs/SM = 6641 GB/s, 8 CTAs/SM = 6296 GB/s on the 8.2 GB wave */);
    add("payload_checksum_4k", 4096, 4, FBR_RES_U32, FBR_BODY_SUMMABLE, 256, launch_payload_checksum, occ_payload_checksum, 0);
    add("sleep_f64", 8, 1, FBR_RES_NONE, 0, 1, launch_thread<SleepF64>, occ_thread<SleepF64>, 0);
    add("fault_identity_i64", 8, 8, FBR_RES_I64, FBR_BODY_INDEX_ARG | FBR_BODY_SUMMABLE, 2, launch_thread<FaultIdentityI64>, occ_thread<FaultIdentityI64>, 0);
    // a byte-task = 8 items: 8 range() indices (arg_stride 0) or 8 int64 argument items (arg_stride 64)
    add("pi_inside_bits8", 64, 1, FBR_RES_BITS8, FBR_BODY_INDEX_ARG | FBR_BODY_SUMMABLE, 512, launch_pi_bits, occ_pi_bits, 0);
    add("trap_identity_i64", 8, 8, FBR_RES_I64, FBR_BODY_INDEX_ARG | FBR_BODY_SUMMABLE, 4096, launch_thread<TrapIdentityI64>, occ_thread<TrapIdentityI64>, 0);
}
static int body_count() {
    std::lock_guard<std::mutex> g(g_body_mu);
    builtin_bodies_once();
    return (int)g_bodies.size();
}
// nullptr if func_id is out of range
static const BodyEntry* body_of(int func_id) {
    std::lock_guard<std::mutex> g(g_body_mu);
    builtin_bodies_once();
    if (func_id < 0 || func_id >= (int)g_bodies.size()) return nullptr;
    return &g_bodies[func_id];
}

// ------------------------------------------------------------------------------------------------
// pool structures
// ------------------------------------------------------------------------------------------------
enum { ST_RUN = 0, ST_CLOSE = 1, ST_TERMINATE = 2 };
constexpr int kRecWindows = 4;         // task-ring windows in flight
constexpr uint32_t kRecCapacity = 65536;  // claim units per wave
constexpr int kCtrlSlots = 65536;      // maps in flight (submitted, not yet released) per worker
constexpr int kTickets = 64;

struct SeqCtrl {              // per (seq, worker) control block, device + pinned mirror
    long long sum;            // 8-byte results: sum of the low 32-bit halves; other kinds: the sum itself
    unsigned long long err;   // (task_index << 8 | code), ~0 = none
    uint32_t lost_count;
    uint32_t pad;
    long long sum_hi;         // 8-byte results: sum of the high halves (exact total = sum_hi * 2^32 + sum)
};
static_assert(sizeof(SeqCtrl) == 32, "");

struct Worker {
    int device = -1;
    bool dead = false;                     // the device's CUDA context took a sticky error: the worker process is gone
    int death_error = 0;                   // cudaError_t that killed it
    int numa_node = -1;                    // host NUMA node the GPU hangs off (-1 unknown)
    int sm_count = 0;
    cudaStream_t s_in = nullptr, s_comp = nullptr, s_out = nullptr;
    cudaStream_t s_gath = nullptr;         // higher-priority stream for gathers that overlap the next dispatch
    bool prev_wave_overlap = false;        // the previous wave used only its half of the ring
    cudaStream_t s_push = nullptr;         // a stream of the ROOT worker's device: its copy engine pushes this worker's argument waves
    cudaStream_t s_push2 = nullptr;        // (waves alternate between the two, like the copy-outs)
    cudaEvent_t ev_push[kRecWindows] = {}; // ... and these (root-device) events say when a pushed wave has landed
    int push_root_device = -1;
    uint32_t gath_hist = 0;                // bit k: wave wno-1-k ran its gather on s_gath (its ev_comp is not ordered by s_comp)
    TaskRecord* h_records = nullptr;   // pinned task ring: kRecWindows x kRecCapacity
    TaskRecord* d_records = nullptr;   // device mirror
    SlotHeader* d_headers = nullptr;   // kRecCapacity
    uint8_t* d_ring = nullptr;         // result ring arena (ring_bytes)
    uint8_t* d_args[2] = {nullptr, nullptr};
    uint8_t* d_out[2] = {nullptr, nullptr};
    uint32_t* d_tickets = nullptr;
    SeqCtrl* d_ctrl = nullptr;
    SeqCtrl* h_ctrl = nullptr;         // pinned: [0,kCtrlSlots) results, [kCtrlSlots] init pattern
    cudaEvent_t ev_rec_h2d[kRecWindows];   // window's H2D finished (host may rewrite the pinned window)
    cudaEvent_t ev_comp[kRecWindows];      // wave's kernels finished (device window / arg half reusable)
    cudaEvent_t ev_disp[kRecWindows];      // wave's dispatch kernel finished (its gather may start)
    cudaEvent_t ev_out[2];                 // out half's D2H finished
    uint64_t wave_no = 0;
    std::vector<int> occ, occ_index;   // per func_id: resident CTAs/SM of the explicit-argument / range() instantiation (0 = not asked yet)
    int occ_gather = 1, occ_fill = 1, occ_gather_rows = 1;
    std::vector<int> ctrl_free;        // free-list of control-block slots
};

// resident CTAs per SM of body `func_id` on this worker's device (current device must be w.device)
static int worker_occ(Worker& w, int func_id, const BodyEntry& body, bool index_mode) {
    std::vector<int>& v = index_mode ? w.occ_index : w.occ;
    if ((int)v.size() <= func_id) v.resize(func_id + 1, 0);
    if (v[func_id] == 0) v[func_id] = std::max(1, body.occupancy(index_mode ? 1 : 0));
    return v[func_id];
}

struct TimedPair { cudaEvent_t a, b; };

struct PartPlan {                         // how one worker's block of one map runs (plan_part)
    uint32_t unit = 0, slot_stride = 0, R = 0, sum_kind = 0;
    bool args_dev = false, out_dev = false, full_window = false, host_args = false, resilient = false, keep_on_device = false;
    bool overlap = false;                 // gather(w) on s_gath concurrently with dispatch(w+1); ring used in halves
    bool zero_copy = false;               // small host-resident results: the dispatch kernel stores them straight into the pinned
                                          // result segment over PCIe (no staging, no D2H copy, one wave)
    bool peer_out = false;                // the ordered output lives on worker 0 (another GPU): results are computed into the local
                                          // out-staging halves and PUSHED there by this worker's copy engine (the D2H machinery)
    bool peer_push = false;               // arguments live on worker 0 (another GPU): worker 0's copy engine PUSHES each wave's
                                          // records into this worker's staging halves over NVLink (host_args machinery)
    bool direct = false;                  // contiguous, unshuffled, non-resilient block: the dispatch kernel stores every
                                          // unit at its final index (no ring, no task records, no gather launch)
    uint64_t wave_tasks_cap = 0;          // tasks per wave: every wave but the last has exactly this many
    uint64_t args_limit_bytes = 0;        // host arguments end here (n_items records); 0 = n_tasks * arg_stride
};

struct PartCtx : PartPlan {               // ... and the memory submit_part acquired for it
    const uint8_t* d_shared = nullptr;
    uint8_t* window_base = nullptr;       // device output of a FULL_WINDOW part
    const uint8_t* args_full = nullptr;   // device-resident arguments of the whole map (args_dev / resilient)
};

struct SeqPart {
    int worker = 0;
    uint64_t first = 0, count = 0;        // task block of this worker inside the map
    int ctrl_slot = -1;
    cudaEvent_t done = nullptr;
    std::vector<cudaEvent_t> wave_done;
    std::vector<uint64_t> wave_cum;       // tasks finished once wave i is done
    std::vector<TimedPair> t_dispatch, t_gather;
    void* d_shared_tmp = nullptr;         // per-seq device copy of a host shared block
    void* d_window = nullptr;             // FULL_WINDOW device output
    void* d_args_full = nullptr;          // resilient: device copy of all argument records
    LostUnit* d_lost = nullptr;           // resilient: units whose worker "died" (filled by gather)
    LostUnit* h_lost = nullptr;           // pinned mirror
    uint32_t lost_cap = 0, attempt = 0;
    bool finalized = false;               // resilient: window copied back to the host
    bool first_wave_pending = true;       // the block's first wave must wait for what submit_part put on s_in
    PartCtx cx;
};

struct SeqState {
    uint64_t seq = 0, n_tasks = 0;
    int func_id = 0;
    uint32_t flags = 0, result_bytes = 0, result_kind = 0;
    void* out = nullptr;
    bool own_out = false;
    bool finished = false;
    int64_t sum = 0;              // total wrapped to int64 ...
    uint64_t sum_lo = 0;          // ... and its exact form: sum_hi * 2^32 + sum_lo
    int64_t sum_hi = 0;
    bool sum_overflow = false;    // the exact total does not fit int64
    uint32_t err_code = 0;
    uint64_t err_task = 0;
    uint32_t n_waves = 0;
    uint32_t redispatched_units = 0;
    fbr_map_desc_t desc;
    std::vector<SeqPart> parts;
    std::vector<SeqPart> graveyard;        // parts that were running on a worker when it died (their blocks were re-dispatched)
    int waiters = 0;                       // threads inside fbr_result_wait for this seq (they hold event handles outside the lock)
    bool release_pending = false;          // fbr_result_release arrived while they were waiting: the last one out frees the seq
    int dead_worker = -1;                  // a worker died under this map and the map could not be re-dispatched
    int dead_error = 0;
};

struct SharedBlock {
    uint64_t bytes = 0;
    std::vector<void*> d_ptr;  // per worker
};

struct fbr_pool {
    std::mutex mu;
    int state = ST_RUN;
    uint32_t flags = 0;
    uint64_t ring_bytes = 0;
    bool peer_ok = false;             // every worker can load/store every other worker's memory (NVLink P2P)
    bool peer_checked = false;        // ... decided (and enabled) by the first map with device-resident args / output
    std::vector<Worker> workers;
    uint64_t next_seq = 0;
    std::unordered_map<uint64_t, std::unique_ptr<SeqState>> seqs;
    std::unordered_map<uint64_t, SharedBlock> shared;
    uint64_t next_shared = 1;
    std::vector<std::unique_ptr<SubmitThread>> submitters;   // per worker, started with the first multi-worker map
    // pinned host segment cache (size class -> free blocks), and live blocks -> class
    std::unordered_map<uint64_t, std::vector<void*>> pin_free;
    std::unordered_map<void*, uint64_t> pin_live;
    uint64_t pin_cached_bytes = 0;    // bytes sitting in pin_free (bounded by kPinCacheCap)
    // NUMA-split result segments of multi-worker maps: exact byte size -> free blocks; live -> mapped bytes
    std::unordered_map<uint64_t, std::vector<void*>> numa_free;
    std::unordered_map<void*, std::pair<uint64_t, uint64_t>> numa_live;   // ptr -> (key bytes, mapped bytes)
    fbr_stats_t stats;
};

// ------------------------------------------------------------------------------------------------
// helpers
// ------------------------------------------------------------------------------------------------
// the parts of a multi-worker map are submitted from one host thread per worker: counters are added atomically
#define STAT_ADD(p, field, v) __atomic_fetch_add(&(p)->stats.field, (uint64_t)(v), __ATOMIC_RELAXED)

void SubmitThread_loop_impl(SubmitThread* t) {
    std::unique_lock<std::mutex> g(t->mu);
    for (;;) {
        t->cv.wait(g, [t] { return t->pending || t->quit; });
        if (t->quit) return;
        std::function<int()> f = std::move(t->job);
        t->pending = false;
        g.unlock();
        const int rc = f();
        const std::string msg = rc != FBR_OK ? last_error_of_this_thread() : std::string();
        g.lock();
        t->rc = rc;
        t->err = msg;
        t->finished = true;
        t->cv.notify_all();
    }
}

static uint64_t round_up(uint64_t x, uint64_t m) { return (x + m - 1) / m * m; }

// ring arena size of a pool created with `ring_bytes` (0: the default, 256 MiB)
static uint64_t pool_ring_bytes(uint64_t ring_bytes) { return round_up(ring_bytes ? ring_bytes : (256ull << 20), 4096); }

static uint64_t pin_class(uint64_t bytes) {
    uint64_t c = 4096;
    while (c < bytes) c <<= 1;
    return c;
}

constexpr uint64_t kPinCacheCap = 24ull << 30;   // keep at most this much idle pinned memory per pool

static int pinned_acquire(fbr_pool* p, uint64_t bytes, void** out) {
    const uint64_t c = pin_class(bytes ? bytes : 1);
    auto& fl = p->pin_free[c];
    void* ptr = nullptr;
    if (!fl.empty()) {
        ptr = fl.back();
        fl.pop_back();
        p->pin_cached_bytes -= c;
    } else {
        CK(cudaHostAlloc(&ptr, c, cudaHostAllocPortable));
    }
    p->pin_live[ptr] = c;
    *out = ptr;
    return FBR_OK;
}

static void pinned_release(fbr_pool* p, void* ptr) {
    auto it = p->pin_live.find(ptr);
    if (it == p->pin_live.end()) return;
    const uint64_t c = it->second;
    p->pin_live.erase(it);
    if (p->pin_cached_bytes + c > kPinCacheCap) {
        cudaFreeHost(ptr);            // cache full: give the pages back
        return;
    }
    p->pin_free[c].push_back(ptr);
    p->pin_cached_bytes += c;
}

// ---- NUMA-split pinned segments ------------------------------------------------------------------
// One process driving several GPUs writes one ordered result segment; with a plain cudaHostAlloc the
// whole segment sits on the allocating thread's NUMA node and half of the GPUs push their D2H
// stream across the socket link (measured: 95 GB/s aggregate for 8 GPUs vs ~216 GB/s when every
// block is socket-local).  Here each worker's block of the segment is bound (mbind) to the node its
// GPU hangs off before the pages are faulted in by cudaHostRegister.
static int numa_node_of_device(int device) {
    char bdf[32] = {0};
    if (cudaDeviceGetPCIBusId(bdf, sizeof bdf, device) != cudaSuccess) { cudaGetLastError(); return -1; }
    for (char* c = bdf; *c; ++c) if (*c >= 'A' && *c <= 'F') *c = (char)(*c - 'A' + 'a');
    char path[128];
    snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", bdf);
    FILE* f = fopen(path, "r");
    if (!f) return -1;
    int node = -1;
    if (fscanf(f, "%d", &node) != 1) node = -1;
    fclose(f);
    return node;
}

static void bind_range_to_node(void* addr, uint64_t len, int node) {
    if (node < 0 || node >= 64 || len == 0) return;
    unsigned long mask = 1ul << node;
    // MPOL_BIND = 2; failure (no NUMA, no permission) only costs locality
    syscall(SYS_mbind, addr, (unsigned long)len, 2, &mask, 65ul, 0u);
}

struct NumaBlock { uint64_t off, len; int node; };

static int numa_pinned_acquire(fbr_pool* p, uint64_t bytes, const std::vector<NumaBlock>& blocks, void** out) {
    auto& fl = p->numa_free[bytes];
    if (!fl.empty()) {
        void* ptr = fl.back();
        fl.pop_back();
        p->numa_live[ptr].first = bytes;
        *out = ptr;
        return FBR_OK;
    }
    const uint64_t page = 1ull << 21;
    const uint64_t mapped = round_up(std::max<uint64_t>(bytes, 1), page);
    void* ptr = mmap(nullptr, mapped, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
    if (ptr == MAP_FAILED) return fail(FBR_ENOMEM, "mmap of %llu bytes failed", (unsigned long long)mapped);
    const uint64_t small = 4096;
    for (const NumaBlock& b : blocks) {
        const uint64_t lo = b.off / small * small, hi = std::min(mapped, round_up(b.off + b.len, small));
        bind_range_to_node((uint8_t*)ptr + lo, hi - lo, b.node);
    }
    cudaError_t e = cudaHostRegister(ptr, mapped, cudaHostRegisterPortable | cudaHostRegisterMapped);
    if (e != cudaSuccess) {
        munmap(ptr, mapped);
        return fail(FBR_ECUDA, "cudaHostRegister failed: %s", cudaGetErrorString(e));
    }
    p->numa_live[ptr] = {bytes, mapped};
    *out = ptr;
    return FBR_OK;
}

static bool numa_pinned_release(fbr_pool* p, void* ptr) {
    auto it = p->numa_live.find(ptr);
    if (it == p->numa_live.end()) return false;
    p->numa_free[it->second.first].push_back(ptr);
    return true;
}

static int worker_init(fbr_pool* p, Worker& w, int device) {
    w.device = device;
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail(FBR_ENODEV, "device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor);
    w.sm_count = prop.multiProcessorCount;
    w.numa_node = numa_node_of_device(device);
    {
        // stream-ordered allocations (per-map windows, shared blocks) come from the device's default pool: keep what is
        // freed cached instead of handing it back to the driver at every synchronisation (the default threshold is 0;
        // with 8 ranks on one box a 100 MB cudaMallocAsync/cudaFreeAsync pair per map then costs a millisecond)
        cudaMemPool_t mp = nullptr;
        if (cudaDeviceGetDefaultMemPool(&mp, device) == cudaSuccess) {
            uint64_t keep = ~0ull;
            cudaMemPoolSetAttribute(mp, cudaMemPoolAttrReleaseThreshold, &keep);
        }
        cudaGetLastError();
    }
    CK(cudaStreamCreateWithFlags(&w.s_in, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&w.s_comp, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&w.s_out, cudaStreamNonBlocking));
    {
        int lo_prio = 0, hi_prio = 0;
        CK(cudaDeviceGetStreamPriorityRange(&lo_prio, &hi_prio));
        CK(cudaStreamCreateWithPriority(&w.s_gath, cudaStreamNonBlocking, hi_prio));
    }
    CK(cudaHostAlloc((void**)&w.h_records, sizeof(TaskRecord) * kRecCapacity * kRecWindows, cudaHostAllocPortable));
    CK(cudaMalloc((void**)&w.d_records, sizeof(TaskRecord) * kRecCapacity * kRecWindows));
    CK(cudaMalloc((void**)&w.d_headers, sizeof(SlotHeader) * kRecCapacity * 2));   // two halves (overlapped waves)
    CK(cudaMalloc((void**)&w.d_ring, p->ring_bytes));
    CK(cudaMalloc((void**)&w.d_tickets, sizeof(uint32_t) * kTickets * 2));
    CK(cudaMemsetAsync(w.d_tickets, 0, sizeof(uint32_t) * kTickets * 2, w.s_comp));
    CK(cudaMalloc((void**)&w.d_ctrl, sizeof(SeqCtrl) * kCtrlSlots));
    CK(cudaHostAlloc((void**)&w.h_ctrl, sizeof(SeqCtrl) * (kCtrlSlots + 1), cudaHostAllocPortable));
    w.h_ctrl[kCtrlSlots] = SeqCtrl{0, ~0ull, 0u, 0u, 0};
    w.ctrl_free.resize(kCtrlSlots);
    for (int i = 0; i < kCtrlSlots; ++i) w.ctrl_free[i] = kCtrlSlots - 1 - i;
    for (int i = 0; i < kRecWindows; ++i) {
        CK(cudaEventCreateWithFlags(&w.ev_rec_h2d[i], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&w.ev_comp[i], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&w.ev_disp[i], cudaEventDisableTiming));
    }
    for (int i = 0; i < 2; ++i) CK(cudaEventCreateWithFlags(&w.ev_out[i], cudaEventDisableTiming));
    // occupancy of every body known now (also force-loads their kernels: a lazy module load would
    // synchronise with resident device processes, queues.cu); bodies registered later are asked on first use
    for (int f = 0, n = body_count(); f < n; ++f) {
        const BodyEntry& b = *body_of(f);
        worker_occ(w, f, b, false);
        if (b.flags & FBR_BODY_INDEX_ARG) worker_occ(w, f, b, true);
    }
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&w.occ_gather, (const void*)gather_ordered_kernel, kThreads, 0));
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&w.occ_fill, (const void*)payload_fill_kernel, kThreads, 0));
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&w.occ_gather_rows, (const void*)gather_rows_kernel, kThreads, 0));
    if (w.occ_gather_rows < 1) w.occ_gather_rows = 1;
    CK(cudaFuncSetAttribute(gather_bulk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bulk::kStages * bulk::kChunk)));
    if (w.occ_gather < 1) w.occ_gather = 1;
    if (w.occ_fill < 1) w.occ_fill = 1;
    // no cudaDeviceSynchronize here: it would wait for resident device processes (queues.cu)
    CK(cudaStreamSynchronize(w.s_comp));
    return FBR_OK;
}

static void worker_destroy(Worker& w) {
    if (w.device < 0) return;
    if (w.dead) {                          // a corrupted context: every call on it fails; its memory goes with the process
        cudaGetLastError();
        w.device = -1;
        return;
    }
    cudaSetDevice(w.device);
    if (w.s_in) cudaStreamSynchronize(w.s_in);
    if (w.s_comp) cudaStreamSynchronize(w.s_comp);
    if (w.s_out) cudaStreamSynchronize(w.s_out);
    if (w.s_gath) { cudaStreamSynchronize(w.s_gath); cudaStreamDestroy(w.s_gath); }
    if (w.s_push) {                        // lives on the root worker's device
        cudaSetDevice(w.push_root_device);
        cudaStreamSynchronize(w.s_push);
        cudaStreamDestroy(w.s_push);
        if (w.s_push2) { cudaStreamSynchronize(w.s_push2); cudaStreamDestroy(w.s_push2); }
        for (int i = 0; i < kRecWindows; ++i) cudaEventDestroy(w.ev_push[i]);
        cudaGetLastError();
        cudaSetDevice(w.device);
        w.s_push = nullptr;
    }
    if (w.s_in) cudaStreamDestroy(w.s_in);
    if (w.s_comp) cudaStreamDestroy(w.s_comp);
    if (w.s_out) cudaStreamDestroy(w.s_out);
    cudaFreeHost(w.h_records);
    cudaFree(w.d_records);
    cudaFree(w.d_headers);
    cudaFree(w.d_ring);
    for (int i = 0; i < 2; ++i) {
        cudaFree(w.d_args[i]);
        cudaFree(w.d_out[i]);
    }
    cudaFree(w.d_tickets);
    cudaFree(w.d_ctrl);
    cudaFreeHost(w.h_ctrl);
    for (int i = 0; i < kRecWindows; ++i) {
        cudaEventDestroy(w.ev_rec_h2d[i]);
        cudaEventDestroy(w.ev_comp[i]);
        cudaEventDestroy(w.ev_disp[i]);
    }
    for (int i = 0; i < 2; ++i) cudaEventDestroy(w.ev_out[i]);
    w.device = -1;
}

// Claim-unit size: near the body's preferred size, a multiple of the API chunksize when the chunk
// is smaller (so chunk boundaries coincide with unit boundaries), and a multiple of 16/gcd(R, 16) tasks so
// every full slot is 16 B aligned on both sides of the gather (R = 12: units of 4k tasks).  `chunksize` 0 stands for
// the default, 32.
static uint32_t pick_unit(const BodyEntry& b, uint32_t chunksize, uint64_t n_tasks, int sm_count, uint64_t ring_bytes) {
    uint32_t pref = b.unit_tasks;
    if (pref == 1) return 1;
    if (chunksize == 0) chunksize = 32;
    // a unit's results (and its argument records) must fit the ring arenas
    const uint64_t per_task = std::max<uint64_t>(std::max(b.result_bytes, b.arg_bytes), 1);
    while (pref > 1 && (uint64_t)pref * per_task > ring_bytes / 2) pref >>= 1;
    // small maps: shrink the unit so the work still spreads over the SMs
    while (pref > 256 && (uint64_t)pref * (uint64_t)sm_count > n_tasks) pref >>= 1;
    const uint32_t align = 16u / std::gcd(b.result_bytes, 16u);
    uint32_t unit = pref;
    if (chunksize <= pref) {
        uint32_t m = chunksize;  // lcm(chunksize, align)
        while (m % align) m += chunksize;
        if (m <= 2 * pref) unit = std::max(m, pref / m * m);
    }
    unit = (uint32_t)round_up(unit, align);
    while (unit > align && (uint64_t)unit * per_task > ring_bytes) unit -= align;   // chunk-aligned unit too big for the ring
    return unit;
}

// Tasks [*b0, *b1) of block `i` when `count` tasks are cut into `nw` contiguous blocks on the boundaries of the
// map-level claim unit (block partition == PUSH round-robin with chunk = block, SURVEY.md 8(e)); empty if *b1 <= *b0.
static void block_range(const BodyEntry& body, uint32_t chunksize, uint64_t count, int nw, int i, int sm_count,
                        uint64_t ring_bytes, uint64_t* b0, uint64_t* b1) {
    const uint32_t unit = pick_unit(body, chunksize, (count + nw - 1) / nw, sm_count, ring_bytes);
    const uint64_t units_per = ((count + unit - 1) / unit + nw - 1) / nw;
    *b0 = std::min<uint64_t>(count, (uint64_t)i * units_per * unit);
    *b1 = std::min<uint64_t>(count, (uint64_t)(i + 1) * units_per * unit);
}

// How worker `worker`'s block [first, first + count) of map `d` runs: its claim unit, its data path and the size of
// its waves.  Host arithmetic only -- no CUDA call, and the pool's state comes in through the arguments -- so the
// schedule can be checked without a device (fbr_internal_plan_part).  `root_alive`: worker 0, which holds
// device-resident arguments and output, is alive; `has_out`: the map has a result buffer (the caller's `out` or the
// engine's pinned segment; maps with FBR_RESULTS_ON_DEVICE have none).
static int plan_part(const BodyEntry& body, const fbr_map_desc_t& d, uint64_t first, uint64_t count, int worker,
                     bool root_alive, int sm_count, uint64_t ring_bytes, uint32_t pool_flags, bool has_out, PartPlan* out) {
    PartPlan c;
    c.R = body.result_bytes;
    c.resilient = (d.flags & FBR_RESILIENT) != 0;
    c.args_dev = (d.flags & FBR_ARGS_DEVICE) != 0;
    c.out_dev = (d.flags & FBR_OUT_DEVICE) != 0;
    c.keep_on_device = (d.flags & FBR_RESULTS_ON_DEVICE) != 0;
    // Output resident on worker 0, computed by another worker: kernels storing over NVLink top out near 510 GB/s
    // (TMA bulk or register stores alike), a copy engine pushes at the peer-copy rate (~770 GB/s).  So the block is
    // computed into the local out-staging halves and each wave is pushed to the root by this worker's copy engine,
    // overlapping the next wave's kernel (DESIGN.md section 6).
    c.peer_out = c.out_dev && worker != 0 && !c.resilient && !(d.flags & FBR_FULL_WINDOW);
    // Bit-packed bool results are small (1/8 B per task): instead of staging them in HBM and copying them out wave
    // by wave (6 x (2 MB D2H + ~8 us set-up) = the critical path of the e2e step), the dispatch kernel stores them
    // straight into the pinned host segment (zero copy): the PCIe writes spread over the whole kernel.
    // Measured (C ABI, 1e8 index tasks, 12.5 MB of results): 0.304 ms per map against 0.349 ms staged + copied in 6 waves.
    c.zero_copy = body.result_kind == FBR_RES_BITS8 && !c.out_dev && !c.resilient && !c.keep_on_device &&
                  !(d.flags & (FBR_FULL_WINDOW | FBR_SHUFFLE | FBR_VIA_RING | FBR_NO_ZERO_COPY)) && has_out;
    c.full_window = (c.out_dev && !c.peer_out) || c.resilient || c.keep_on_device || (d.flags & FBR_FULL_WINDOW) || c.zero_copy;
    // Device-resident arguments on worker 0, consumed by another worker: worker 0's copy engine pushes them wave by
    // wave into this worker's staging halves, the same wave / staging machinery as host-resident arguments.
    c.peer_push = c.args_dev && d.arg_stride != 0 && worker != 0 && !c.resilient && root_alive;
    c.host_args = d.arg_stride != 0 && !c.resilient && (!c.args_dev || c.peer_push);
    c.unit = pick_unit(body, d.chunksize, count, sm_count, ring_bytes);
    c.slot_stride = (uint32_t)round_up((uint64_t)c.unit * c.R, 16);
    const uint32_t unit = c.unit, R = c.R;
    if (d.n_items && d.arg_stride && body.result_kind == FBR_RES_BITS8)
        c.args_limit_bytes = d.n_items * (uint64_t)(d.arg_stride / 8);   // a byte-task's record is 8 items
    if (d.flags & FBR_WANT_SUM) {
        if (!(body.flags & FBR_BODY_SUMMABLE)) return fail(FBR_EINVAL, "body %s results cannot be summed", body.name.c_str());
        c.sum_kind = 1;   // the dispatch kernel folds sum(results) while they are in registers
    }

    // Opt-in (FBR_POOL_OVERLAP): gather(w) runs on a second, higher-priority stream while the next
    // wave's / next map's dispatch kernel computes; the ring is then used in alternating halves.
    // Measured on the pi map (ALU-bound dispatch + HBM-bound gather, maps pipelined back to back):
    // 0.3837 vs 0.3876 ms/step -- the gather is only 9 % of the step and the two kernels contend for
    // SM slots, so it is off by default.
    c.overlap = c.full_window && !c.resilient && (pool_flags & FBR_POOL_OVERLAP) != 0;
    // Direct placement: a contiguous, unshuffled, non-resilient block needs neither task records nor the
    // ring -- unit t of a wave is tasks [wave_first + t*unit, ...) and its results belong at exactly that
    // index of the ordered window, so the dispatch kernel stores them there and no gather is launched.
    // (Shuffled arrival, several attempts per unit and FBR_VIA_RING keep the ring + gather_ordered path.)
    const bool unit_ok = ((uint64_t)unit * R) % 16 == 0 || unit == 1;   // full vectors are stored 16 B at a time
    const bool base_ok = !c.out_dev || (((uintptr_t)d.out + first * R) & 15) == 0;
    c.direct = !c.resilient && !(d.flags & (FBR_SHUFFLE | FBR_VIA_RING)) && unit_ok && base_ok;

    // wave capacity in claim units
    uint64_t units_cap = c.direct ? (1ull << 31) :   // 32-bit unit counter; a direct wave needs no ring space
        std::min<uint64_t>(kRecCapacity, (c.overlap ? ring_bytes / 2 : ring_bytes) / c.slot_stride);
    if (c.host_args) units_cap = std::min<uint64_t>(units_cap, ring_bytes / ((uint64_t)unit * d.arg_stride));
    if (!c.full_window) units_cap = std::min<uint64_t>(units_cap, ring_bytes / ((uint64_t)unit * R));
    if (units_cap == 0) return fail(FBR_ENOMEM, "ring_bytes=%llu too small for one claim unit of %u tasks", (unsigned long long)ring_bytes, unit);
    c.wave_tasks_cap = units_cap * unit;
    // Host-resident output: cut large maps into ~8 waves (>= 8 MiB of results each) so the D2H of
    // wave w overlaps the kernels of wave w+1 instead of trailing one monolithic launch.  The waves are equal: ramps,
    // tapers and pyramids of wave sizes were measured and lost (profiles/r02_peer_sweep.txt, DESIGN.md section 6).
    if (!c.full_window || c.host_args) {
        const uint64_t bytes_per_task = std::max<uint64_t>(R, c.host_args ? d.arg_stride : 0);
        // a wave must carry enough kernel time to hide its launches: 8 MiB of byte results is ~22 us of
        // pi dispatch; a byte of bit-packed results stands for 8 tasks, so 1 MiB is the same work
        const uint64_t min_wave_bytes = body.result_kind == FBR_RES_BITS8 ? (1ull << 20) : (8ull << 20);
        const uint64_t min_wave_tasks = round_up(std::max<uint64_t>(1, min_wave_bytes / bytes_per_task), unit);
        // 8 waves for ~100 MB maps, up to 64 for multi-GB ones (~64 MiB per wave): the first wave's
        // H2D and the last wave's D2H are the only copies nothing overlaps with
        uint64_t n_waves = std::min<uint64_t>(64, std::max<uint64_t>(8, count * bytes_per_task / (64ull << 20)));
        // small outputs (bit-packed bools): per-copy set-up weighs more: T_kernel/n + n * 8 us is flattest at n = 5..6
        if (body.result_kind == FBR_RES_BITS8 && !c.host_args) n_waves = 6;
        const uint64_t share = round_up((count + n_waves - 1) / n_waves, unit);
        c.wave_tasks_cap = std::min(c.wave_tasks_cap, std::max(min_wave_tasks, share));
    }
    *out = c;
    return FBR_OK;
}

// Which gather kernel (see kernels.cuh) places a wave of `n_units` ring slots into its ordered window, and its grid.
// `out_aligned`: the window starts on a 16-byte boundary.  Host arithmetic only, like plan_part.
enum GatherKind { GATHER_FLAT, GATHER_ROWS, GATHER_BULK };
struct GatherPlan {
    GatherKind kind;
    int grid;
    uint32_t group_slots;                 // slots per ticket (rows / bulk)
    bool reverse;                         // rows: newest slot first
};
static GatherPlan plan_gather(const PartPlan& cx, bool out_aligned, uint32_t n_units, int sm_count, int occ_gather,
                              int occ_gather_rows) {
    const bool rows_ok = out_aligned && (uint64_t)cx.unit * cx.R == cx.slot_stride && cx.slot_stride % 4096 == 0;
    // TMA bulk pipeline for slots of whole 16 KB chunks (4 KB slots: the rows kernel is faster, 37 vs 41 us on the pi wave)
    if (rows_ok && !cx.resilient && cx.slot_stride % bulk::kChunk == 0) {
        // ONE warp per SM saturates HBM (measured 104 % of the copy peak vs 102.5 % with two);
        // ~256 KB of ring per ticket (<= 32 slots: one header per lane), >= ~8 tickets per CTA
        const uint64_t max_ctas = (uint64_t)sm_count;
        const uint32_t group_slots = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(
            std::min<uint64_t>(bulk::kGroup, (256u << 10) / cx.slot_stride), n_units / (8 * max_ctas)));
        const uint32_t n_groups = (n_units + group_slots - 1) / group_slots;
        return {GATHER_BULK, (int)std::min<uint64_t>(n_groups, max_ctas), group_slots, false};
    }
    if (rows_ok) {
        // ~128 KB of ring per ticket, but never fewer than ~4 tickets per resident CTA (small waves);
        // big slots (>= 32 KB): 4 fat streams per SM measured best (100 % of the copy peak vs 99 %)
        const int occ_g = cx.slot_stride >= (32u << 10) ? std::min(occ_gather_rows, 4) : occ_gather_rows;
        const uint64_t max_ctas = (uint64_t)sm_count * occ_g;
        const uint32_t group_slots = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>((128u << 10) / cx.slot_stride, n_units / (4 * max_ctas)));
        const uint32_t n_groups = (n_units + group_slots - 1) / group_slots;
        // waves that fit the L2 are gathered newest-slot-first (see the kernel)
        const bool reverse = (uint64_t)n_units * cx.slot_stride <= (128ull << 20);
        return {GATHER_ROWS, (int)std::min<uint64_t>(n_groups, max_ctas), group_slots, reverse};
    }
    const uint64_t total_vec = (uint64_t)n_units * (cx.slot_stride >> 4);
    const int grid = (int)std::max<uint64_t>(1, std::min<uint64_t>((total_vec + kThreads * 4 - 1) / (kThreads * 4),
                                                                   (uint64_t)sm_count * occ_gather));
    return {GATHER_FLAT, grid, 0, false};
}

static void shuffle_records(TaskRecord* r, uint32_t n, uint64_t seed) {
    for (uint32_t i = n; i > 1; --i) {
        seed = splitmix64(seed);
        const uint32_t j = (uint32_t)(seed % i);
        std::swap(r[i - 1], r[j]);
    }
}

// ------------------------------------------------------------------------------------------------
// wave pipeline for one worker's block of one map
// ------------------------------------------------------------------------------------------------
// One wave: `n_units` claim units -> copy-in, dispatch, gather, (streaming parts) copy-out.
// `wave_first`/`wt` describe the contiguous task window of a regular wave; a re-dispatch wave
// (arbitrary lost units) passes contiguous=false.  `have_records`: the caller wrote the wave's task
// records into the pinned window (shuffled, resilient or re-dispatch waves); otherwise the records
// are an arithmetic progression the kernels compute themselves.
static int run_wave(fbr_pool* p, SeqState& st, SeqPart& part, const BodyEntry& body, uint32_t n_units,
                    uint64_t wave_first, uint64_t wt, bool contiguous, bool have_records, uint64_t wno) {
    Worker& w = p->workers[part.worker];
    const PartCtx& cx = part.cx;
    const fbr_map_desc_t& d = st.desc;
    const bool timing = (p->flags & FBR_POOL_TIMING) != 0;
    const int rw = (int)(wno % kRecWindows);
    const int half = (int)(wno & 1);
    const int slot = part.ctrl_slot;
    const bool direct = cx.direct && contiguous && !have_records;
    TaskRecord* hrec = w.h_records + (size_t)rw * kRecCapacity;
    TaskRecord* drec = w.d_records + (size_t)rw * kRecCapacity;

    // copy-in stream: wait until the device window / arg half were consumed, then H2D.  A wave that copies
    // nothing in (computed records, range() or device-resident arguments) skips the hop through s_in -- every
    // cross-stream event costs the GPU a few microseconds per wave -- except the first wave of a block, which
    // has to see the control block (and shared block) its submit_part put on s_in.
    const bool in_copies = have_records || cx.host_args || part.first_wave_pending;
    part.first_wave_pending = false;
    if (in_copies) {
        CK(cudaStreamWaitEvent(w.s_in, w.ev_comp[rw], 0));  // wave wno-4 kernels done (device window free)
        if (wno >= 2) CK(cudaStreamWaitEvent(w.s_in, w.ev_comp[(wno - 2) % kRecWindows], 0));  // arg half free
    }
    if (have_records) {
        CK(cudaMemcpyAsync(drec, hrec, sizeof(TaskRecord) * n_units, cudaMemcpyHostToDevice, w.s_in));
        STAT_ADD(p, h2d_bytes, sizeof(TaskRecord) * n_units);
        STAT_ADD(p, records_copied, n_units);
    }
    const uint8_t* wave_args = cx.args_full;
    bool pushed = false;
    if (cx.host_args) {   // streaming arguments (contiguous waves only): from the host, or pushed by the root GPU
        uint64_t bytes = wt * d.arg_stride;
        if (cx.args_limit_bytes) {   // the last task of the map may cover fewer argument items than a full record
            const uint64_t start = wave_first * (uint64_t)d.arg_stride;
            bytes = start >= cx.args_limit_bytes ? 0 : std::min(bytes, cx.args_limit_bytes - start);
        }
        const uint8_t* src = (const uint8_t*)d.args + wave_first * (uint64_t)d.arg_stride;
        if (cx.peer_push) {
            // The copy runs on a stream of the ROOT device, so the root's copy engine WRITES the wave into this
            // worker's staging half (posted NVLink writes, root TX), while this worker's kernels store their results
            // into the root's output (posted writes, root RX): both directions of the root's links carry payload at
            // the same time and neither carries read requests.  (Peer LOADS + peer stores from one kernel reach
            // 504 GB/s each way; see DESIGN.md section 6.)
            if (bytes) {
                CK(cudaSetDevice(w.push_root_device));
                cudaStream_t sp = half ? w.s_push2 : w.s_push;
                cudaError_t e = cudaStreamWaitEvent(sp, w.ev_comp[rw], 0);                 // device window free
                if (e == cudaSuccess && wno >= 2) e = cudaStreamWaitEvent(sp, w.ev_comp[(wno - 2) % kRecWindows], 0);   // staging half free
                if (e == cudaSuccess) e = cudaMemcpyPeerAsync(w.d_args[half], w.device, src, w.push_root_device, bytes, sp);
                if (e == cudaSuccess) e = cudaEventRecord(w.ev_push[rw], sp);
                cudaSetDevice(w.device);
                if (e != cudaSuccess) return fail(FBR_ECUDA, "peer push of wave %llu failed: %s", (unsigned long long)wno, cudaGetErrorString(e));
                pushed = true;
                STAT_ADD(p, peer_push_bytes, bytes);
            }
        } else {
            if (bytes) CK(cudaMemcpyAsync(w.d_args[half], src, bytes, cudaMemcpyHostToDevice, w.s_in));
            STAT_ADD(p, h2d_bytes, bytes);
        }
        wave_args = w.d_args[half];
    }
    if (in_copies) CK(cudaEventRecord(w.ev_rec_h2d[rw], w.s_in));

    // compute streams: dispatch on s_comp; gather on s_comp too, or -- overlapped waves -- on the
    // higher-priority s_gath so that it runs while the next wave's dispatch kernel computes.
    // Overlapped waves use alternating halves of the ring / header array.  Direct waves use neither.
    const bool ov = cx.overlap && !direct;
    cudaStream_t s_g = ov ? w.s_gath : w.s_comp;
    uint8_t* ring_base = ov ? w.d_ring + (size_t)half * (p->ring_bytes / 2) : w.d_ring;
    SlotHeader* hdr_base = ov ? w.d_headers + (size_t)half * kRecCapacity : w.d_headers;
    if (in_copies) CK(cudaStreamWaitEvent(w.s_comp, w.ev_rec_h2d[rw], 0));
    if (pushed) CK(cudaStreamWaitEvent(w.s_comp, w.ev_push[rw], 0));
    // the ring region this dispatch writes must have been drained by the gather that last read it (gathers on
    // s_comp itself are ordered by the stream: only a gather that ran on s_gath needs the event)
    if ((w.gath_hist & 3u) || ov) {
        if (wno >= 1 && !(ov && w.prev_wave_overlap)) CK(cudaStreamWaitEvent(w.s_comp, w.ev_comp[(wno - 1) % kRecWindows], 0));
        if (wno >= 2) CK(cudaStreamWaitEvent(w.s_comp, w.ev_comp[(wno - 2) % kRecWindows], 0));
    }
    w.prev_wave_overlap = ov;
    w.gath_hist = ((w.gath_hist << 1) | (ov ? 1u : 0u)) & 3u;
    if (!cx.full_window) CK(cudaStreamWaitEvent(w.s_comp, w.ev_out[half], 0));  // out half drained
    uint8_t* const out_window = cx.full_window ? cx.window_base : w.d_out[half];      // ordered output of this wave's window
    const uint64_t out_first = cx.full_window ? part.first : wave_first;               // map index of out_window[0]
    WaveParams wp;
    memset(&wp, 0, sizeof wp);
    wp.records = have_records ? drec : nullptr;
    wp.headers = direct ? nullptr : hdr_base;
    wp.ring = direct ? out_window + (wave_first - out_first) * cx.R : ring_base;
    wp.ticket = w.d_tickets + (wno % kTickets);
    wp.n_units = n_units;
    wp.slot_stride = direct ? cx.unit * cx.R : cx.slot_stride;
    wp.args = wave_args;
    wp.arg_stride = d.arg_stride;
    wp.index_start = d.index_start;
    wp.index_step = d.index_step;
    wp.index_base = d.task_index_base;
    wp.shared = cx.d_shared;
    wp.shared_bytes = d.shared_bytes;
    wp.err_word = &w.d_ctrl[slot].err;
    wp.resilient = cx.resilient ? 1u : 0u;
    wp.sum = cx.sum_kind ? &w.d_ctrl[slot].sum : nullptr;
    wp.sum_hi = cx.sum_kind ? &w.d_ctrl[slot].sum_hi : nullptr;
    wp.syn_first = wave_first;
    wp.syn_tasks = wt;
    wp.syn_arg_off = cx.host_args ? 0 : wave_first * (uint64_t)d.arg_stride;
    wp.syn_unit = cx.unit;
    wp.syn_seq = (uint32_t)st.seq;
    wp.syn_func = (uint32_t)st.func_id;
    wp.syn_attempt = part.attempt;
    wp.n_items = d.n_items ? d.n_items : ~0ull;
    int occ_d = worker_occ(w, st.func_id, body, d.arg_stride == 0);
    if (body.max_ctas_per_sm) occ_d = std::min(occ_d, body.max_ctas_per_sm);
    if (ov && occ_d > 1) occ_d -= 1;     // leave SM slots for the concurrently running gather CTAs
    const int grid_d = (int)std::min<uint64_t>(n_units, (uint64_t)w.sm_count * occ_d);
    TimedPair td{nullptr, nullptr}, tg{nullptr, nullptr};
    if (timing) {
        CK(cudaEventCreate(&td.a)); CK(cudaEventCreate(&td.b));
        CK(cudaEventRecord(td.a, w.s_comp));
    }
    body.launch(&wp, grid_d, (void*)w.s_comp);
    CK(cudaGetLastError());
    if (timing) {
        CK(cudaEventRecord(td.b, w.s_comp));
        part.t_dispatch.push_back(td);
    }
    STAT_ADD(p, dispatch_launches, 1);
    STAT_ADD(p, units_dispatched, n_units);
    STAT_ADD(p, dispatch_bytes, wt * ((uint64_t)(d.arg_stride ? body.arg_bytes : 0) + cx.R));

    if (direct) {
        STAT_ADD(p, direct_waves, 1);
        CK(cudaEventRecord(w.ev_comp[rw], w.s_comp));
    } else {
        if (ov) {
            CK(cudaEventRecord(w.ev_disp[rw], w.s_comp));
            CK(cudaStreamWaitEvent(s_g, w.ev_disp[rw], 0));
        }
        if (timing) {
            CK(cudaEventCreate(&tg.a)); CK(cudaEventCreate(&tg.b));
            CK(cudaEventRecord(tg.a, s_g));
        }
        GatherParams gp;
        gp.headers = hdr_base;
        gp.ring = ring_base;
        gp.n_units = n_units;
        gp.slot_stride = cx.slot_stride;
        gp.result_bytes = cx.R;
        gp.pad = 0;
        gp.out = out_window;
        gp.win_first = out_first;
        gp.ticket_to_reset = nullptr;     // dispatch kernels re-arm their own ticket (TicketClaimer::rearm)
        gp.lost_count = cx.resilient ? &w.d_ctrl[slot].lost_count : nullptr;
        gp.lost_units = part.d_lost;
        gp.lost_capacity = part.lost_cap;
        const GatherPlan g = plan_gather(cx, ((uintptr_t)gp.out & 15) == 0, n_units, w.sm_count, w.occ_gather, w.occ_gather_rows);
        uint32_t* gticket = w.d_tickets + kTickets + (wno % kTickets);   // zero at launch, re-armed below
        if (g.kind == GATHER_BULK) {
            gather_bulk_kernel<<<g.grid, 32, (size_t)bulk::kStages * bulk::kChunk, s_g>>>(gp, gticket, bulk::kChunk, g.group_slots);
            CK(cudaMemsetAsync(gticket, 0, sizeof(uint32_t), s_g));
        } else if (g.kind == GATHER_ROWS) {
            gather_rows_kernel<<<g.grid, kThreads, 0, s_g>>>(gp, gticket, g.group_slots, g.reverse);
            CK(cudaMemsetAsync(gticket, 0, sizeof(uint32_t), s_g));
        } else {
            gather_ordered_kernel<<<g.grid, kThreads, 0, s_g>>>(gp);
        }
        CK(cudaGetLastError());
        if (timing) {
            CK(cudaEventRecord(tg.b, s_g));
            part.t_gather.push_back(tg);
        }
        CK(cudaEventRecord(w.ev_comp[rw], s_g));
        STAT_ADD(p, gather_launches, 1);
        STAT_ADD(p, gather_bytes, 2 * wt * cx.R);
    }

    // copy-out stream (streaming parts): D2H of the ordered window of this wave
    if (contiguous) {
        cudaEvent_t wd;
        CK(cudaEventCreateWithFlags(&wd, cudaEventDisableTiming));
        if (!cx.full_window) {
            // one copy-out stream: alternating two did not pay (0.362 vs 0.347 ms per 1e8-task map over PCIe, 3.40 vs
            // 3.41 ms for the NVLink push of 2 GB)
            cudaStream_t so = w.s_out;
            CK(cudaStreamWaitEvent(so, w.ev_comp[rw], 0));
            if (cx.peer_out) {      // this worker's copy engine writes the wave into the root's ordered output (posted NVLink writes)
                CK(cudaMemcpyPeerAsync((uint8_t*)st.out + wave_first * cx.R, p->workers[0].device, w.d_out[half], w.device, wt * cx.R, so));
                STAT_ADD(p, peer_push_bytes, wt * cx.R);
            } else {
                CK(cudaMemcpyAsync((uint8_t*)st.out + wave_first * cx.R, w.d_out[half], wt * cx.R, cudaMemcpyDeviceToHost, so));
                STAT_ADD(p, d2h_bytes, wt * cx.R);
            }
            CK(cudaEventRecord(w.ev_out[half], so));
            CK(cudaEventRecord(wd, so));
        } else {
            CK(cudaEventRecord(wd, direct ? w.s_comp : s_g));
        }
        part.wave_done.push_back(wd);
    }
    __atomic_fetch_add(&st.n_waves, 1u, __ATOMIC_RELAXED);
    return FBR_OK;
}

// Control block (+ lost list) back to the pinned mirror, completion event.
static int finish_round(fbr_pool* p, SeqState& st, SeqPart& part, bool copy_window) {
    Worker& w = p->workers[part.worker];
    const PartCtx& cx = part.cx;
    const int slot = part.ctrl_slot;
    const int last_rw = (int)((w.wave_no - 1) % kRecWindows);
    // The round finishes on s_out, behind the block's last kernels and its copy-outs, even when nothing was copied out:
    // a copy on the compute stream would put a DMA hop between the back-to-back kernels of pipelined maps.
    cudaStream_t sf = w.s_out;
    CK(cudaStreamWaitEvent(sf, w.ev_comp[last_rw], 0));
    if (copy_window && cx.full_window && !cx.out_dev && !cx.keep_on_device && !cx.zero_copy && part.count) {
        CK(cudaMemcpyAsync((uint8_t*)st.out + part.first * cx.R, cx.window_base, part.count * cx.R, cudaMemcpyDeviceToHost, sf));
        STAT_ADD(p, d2h_bytes, part.count * cx.R);
    }
    CK(cudaMemcpyAsync(&w.h_ctrl[slot], &w.d_ctrl[slot], sizeof(SeqCtrl), cudaMemcpyDeviceToHost, sf));
    if (cx.resilient && part.lost_cap)
        CK(cudaMemcpyAsync(part.h_lost, part.d_lost, sizeof(LostUnit) * part.lost_cap, cudaMemcpyDeviceToHost, sf));
    // one event per part for its whole life, re-recorded every round: another waiter may hold the handle
    // (fbr_result_wait blocks on it outside the pool lock), so it must never be destroyed under it
    if (!part.done) CK(cudaEventCreateWithFlags(&part.done, cudaEventDisableTiming));
    CK(cudaEventRecord(part.done, sf));
    return FBR_OK;
}

static int submit_part(fbr_pool* p, SeqState& st, SeqPart& part, const BodyEntry& body) {
    Worker& w = p->workers[part.worker];
    const fbr_map_desc_t& d = st.desc;
    PartCtx& cx = part.cx;
    CK(cudaSetDevice(w.device));
    const int prc = plan_part(body, d, part.first, part.count, part.worker, !p->workers[0].dead, w.sm_count, p->ring_bytes,
                              p->flags, st.out != nullptr, &cx);
    if (prc != FBR_OK) return prc;
    const uint32_t unit = cx.unit, R = cx.R;

    // push streams: a stream of the root device whose copy engine pushes this worker's argument waves
    if (cx.peer_push && w.s_push == nullptr) {
        const int root = p->workers[0].device;
        CK(cudaSetDevice(root));
        cudaError_t e = cudaStreamCreateWithFlags(&w.s_push, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&w.s_push2, cudaStreamNonBlocking);
        for (int i = 0; i < kRecWindows && e == cudaSuccess; ++i) e = cudaEventCreateWithFlags(&w.ev_push[i], cudaEventDisableTiming);
        cudaSetDevice(w.device);
        if (e != cudaSuccess) return fail(FBR_ECUDA, "creating the push stream on device %d failed: %s", root, cudaGetErrorString(e));
        w.push_root_device = root;
    }

    // control block
    if (w.ctrl_free.empty()) return fail(FBR_ENOMEM, "more than %d maps in flight on worker %d", kCtrlSlots, part.worker);
    const int slot = w.ctrl_free.back();
    w.ctrl_free.pop_back();
    part.ctrl_slot = slot;
    CK(cudaMemcpyAsync(&w.d_ctrl[slot], &w.h_ctrl[kCtrlSlots], sizeof(SeqCtrl), cudaMemcpyHostToDevice, w.s_in));

    // shared (broadcast) block
    if (d.shared != nullptr && d.shared_bytes) {
        if (d.flags & FBR_SHARED_HANDLE) {
            auto it = p->shared.find((uint64_t)(uintptr_t)d.shared);
            if (it == p->shared.end()) return fail(FBR_ENOENT, "unknown shared handle");
            cx.d_shared = (const uint8_t*)it->second.d_ptr[part.worker];
        } else if (cx.args_dev) {
            cx.d_shared = (const uint8_t*)d.shared;
        } else {
            CK(cudaMallocAsync(&part.d_shared_tmp, d.shared_bytes, w.s_in));
            CK(cudaMemcpyAsync(part.d_shared_tmp, d.shared, d.shared_bytes, cudaMemcpyHostToDevice, w.s_in));
            STAT_ADD(p, h2d_bytes, d.shared_bytes);
            cx.d_shared = (const uint8_t*)part.d_shared_tmp;
        }
    }

    // arguments that stay device-resident for the whole map
    if (cx.args_dev && !cx.peer_push) {
        cx.args_full = (const uint8_t*)d.args;
    } else if (cx.resilient && d.arg_stride) {
        // lost units may be re-dispatched at any time: keep every argument record on the device
        CK(cudaMallocAsync(&part.d_args_full, std::max<uint64_t>(16, st.n_tasks * (uint64_t)d.arg_stride), w.s_in));
        uint64_t abytes = part.count * (uint64_t)d.arg_stride;
        if (cx.args_limit_bytes) {
            const uint64_t start = part.first * (uint64_t)d.arg_stride;
            abytes = start >= cx.args_limit_bytes ? 0 : std::min(abytes, cx.args_limit_bytes - start);
        }
        if (abytes)
            CK(cudaMemcpyAsync((uint8_t*)part.d_args_full + part.first * (uint64_t)d.arg_stride,
                               (const uint8_t*)d.args + part.first * (uint64_t)d.arg_stride, abytes, cudaMemcpyHostToDevice, w.s_in));
        STAT_ADD(p, h2d_bytes, abytes);
        cx.args_full = (const uint8_t*)part.d_args_full;
    }

    // staging
    if (cx.host_args)
        for (int i = 0; i < 2; ++i)
            if (!w.d_args[i]) CK(cudaMalloc((void**)&w.d_args[i], p->ring_bytes));
    if (!cx.full_window)
        for (int i = 0; i < 2; ++i)
            if (!w.d_out[i]) CK(cudaMalloc((void**)&w.d_out[i], p->ring_bytes));
    if (cx.full_window) {
        if (cx.out_dev) {
            cx.window_base = (uint8_t*)d.out + part.first * R;
        } else if (cx.zero_copy) {
            cx.window_base = (uint8_t*)st.out + part.first * R;     // pinned host memory, mapped into the device's address space (UVA)
            STAT_ADD(p, d2h_bytes, part.count * (uint64_t)R);        // these bytes cross PCIe as the kernel's own stores
        } else {
            CK(cudaMallocAsync(&part.d_window, std::max<uint64_t>(part.count * R, 16), w.s_in));
            cx.window_base = (uint8_t*)part.d_window;
        }
    }
    if (cx.resilient) {
        part.lost_cap = (uint32_t)std::min<uint64_t>((part.count + unit - 1) / unit, 1u << 22);
        CK(cudaMallocAsync((void**)&part.d_lost, sizeof(LostUnit) * std::max<uint32_t>(1, part.lost_cap), w.s_in));
        CK(cudaHostAlloc((void**)&part.h_lost, sizeof(LostUnit) * std::max<uint32_t>(1, part.lost_cap), cudaHostAllocPortable));
    }

    // Equal waves of wave_tasks_cap tasks.  Task records go through the pinned ring window only when they are not an
    // arithmetic progression the kernels can compute (shuffled arrival).  (The host may not overwrite a window whose
    // previous H2D is in flight.)
    const bool have_records = (d.flags & FBR_SHUFFLE) != 0;
    for (uint64_t done_tasks = 0; done_tasks < part.count;) {
        const uint64_t wt = std::min<uint64_t>(cx.wave_tasks_cap, part.count - done_tasks);
        const uint32_t n_units = (uint32_t)((wt + unit - 1) / unit);
        const uint64_t wno = w.wave_no++;
        const int rw = (int)(wno % kRecWindows);
        const uint64_t wave_first = part.first + done_tasks;  // map index of the wave's first task
        if (have_records) {
            CK(cudaEventSynchronize(w.ev_rec_h2d[rw]));
            TaskRecord* hrec = w.h_records + (size_t)rw * kRecCapacity;
            for (uint32_t u = 0; u < n_units; ++u) {
                const uint64_t off = (uint64_t)u * unit;
                TaskRecord& r = hrec[u];
                r.seq = (uint32_t)st.seq;
                r.count = (uint32_t)std::min<uint64_t>(unit, wt - off);
                r.first = wave_first + off;
                r.arg_off = cx.host_args ? off * (uint64_t)d.arg_stride : (wave_first + off) * (uint64_t)d.arg_stride;
                r.func_id = (uint32_t)st.func_id;
                r.attempt = part.attempt;
            }
            shuffle_records(hrec, n_units, d.shuffle_seed ^ (wno * 0x9E3779B97F4A7C15ull));
        }
        int rc = run_wave(p, st, part, body, n_units, wave_first, wt, true, have_records, wno);
        if (rc != FBR_OK) return rc;
        done_tasks += wt;
        part.wave_cum.push_back(done_tasks);
    }
    // resilient parts copy the window back only once no unit is lost any more (resilient_advance)
    return finish_round(p, st, part, !cx.resilient);
}

// ResilientZPool semantics (fiber/pool.py:1612-1659): once a round has finished, re-queue the units
// whose worker died (their slot header carries kUnitLost; gather listed them) with attempt+1, until
// none is lost; then copy the ordered window back.  Returns 1 while more work was launched.
static int resilient_advance(fbr_pool* p, SeqState& st, SeqPart& part) {
    if (!part.cx.resilient || part.finalized) return 0;
    Worker& w = p->workers[part.worker];
    CK(cudaSetDevice(w.device));
    const BodyEntry& body = *body_of(st.func_id);
    const uint32_t lost = std::min(w.h_ctrl[part.ctrl_slot].lost_count, part.lost_cap);
    if (lost == 0) {
        part.finalized = true;
        int rc = finish_round(p, st, part, true);
        return rc != FBR_OK ? rc : 1;
    }
    if (++part.attempt > 200) return fail(FBR_ETASK, "units still failing after 200 re-dispatch rounds");
    st.redispatched_units += lost;
    std::vector<LostUnit> todo(part.h_lost, part.h_lost + lost);
    // clear the device lost counter (sum/err keep accumulating: lost units were never placed)
    static const uint32_t kZero = 0;
    CK(cudaMemcpyAsync(&w.d_ctrl[part.ctrl_slot].lost_count, &kZero, sizeof(uint32_t), cudaMemcpyHostToDevice, w.s_in));
    const uint64_t units_cap = std::max<uint64_t>(1, std::min<uint64_t>(kRecCapacity, p->ring_bytes / part.cx.slot_stride));
    for (size_t i = 0; i < todo.size(); i += units_cap) {
        const uint32_t n_units = (uint32_t)std::min<uint64_t>(units_cap, todo.size() - i);
        const uint64_t wno = w.wave_no++;
        const int rw = (int)(wno % kRecWindows);
        CK(cudaEventSynchronize(w.ev_rec_h2d[rw]));
        TaskRecord* hrec = w.h_records + (size_t)rw * kRecCapacity;
        uint64_t wt = 0;
        for (uint32_t u = 0; u < n_units; ++u) {
            const LostUnit& l = todo[i + u];
            TaskRecord& r = hrec[u];
            r.seq = (uint32_t)st.seq;
            r.count = l.count;
            r.first = l.first;
            r.arg_off = l.first * (uint64_t)st.desc.arg_stride;
            r.func_id = (uint32_t)st.func_id;
            r.attempt = part.attempt;
            wt += l.count;
        }
        int rc = run_wave(p, st, part, body, n_units, 0, wt, false, true, wno);
        if (rc != FBR_OK) return rc;
    }
    int rc = finish_round(p, st, part, false);
    return rc != FBR_OK ? rc : 1;
}

// ------------------------------------------------------------------------------------------------
// fault domain: a worker is a CUDA device; it "dies" when its context takes a sticky error (a kernel that
// trapped, an illegal address, an ECC error, a lost device).  The reference notices dead worker processes by
// their exit code and re-queues their pending chunks on the other workers (fiber/pool.py:1623-1656).
// ------------------------------------------------------------------------------------------------
// Every call on a corrupted context returns its sticky error; a healthy stream answers Success / NotReady.
static bool worker_context_dead(Worker& w, cudaError_t* why) {
    if (w.dead) return true;
    cudaError_t e = cudaSetDevice(w.device);
    if (e == cudaSuccess) e = cudaStreamQuery(w.s_comp);
    cudaGetLastError();
    if (e == cudaSuccess || e == cudaErrorNotReady) return false;
    if (why) *why = e;
    return true;
}

// contiguous, claim-unit aligned sub-blocks of tasks [first, first + count) over `workers`
static void cut_blocks(fbr_pool* p, const BodyEntry& body, const fbr_map_desc_t& d, uint64_t first, uint64_t count,
                       const std::vector<int>& workers, uint32_t attempt, std::vector<SeqPart>& out) {
    const int nw = (int)workers.size();
    if (nw == 0 || count == 0) return;
    for (int i = 0; i < nw; ++i) {
        uint64_t b0, b1;
        block_range(body, d.chunksize, count, nw, i, p->workers[workers[0]].sm_count, p->ring_bytes, &b0, &b1);
        if (b1 <= b0) continue;
        SeqPart part;
        part.worker = workers[i];
        part.first = first + b0;
        part.count = b1 - b0;
        part.attempt = attempt;
        out.push_back(std::move(part));
    }
}

static int submit_part(fbr_pool* p, SeqState& st, SeqPart& part, const BodyEntry& body);

// Worker `wi` is dead.  Maps that asked for ResilientZPool semantics get the blocks it was working on cut
// over the surviving workers and re-dispatched with attempt + 1 (whole blocks: what a dead context had
// finished cannot be asked any more); other maps are failed (a plain ZPool map whose worker dies never
// returns, fiber/pool.py:801-824 -- here it raises).  The pool keeps serving on the survivors.
static void on_worker_death(fbr_pool* p, int wi, cudaError_t err) {
    Worker& w = p->workers[wi];
    if (w.dead) return;
    w.dead = true;
    w.death_error = (int)err;
    p->stats.workers_lost++;
    cudaGetLastError();
    std::vector<int> live;
    for (size_t i = 0; i < p->workers.size(); ++i)
        if (!p->workers[i].dead) live.push_back((int)i);
    std::vector<uint64_t> ids;
    for (auto& kv : p->seqs) ids.push_back(kv.first);
    for (uint64_t id : ids) {
        auto it = p->seqs.find(id);
        if (it == p->seqs.end()) continue;
        SeqState& st = *it->second;
        if (st.finished || st.dead_worker >= 0) continue;
        bool touched = false;
        for (auto& part : st.parts) touched |= part.worker == wi;
        if (!touched) continue;
        // device-resident arguments / outputs of a map live on worker 0
        const bool on_w0 = (st.flags & (FBR_ARGS_DEVICE | FBR_OUT_DEVICE)) != 0;
        if (!(st.flags & FBR_RESILIENT) || live.empty() || (on_w0 && p->workers[0].dead)) {
            st.dead_worker = wi;
            st.dead_error = (int)err;
            continue;
        }
        const BodyEntry& body = *body_of(st.func_id);
        std::vector<SeqPart> next;
        for (auto& part : st.parts) {
            if (part.worker != wi) { next.push_back(std::move(part)); continue; }
            cut_blocks(p, body, st.desc, part.first, part.count, live, part.attempt + 1, next);
            st.redispatched_units += (uint32_t)((part.count + std::max<uint32_t>(1, part.cx.unit) - 1) / std::max<uint32_t>(1, part.cx.unit));
            st.graveyard.push_back(std::move(part));
        }
        st.parts.swap(next);
        for (size_t i = 0; i < st.parts.size(); ++i) {
            SeqPart& part = st.parts[i];
            if (part.ctrl_slot >= 0) continue;            // submitted before
            const int pw = part.worker;
            if (p->workers[pw].dead) continue;            // re-cut by a nested call below
            if (submit_part(p, st, part, body) != FBR_OK) {
                cudaError_t why = cudaSuccess;
                if (worker_context_dead(p->workers[pw], &why)) {
                    on_worker_death(p, pw, why);          // a survivor turned out dead as well: cut again (st.parts changes)
                    i = (size_t)-1;                       // restart: submit whatever is still unsubmitted
                    if (st.dead_worker >= 0) break;
                } else {
                    st.dead_worker = wi;                  // a real submission error: fail the map
                    st.dead_error = (int)err;
                    break;
                }
            }
        }
    }
}

static void free_seq(fbr_pool* p, SeqState& st) {
    for (auto& part : st.graveyard)        // device-side resources died with the worker's context
        if (part.h_lost) cudaFreeHost(part.h_lost);
    st.graveyard.clear();
    for (auto& part : st.parts) {
        Worker& w = p->workers[part.worker];
        if (w.dead) {                      // nothing on a dead context can be freed (or needs to be)
            if (part.h_lost) cudaFreeHost(part.h_lost);
            continue;
        }
        cudaSetDevice(w.device);
        if (part.done) { cudaEventSynchronize(part.done); cudaEventDestroy(part.done); }
        for (auto e : part.wave_done) cudaEventDestroy(e);
        for (auto& t : part.t_dispatch) { cudaEventDestroy(t.a); cudaEventDestroy(t.b); }
        for (auto& t : part.t_gather) { cudaEventDestroy(t.a); cudaEventDestroy(t.b); }
        // stream-ordered frees: cudaFree would synchronise the whole device, i.e. wait for resident
        // device processes (queues.cu) that may themselves be waiting for this host thread
        if (part.d_shared_tmp) cudaFreeAsync(part.d_shared_tmp, w.s_in);
        if (part.d_window) cudaFreeAsync(part.d_window, w.s_in);
        if (part.d_args_full) cudaFreeAsync(part.d_args_full, w.s_in);
        if (part.d_lost) cudaFreeAsync(part.d_lost, w.s_in);
        if (part.h_lost) cudaFreeHost(part.h_lost);
        if (part.ctrl_slot >= 0) w.ctrl_free.push_back(part.ctrl_slot);
    }
    if (st.own_out && st.out && !numa_pinned_release(p, st.out)) pinned_release(p, st.out);
}

// ------------------------------------------------------------------------------------------------
// extern "C" API
// ------------------------------------------------------------------------------------------------
extern "C" {

int fbr_abi_version(void) { return FBR_ABI_VERSION; }

// Force-load every kernel of this library on `device`.  With CUDA's lazy module loading the first
// launch of a kernel may synchronise the context; if a resident device process (queues.cu) is
// spinning on a host message at that moment the two deadlock.  queues.cu calls this before it
// starts a resident kernel.  (Internal: not part of the public header.)
int fbr_internal_preload(int device) {
    if (cudaSetDevice(device) != cudaSuccess) return FBR_ECUDA;
    cudaFuncAttributes at;
    for (int f = 0, n = body_count(); f < n; ++f) {   // asking for the occupancy loads the kernels
        const BodyEntry& b = *body_of(f);
        b.occupancy(0);
        if (b.flags & FBR_BODY_INDEX_ARG) b.occupancy(1);
    }
    cudaFuncGetAttributes(&at, (const void*)gather_ordered_kernel);
    cudaFuncGetAttributes(&at, (const void*)gather_rows_kernel);
    cudaFuncGetAttributes(&at, (const void*)gather_bulk_kernel);
    cudaFuncGetAttributes(&at, (const void*)dispatch_payload_map_tma_kernel<3, 2>);
    cudaFuncGetAttributes(&at, (const void*)payload_fill_kernel);
    cudaGetLastError();
    return FBR_OK;
}
const char* fbr_last_error(void) { return g_err.c_str(); }

int fbr_device_count(int* n) {
    if (!n) return fail(FBR_EINVAL, "n is NULL");
    int c = 0;
    cudaError_t e = cudaGetDeviceCount(&c);
    if (e != cudaSuccess) {
        *n = 0;
        cudaGetLastError();
        return fail(FBR_ENODEV, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
    }
    *n = c;
    return FBR_OK;
}

int fbr_body_count(int* n) {
    if (!n) return fail(FBR_EINVAL, "n is NULL");
    *n = body_count();
    return FBR_OK;
}

int fbr_body_info(int func_id, fbr_body_info_t* info) {
    const BodyEntry* bp = body_of(func_id);
    if (!info || !bp) return fail(FBR_EINVAL, "bad func_id %d", func_id);
    const BodyEntry& b = *bp;
    memset(info, 0, sizeof *info);
    info->func_id = func_id;
    info->arg_bytes = b.arg_bytes;
    info->result_bytes = b.result_bytes;
    info->result_kind = b.result_kind;
    info->flags = b.flags;
    info->unit_tasks = b.unit_tasks;
    snprintf(info->name, sizeof info->name, "%s", b.name.c_str());
    return FBR_OK;
}

int fbr_body_lookup(const char* name, int* func_id) {
    if (!name || !func_id) return fail(FBR_EINVAL, "NULL argument");
    for (int f = 0, n = body_count(); f < n; ++f)
        if (body_of(f)->name == name) { *func_id = f; return FBR_OK; }
    return fail(FBR_ENOENT, "no device body named '%s' is compiled into libfiber_b200 or registered with fbr_register_body", name);
}

int fbr_register_body(const char* name, const char* module_path, const char* entry, int* func_id) {
    if (!name || !module_path || !entry || !func_id) return fail(FBR_EINVAL, "NULL argument");
    // RTLD_LOCAL: several body modules may define the same helper symbols
    void* h = dlopen(module_path, RTLD_NOW | RTLD_LOCAL);
    if (!h) return fail(FBR_ENOENT, "dlopen(%s) failed: %s", module_path, dlerror());
    fbr_body_entry_fn fn = (fbr_body_entry_fn)dlsym(h, entry);
    if (!fn) {
        dlclose(h);
        return fail(FBR_ENOENT, "module %s has no entry point '%s'", module_path, entry);
    }
    const fbr_body_module_t* m = fn();
    if (!m || m->abi != FBR_BODY_MODULE_ABI || m->wave_params_bytes != sizeof(WaveParams) || !m->launch || !m->occupancy || !m->name) {
        const unsigned abi = m ? m->abi : 0u, wpb = m ? m->wave_params_bytes : 0u;
        dlclose(h);
        return fail(FBR_EINVAL, "module %s: descriptor ABI %u / wave-parameter size %u do not match this library (%u / %u); rebuild it against include/fiber_b200_body.cuh",
                    module_path, abi, wpb, (unsigned)FBR_BODY_MODULE_ABI, (unsigned)sizeof(WaveParams));
    }
    if (strcmp(m->name, name) != 0) {
        dlclose(h);
        return fail(FBR_EINVAL, "module %s exports body '%s', not '%s'", module_path, m->name, name);
    }
    if (m->flags & FBR_BODY_RECORD) {
        // record bodies (dispatch_record_kernel): 4..256-byte records in whole words, explicit arguments, opaque results
        auto bad = [](uint32_t b) { return b < 4 || b > 256 || b % 4 != 0; };
        if (bad(m->arg_bytes) || bad(m->result_bytes) || m->unit_tasks == 0 || m->result_kind != FBR_RES_BYTES) {
            dlclose(h);
            return fail(FBR_EINVAL, "module %s: record body '%s' needs argument and result records of 4..256 bytes in whole "
                        "words (got %u / %u) and result kind FBR_RES_BYTES", module_path, name, m->arg_bytes, m->result_bytes);
        }
        if (m->flags & (FBR_BODY_SUMMABLE | FBR_BODY_INDEX_ARG | FBR_BODY_INDEX_ONLY | FBR_BODY_NEEDS_SHARED)) {
            dlclose(h);
            return fail(FBR_EINVAL, "module %s: record body '%s' cannot be summable, take range() indices or a shared block",
                        module_path, name);
        }
    } else if (m->result_bytes == 0 || m->unit_tasks == 0 || (m->arg_bytes % 8) != 0 || m->result_kind > FBR_RES_BITS8) {
        dlclose(h);
        return fail(FBR_EINVAL, "module %s: body '%s' has an invalid record layout", module_path, name);
    }
    std::lock_guard<std::mutex> g(g_body_mu);
    builtin_bodies_once();
    for (size_t f = 0; f < g_bodies.size(); ++f)
        if (g_bodies[f].name == name) {
            if (g_bodies[f].module == nullptr) { dlclose(h); return fail(FBR_EINVAL, "'%s' is a compiled-in body", name); }
            dlclose(h);             // same name registered before: idempotent, keep the first module
            *func_id = (int)f;
            return FBR_OK;
        }
    BodyEntry b;
    b.name = name;
    b.arg_bytes = m->arg_bytes; b.result_bytes = m->result_bytes; b.result_kind = m->result_kind;
    b.flags = m->flags; b.unit_tasks = m->unit_tasks;
    b.launch = m->launch; b.occupancy = m->occupancy;
    b.module = h;
    g_bodies.push_back(b);
    *func_id = (int)g_bodies.size() - 1;
    return FBR_OK;
}

int fbr_plan_query(int func_id, uint64_t n_tasks, uint32_t chunksize, uint64_t ring_bytes, int n_workers,
                   int worker, int sm_count, fbr_plan_t* plan) {
    if (!plan || !body_of(func_id) || n_workers < 1 || worker < 0 || worker >= n_workers)
        return fail(FBR_EINVAL, "bad arguments");
    const BodyEntry& body = *body_of(func_id);
    const uint64_t ring = pool_ring_bytes(ring_bytes);
    if (sm_count <= 0) sm_count = 148;
    // the same two steps fbr_map_submit takes: blocks on the map-level unit (cut_blocks), then the block's own unit
    // (plan_part)
    uint64_t b0, b1;
    block_range(body, chunksize, n_tasks, n_workers, worker, sm_count, ring, &b0, &b1);
    plan->block_first = b0;
    plan->block_count = b1 - b0;
    plan->unit_tasks = pick_unit(body, chunksize, b1 - b0, sm_count, ring);
    plan->slot_stride = (uint32_t)round_up((uint64_t)plan->unit_tasks * body.result_bytes, 16);
    plan->n_units = plan->block_count ? (plan->block_count + plan->unit_tasks - 1) / plan->unit_tasks : 0;
    return FBR_OK;
}

// What plan_part decides for the block [first, first + count) of map `d` on worker `worker` of a pool with `ring_bytes`
// (0: the default) and `pool_flags`, on a device with `sm_count` SMs (<= 0: 148): the claim unit, the slot stride, the
// path flags (bit k set = the k-th of args_dev, out_dev, keep_on_device, resilient, peer_out, peer_push, zero_copy,
// full_window, host_args, overlap, direct), the tasks per wave and the number of waves.  Needs no device, so the
// schedule can be tested anywhere.  (Internal: not part of the public header.)
int fbr_internal_plan_part(const fbr_map_desc_t* d, uint64_t first, uint64_t count, int worker, int root_alive,
                           int sm_count, uint64_t ring_bytes, uint32_t pool_flags, int has_out, uint32_t* unit_tasks,
                           uint32_t* slot_stride, uint32_t* path_flags, uint64_t* wave_tasks_cap, uint64_t* n_waves) {
    if (!d || !body_of(d->func_id) || count == 0 || worker < 0 || !unit_tasks || !slot_stride || !path_flags ||
        !wave_tasks_cap || !n_waves)
        return fail(FBR_EINVAL, "bad arguments");
    PartPlan c;
    const int rc = plan_part(*body_of(d->func_id), *d, first, count, worker, root_alive != 0, sm_count > 0 ? sm_count : 148,
                             pool_ring_bytes(ring_bytes), pool_flags, has_out != 0, &c);
    if (rc != FBR_OK) return rc;
    const bool path[] = {c.args_dev, c.out_dev, c.keep_on_device, c.resilient, c.peer_out, c.peer_push,
                         c.zero_copy, c.full_window, c.host_args, c.overlap, c.direct};
    *path_flags = 0;
    for (size_t k = 0; k < sizeof path / sizeof path[0]; ++k) *path_flags |= (uint32_t)path[k] << k;
    *unit_tasks = c.unit;
    *slot_stride = c.slot_stride;
    *wave_tasks_cap = c.wave_tasks_cap;
    *n_waves = (count + c.wave_tasks_cap - 1) / c.wave_tasks_cap;   // submit_part's loop: equal waves, a shorter last one
    return FBR_OK;
}

int fbr_pool_create(int n_workers, const int* device_ids, uint64_t ring_bytes, uint32_t flags, fbr_pool_t** out) {
    if (!out || n_workers <= 0) return fail(FBR_EINVAL, "bad arguments");
    int ndev = 0;
    int rc = fbr_device_count(&ndev);
    if (rc != FBR_OK) return rc;
    if (ndev == 0) return fail(FBR_ENODEV, "no CUDA device visible; fiber_b200 has no CPU fallback");
    std::unique_ptr<fbr_pool> p(new fbr_pool());
    p->flags = flags;
    p->ring_bytes = pool_ring_bytes(ring_bytes);
    if (p->ring_bytes >= (1ull << 35)) return fail(FBR_EINVAL, "ring_bytes must be below 32 GiB (32-bit vector index in gather_ordered)");
    memset(&p->stats, 0, sizeof p->stats);
    p->workers.resize(n_workers);
    for (int i = 0; i < n_workers; ++i) {
        const int dev = device_ids ? device_ids[i] : (i % ndev);
        if (dev < 0 || dev >= ndev) return fail(FBR_EINVAL, "device id %d out of range (have %d)", dev, ndev);
        for (int j = 0; j < i; ++j)
            if (p->workers[j].device == dev) return fail(FBR_EINVAL, "device %d bound to two workers", dev);
        rc = worker_init(p.get(), p->workers[i], dev);
        if (rc != FBR_OK) {
            for (auto& w : p->workers) worker_destroy(w);
            return rc;
        }
    }
    // Peer access (NVLink P2P) is switched on by the first map that needs it (ensure_peer_access): contexts
    // with peer mappings between them share their fate -- a kernel fault on one device takes the peers' contexts
    // down with it -- so a pool that only runs host-resident maps keeps its workers' fault domains separate.
    *out = p.release();
    return FBR_OK;
}

// Peer access between all workers: lets one map keep its arguments / ordered output resident on worker 0
// while every worker's dispatch kernel loads its block from there and stores its results there, straight
// over NVLink (scatter + gather fused into the kernel, no separate collective).
static bool ensure_peer_access(fbr_pool* p) {
    if (p->peer_checked) return p->peer_ok;
    p->peer_checked = true;
    const int n = (int)p->workers.size();
    p->peer_ok = n > 1;
    for (int i = 0; i < n && p->peer_ok; ++i)
        for (int j = 0; j < n; ++j) {
            if (i == j) continue;
            int can = 0;
            cudaDeviceCanAccessPeer(&can, p->workers[i].device, p->workers[j].device);
            if (!can) { p->peer_ok = false; break; }
            cudaSetDevice(p->workers[i].device);
            cudaError_t e = cudaDeviceEnablePeerAccess(p->workers[j].device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) p->peer_ok = false;
            cudaGetLastError();
        }
    return p->peer_ok;
}

int fbr_pool_n_workers(fbr_pool_t* p, int* n) {
    if (!p || !n) return fail(FBR_EINVAL, "NULL argument");
    *n = (int)p->workers.size();
    return FBR_OK;
}

int fbr_pool_worker_device(fbr_pool_t* p, int worker, int* dev) {
    if (!p || !dev || worker < 0 || worker >= (int)p->workers.size()) return fail(FBR_EINVAL, "bad worker");
    *dev = p->workers[worker].device;
    return FBR_OK;
}

int fbr_pool_close(fbr_pool_t* p) {
    if (!p) return fail(FBR_EINVAL, "NULL pool");
    std::lock_guard<std::mutex> g(p->mu);
    if (p->state == ST_RUN) p->state = ST_CLOSE;
    return FBR_OK;
}

int fbr_pool_terminate(fbr_pool_t* p) {
    if (!p) return fail(FBR_EINVAL, "NULL pool");
    std::lock_guard<std::mutex> g(p->mu);
    p->state = ST_TERMINATE;
    return FBR_OK;
}

int fbr_pool_join(fbr_pool_t* p) {
    if (!p) return fail(FBR_EINVAL, "NULL pool");
    std::lock_guard<std::mutex> g(p->mu);
    if (p->state == ST_RUN) return fail(FBR_ESTATE, "join() before close()/terminate()");
    for (auto& w : p->workers) {
        CK(cudaSetDevice(w.device));
        CK(cudaStreamSynchronize(w.s_in));
        CK(cudaStreamSynchronize(w.s_comp));
        CK(cudaStreamSynchronize(w.s_gath));
        CK(cudaStreamSynchronize(w.s_out));
    }
    return FBR_OK;
}

int fbr_pool_destroy(fbr_pool_t* p) {
    if (!p) return FBR_OK;
    {
        std::lock_guard<std::mutex> g(p->mu);
        p->submitters.clear();          // joins the submit threads
        for (auto& kv : p->seqs) free_seq(p, *kv.second);
        p->seqs.clear();
        for (auto& kv : p->shared)
            for (size_t i = 0; i < kv.second.d_ptr.size(); ++i) {
                cudaSetDevice(p->workers[i].device);
                cudaFreeAsync(kv.second.d_ptr[i], p->workers[i].s_comp);
            }
        for (auto& w : p->workers) worker_destroy(w);
        for (auto& kv : p->pin_free)
            for (void* q : kv.second) cudaFreeHost(q);
        for (auto& kv : p->pin_live) cudaFreeHost(kv.first);
        for (auto& kv : p->numa_live) { cudaHostUnregister(kv.first); munmap(kv.first, kv.second.second); }
    }
    delete p;
    return FBR_OK;
}

int fbr_shared_put(fbr_pool_t* p, const void* host, uint64_t bytes, uint64_t* handle) {
    if (!p || !host || !bytes || !handle) return fail(FBR_EINVAL, "bad arguments");
    std::lock_guard<std::mutex> g(p->mu);
    SharedBlock sb;
    sb.bytes = bytes;
    for (auto& w : p->workers) {
        CK(cudaSetDevice(w.device));
        void* dptr = nullptr;
        CK(cudaMallocAsync(&dptr, bytes, w.s_in));
        CK(cudaMemcpyAsync(dptr, host, bytes, cudaMemcpyHostToDevice, w.s_in));
        CK(cudaStreamSynchronize(w.s_in));
        sb.d_ptr.push_back(dptr);
        p->stats.h2d_bytes += bytes;
    }
    *handle = p->next_shared++;
    p->shared[*handle] = sb;
    return FBR_OK;
}

int fbr_shared_drop(fbr_pool_t* p, uint64_t handle) {
    if (!p) return fail(FBR_EINVAL, "NULL pool");
    std::lock_guard<std::mutex> g(p->mu);
    auto it = p->shared.find(handle);
    if (it == p->shared.end()) return fail(FBR_ENOENT, "unknown shared handle");
    for (size_t i = 0; i < it->second.d_ptr.size(); ++i) {
        Worker& w = p->workers[i];
        cudaSetDevice(w.device);
        cudaStreamSynchronize(w.s_comp);   // maps that read the block have been waited for by their owners
        cudaFreeAsync(it->second.d_ptr[i], w.s_comp);
    }
    p->shared.erase(it);
    return FBR_OK;
}

int fbr_map_submit(fbr_pool_t* p, const fbr_map_desc_t* d, uint64_t* seq_out) {
    if (!p || !d || !seq_out) return fail(FBR_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> g(p->mu);
    if (p->state != ST_RUN) return fail(FBR_ESTATE, "Pool is not running");
    if (!body_of(d->func_id)) return fail(FBR_EINVAL, "bad func_id %d", d->func_id);
    const BodyEntry& body = *body_of(d->func_id);
    const bool dev_mode = (d->flags & (FBR_ARGS_DEVICE | FBR_OUT_DEVICE)) != 0;
    if (dev_mode && p->workers.size() != 1 && !ensure_peer_access(p))
        return fail(FBR_EINVAL, "device-resident args/out on a multi-worker pool need peer access between all its GPUs");
    if (d->arg_stride == 0) {
        if (!(body.flags & FBR_BODY_INDEX_ARG))
            return fail(FBR_EINVAL, "body %s needs explicit argument records (arg_stride=0)", body.name.c_str());
    } else if (body.flags & FBR_BODY_INDEX_ONLY) {
        return fail(FBR_EINVAL, "body %s takes range() arguments only (arg_stride must be 0)", body.name.c_str());
    } else if (body.flags & FBR_BODY_RECORD) {
        // the record kernel copies whole words from any 4-byte aligned record (kernels.cuh, dispatch_record_kernel)
        if (d->arg_stride < body.arg_bytes || (d->arg_stride % 4) != 0)
            return fail(FBR_EINVAL, "arg_stride %u invalid for body %s (arg_bytes %u)", d->arg_stride, body.name.c_str(), body.arg_bytes);
        if (d->n_tasks && !d->args) return fail(FBR_EINVAL, "args is NULL");
        if ((uintptr_t)d->args % 4) return fail(FBR_EINVAL, "argument records of body %s must be 4-byte aligned", body.name.c_str());
    } else {
        if (d->arg_stride < body.arg_bytes || (d->arg_stride % 8) != 0)
            return fail(FBR_EINVAL, "arg_stride %u invalid for body %s (arg_bytes %u)", d->arg_stride, body.name.c_str(), body.arg_bytes);
        if (d->n_tasks && !d->args) return fail(FBR_EINVAL, "args is NULL");
        if (body.arg_bytes >= 16 && body.result_kind != FBR_RES_BITS8 && (d->arg_stride % 16 || ((uintptr_t)d->args % 16)))
            return fail(FBR_EINVAL, "argument records of body %s must be 16-byte aligned", body.name.c_str());
    }
    if ((body.flags & FBR_BODY_NEEDS_SHARED) && (!d->shared || d->shared_bytes < sizeof(ParzenShared)))
        return fail(FBR_EINVAL, "body %s needs a shared argument block", body.name.c_str());
    if ((d->flags & FBR_OUT_DEVICE) && !d->out) return fail(FBR_EINVAL, "FBR_OUT_DEVICE without out");
    if ((d->flags & FBR_RESULTS_ON_DEVICE) && ((d->flags & FBR_OUT_DEVICE) || d->out))
        return fail(FBR_EINVAL, "FBR_RESULTS_ON_DEVICE owns its output buffer: do not pass out / FBR_OUT_DEVICE");
    if ((d->flags & FBR_RESILIENT) && (d->flags & FBR_SHUFFLE)) return fail(FBR_EINVAL, "FBR_RESILIENT cannot be combined with FBR_SHUFFLE");
    if ((d->flags & FBR_WANT_SUM) && !(body.flags & FBR_BODY_SUMMABLE))
        return fail(FBR_EINVAL, "body %s results cannot be summed", body.name.c_str());

    // A submission can find out that a worker has died (its context rejects every call): the worker is
    // retired, maps in flight are re-dispatched or failed (on_worker_death) and this map is cut again over
    // the survivors -- at most once per worker.
    for (size_t round = 0; round <= p->workers.size(); ++round) {
        std::vector<int> live;
        for (size_t i = 0; i < p->workers.size(); ++i)
            if (!p->workers[i].dead) live.push_back((int)i);
        if (live.empty()) return fail(FBR_ECUDA, "every worker of this pool has died (last CUDA error: %s)",
                                      cudaGetErrorString((cudaError_t)p->workers[0].death_error));
        if (dev_mode && p->workers[0].dead)
            return fail(FBR_ECUDA, "worker 0, which holds the device-resident arguments / output, has died");
        std::unique_ptr<SeqState> st(new SeqState());
        st->seq = ++p->next_seq;
        st->n_tasks = d->n_tasks;
        st->func_id = d->func_id;
        st->flags = d->flags;
        st->result_bytes = body.result_bytes;
        st->result_kind = body.result_kind;
        st->out = d->out;
        st->desc = *d;
        const bool need_segment = !st->out && d->n_tasks && !(d->flags & FBR_RESULTS_ON_DEVICE);
        // host allocations fail with the sticky error too once a context of this process has died: tell the two apart
        auto died_meanwhile = [&]() {
            bool any = false;
            for (int wi : live) {
                cudaError_t why = cudaSuccess;
                if (worker_context_dead(p->workers[wi], &why)) { on_worker_death(p, wi, why); any = true; }
            }
            return any;
        };
        if (need_segment && live.size() == 1) {
            int rc = pinned_acquire(p, d->n_tasks * body.result_bytes, &st->out);
            if (rc != FBR_OK) {
                const std::string msg = g_err;
                if (died_meanwhile()) continue;
                g_err = msg;
                return rc;
            }
            st->own_out = true;
        }
        // contiguous task blocks per live worker, cut on claim-unit boundaries (block partition ==
        // PUSH round-robin with chunk = block, SURVEY.md 8(e))
        cut_blocks(p, body, *d, 0, d->n_tasks, live, d->attempt, st->parts);
        if (need_segment && live.size() > 1) {
            // several GPUs fill one segment: bind each worker's block to its GPU's NUMA node
            std::vector<NumaBlock> blocks;
            for (auto& part : st->parts)
                blocks.push_back({part.first * body.result_bytes, part.count * body.result_bytes, p->workers[part.worker].numa_node});
            int rc = numa_pinned_acquire(p, d->n_tasks * body.result_bytes, blocks, &st->out);
            if (rc != FBR_OK) {
                const std::string msg = g_err;
                if (died_meanwhile()) continue;
                g_err = msg;
                return rc;
            }
            st->own_out = true;
        }
        int failed_worker = -1, rc = FBR_OK;
        if (st->parts.size() > 1) {
            // one submit thread per worker (see SubmitThread); this thread holds the pool lock meanwhile
            if (p->submitters.size() < p->workers.size()) p->submitters.resize(p->workers.size());
            SeqState* stp = st.get();
            for (auto& part : st->parts) {
                auto& sub = p->submitters[part.worker];
                if (!sub) sub.reset(new SubmitThread());
                SeqPart* pp = &part;
                sub->post([p, stp, pp, &body] { return submit_part(p, *stp, *pp, body); });
            }
            for (auto& part : st->parts) {
                std::string msg;
                const int r = p->submitters[part.worker]->wait(&msg);
                if (r != FBR_OK && rc == FBR_OK) { rc = r; failed_worker = part.worker; g_err = msg; }
            }
        } else {
            for (auto& part : st->parts) {
                rc = submit_part(p, *st, part, body);
                if (rc != FBR_OK) { failed_worker = part.worker; break; }
            }
        }
        if (rc == FBR_OK) {
            p->stats.tasks_submitted += d->n_tasks;
            *seq_out = st->seq;
            p->seqs[st->seq] = std::move(st);
            return FBR_OK;
        }
        const std::string msg = g_err;
        cudaError_t why = cudaSuccess;
        const bool died = worker_context_dead(p->workers[failed_worker], &why);
        if (died) on_worker_death(p, failed_worker, why);   // before free_seq: its parts on that worker are skipped
        free_seq(p, *st);
        if (!died) { g_err = msg; return rc; }
    }
    return fail(FBR_ECUDA, "submission kept failing while workers died");
}

static void harvest(fbr_pool* p, SeqState& st) {
    if (st.finished) return;
    st.sum = 0;
    st.sum_lo = 0;
    st.sum_hi = 0;
    unsigned long long err = ~0ull;
    for (auto& part : st.parts) {
        Worker& w = p->workers[part.worker];
        const SeqCtrl& c = w.h_ctrl[part.ctrl_slot];
        st.sum_lo += (uint64_t)c.sum;       // < 2^32 per task: cannot wrap below 2^32 tasks
        st.sum_hi += c.sum_hi;
        err = std::min(err, c.err);
        for (auto& t : part.t_dispatch) {
            float ms = 0;
            if (cudaEventElapsedTime(&ms, t.a, t.b) == cudaSuccess) p->stats.dispatch_ms += ms;
        }
        for (auto& t : part.t_gather) {
            float ms = 0;
            if (cudaEventElapsedTime(&ms, t.a, t.b) == cudaSuccess) p->stats.gather_ms += ms;
        }
    }
    {
        const __int128 total = (__int128)st.sum_hi * ((__int128)1 << 32) + (__int128)st.sum_lo;
        st.sum = (int64_t)(uint64_t)total;
        st.sum_overflow = total != (__int128)st.sum;
    }
    if (err != ~0ull) {
        st.err_code = (uint32_t)(err & 0xff);
        st.err_task = (uint64_t)(err >> 8);
    }
    st.finished = true;
    p->stats.tasks_completed += st.n_tasks;
    p->stats.units_redispatched += st.redispatched_units;
}

// the map cannot complete: a worker died under it and it was not (or could not be) re-dispatched
static int dead_map_error(fbr_pool* p, const SeqState& st) {
    return fail(FBR_ECUDA, "worker %d (CUDA device %d) died under map %llu: %s; %s", st.dead_worker, p->workers[st.dead_worker].device,
                (unsigned long long)st.seq, cudaGetErrorString((cudaError_t)st.dead_error),
                (st.flags & FBR_RESILIENT) ? "no surviving worker could take its blocks over"
                                           : "the pool was created without error_handling, so its blocks are not re-dispatched");
}

static int result_wait_locked_out(fbr_pool_t* p, uint64_t seq, int timeout_ms, fbr_result_t* res);

// A waiter blocks on CUDA events OUTSIDE the pool lock; a concurrent fbr_result_release must not destroy them under it.
// Waiters are counted per seq; a release that arrives meanwhile is deferred to the last waiter leaving.
int fbr_result_wait(fbr_pool_t* p, uint64_t seq, int timeout_ms, fbr_result_t* res) {
    if (!p || !res) return fail(FBR_EINVAL, "NULL argument");
    {
        std::lock_guard<std::mutex> g(p->mu);
        auto it = p->seqs.find(seq);
        if (it == p->seqs.end()) return fail(FBR_ENOENT, "unknown seq %llu", (unsigned long long)seq);
        it->second->waiters++;
    }
    const int rc = result_wait_locked_out(p, seq, timeout_ms, res);
    const std::string msg = rc != FBR_OK ? g_err : std::string();
    {
        std::lock_guard<std::mutex> g(p->mu);
        auto it = p->seqs.find(seq);
        if (it != p->seqs.end() && --it->second->waiters == 0 && it->second->release_pending) {
            harvest(p, *it->second);
            free_seq(p, *it->second);
            p->seqs.erase(it);
        }
    }
    if (rc != FBR_OK) g_err = msg;
    return rc;
}

static int result_wait_locked_out(fbr_pool_t* p, uint64_t seq, int timeout_ms, fbr_result_t* res) {
    const auto deadline = std::chrono::steady_clock::now() + std::chrono::milliseconds(timeout_ms < 0 ? 0 : timeout_ms);
    for (;;) {
        struct Ev { int worker, device; cudaEvent_t ev; };
        std::vector<Ev> evs;
        {
            std::lock_guard<std::mutex> g(p->mu);
            auto it = p->seqs.find(seq);
            if (it == p->seqs.end()) return fail(FBR_ENOENT, "unknown seq %llu", (unsigned long long)seq);
            if (it->second->dead_worker >= 0) return dead_map_error(p, *it->second);
            for (auto& part : it->second->parts) evs.push_back({part.worker, p->workers[part.worker].device, part.done});
        }
        // block outside the pool lock so other threads can keep submitting
        bool again = false;
        for (auto& e : evs) {
            cudaError_t q = cudaSetDevice(e.device);
            if (q == cudaSuccess) {
                if (timeout_ms < 0) {
                    q = cudaEventSynchronize(e.ev);
                } else {
                    for (;;) {
                        q = cudaEventQuery(e.ev);
                        if (q != cudaErrorNotReady) break;
                        if (std::chrono::steady_clock::now() >= deadline) return fail(FBR_ETIMEOUT, "timeout waiting for seq %llu", (unsigned long long)seq);
                        std::this_thread::sleep_for(std::chrono::microseconds(50));
                    }
                }
            }
            if (q != cudaSuccess) {
                // watchdog: is it the worker (sticky context error) or just this call?
                cudaGetLastError();
                std::lock_guard<std::mutex> g(p->mu);
                cudaError_t why = q;
                if (!worker_context_dead(p->workers[e.worker], &why))
                    return fail(FBR_ECUDA, "waiting for seq %llu on worker %d: %s", (unsigned long long)seq, e.worker, cudaGetErrorString(q));
                on_worker_death(p, e.worker, why);
                again = true;       // the map's parts changed (re-dispatched) or it is marked dead
                break;
            }
        }
        if (again) continue;
        std::lock_guard<std::mutex> g(p->mu);
        auto it = p->seqs.find(seq);
        if (it == p->seqs.end()) return fail(FBR_ENOENT, "seq released while waiting");
        SeqState& st = *it->second;
        if (st.dead_worker >= 0) return dead_map_error(p, st);
        // resilient maps: the round is over; re-dispatch what was lost, or copy the window back
        int more = 0;
        for (size_t i = 0; i < st.parts.size(); ++i) {
            SeqPart& part = st.parts[i];
            Worker& w = p->workers[part.worker];
            cudaError_t q = w.dead ? cudaErrorUnknown : cudaSetDevice(w.device);
            if (q == cudaSuccess) q = cudaEventQuery(part.done);
            if (q == cudaErrorNotReady) { cudaGetLastError(); more = 1; continue; }  // re-recorded by another waiter
            int rc = q == cudaSuccess ? resilient_advance(p, st, part) : FBR_ECUDA;
            if (rc < 0) {
                const std::string msg = g_err;
                cudaError_t why = q;
                if (!worker_context_dead(w, &why)) { g_err = msg; return rc; }
                on_worker_death(p, part.worker, why);     // st.parts is a different vector now
                more = 1;
                break;
            }
            more |= rc;
        }
        if (more) continue;
        harvest(p, st);
        memset(res, 0, sizeof *res);
        res->seq = seq;
        res->n_tasks = st.n_tasks;
        res->result_bytes = st.result_bytes;
        res->result_kind = st.result_kind;
        res->data = st.out;
        res->sum = st.sum;
        res->sum_lo = st.sum_lo;
        res->sum_hi = st.sum_hi;
        res->sum_overflow = st.sum_overflow ? 1u : 0u;
        res->err_code = st.err_code;
        res->err_task = st.err_task;
        res->n_waves = st.n_waves;
        if (st.err_code) return fail(FBR_ETASK, "task %llu failed with code %u in body %s", (unsigned long long)st.err_task, st.err_code, body_of(st.func_id)->name.c_str());
        return FBR_OK;
    }
}

int fbr_result_poll(fbr_pool_t* p, uint64_t seq, uint64_t* n_done) {
    if (!p || !n_done) return fail(FBR_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> g(p->mu);
    auto it = p->seqs.find(seq);
    if (it == p->seqs.end()) return fail(FBR_ENOENT, "unknown seq %llu", (unsigned long long)seq);
    SeqState& st = *it->second;
    if (st.dead_worker >= 0) return dead_map_error(p, st);
    // ordered progress: tasks [0, n_done) are final.  Blocks are contiguous per worker, so count
    // complete waves worker by worker and stop at the first incomplete one.
    uint64_t done = 0;
    for (size_t pi = 0; pi < st.parts.size(); ++pi) {
        SeqPart& part = st.parts[pi];
        Worker& w = p->workers[part.worker];
        cudaError_t q = w.dead ? cudaErrorUnknown : cudaSetDevice(w.device);
        if (q == cudaSuccess) q = cudaEventQuery(part.done);
        if (q != cudaSuccess && q != cudaErrorNotReady) {
            // watchdog (same as fbr_result_wait): a dead worker's blocks move to the survivors
            cudaGetLastError();
            cudaError_t why = q;
            if (!worker_context_dead(w, &why)) return fail(FBR_ECUDA, "polling seq %llu on worker %d: %s", (unsigned long long)seq, part.worker, cudaGetErrorString(q));
            on_worker_death(p, part.worker, why);
            if (st.dead_worker >= 0) return dead_map_error(p, st);
            break;                                        // progress so far stands; the next poll sees the new parts
        }
        cudaGetLastError();
        const bool part_finished = q == cudaSuccess;
        if (part.cx.resilient) {
            // results become visible only once no unit is lost any more; polling drives the rounds
            if (part_finished) {
                if (part.finalized) { done += part.count; continue; }
                int rc = resilient_advance(p, st, part);
                if (rc < 0) {
                    const std::string msg = g_err;
                    cudaError_t why = cudaSuccess;
                    if (!worker_context_dead(w, &why)) { g_err = msg; return rc; }
                    on_worker_death(p, part.worker, why);
                    if (st.dead_worker >= 0) return dead_map_error(p, st);
                }
            }
            break;
        }
        uint64_t part_done = 0;
        if (part.cx.full_window && !part.cx.out_dev && !part.cx.keep_on_device) {
            // the window reaches the host in one copy at the end: nothing is final before that
            if (part_finished) { done += part.count; continue; }
            break;
        }
        for (size_t i = 0; i < part.wave_done.size(); ++i) {
            if (cudaEventQuery(part.wave_done[i]) != cudaSuccess) break;
            part_done = part.wave_cum[i];
        }
        cudaGetLastError();
        done += part_done;
        if (part_done < part.count) break;
    }
    *n_done = done;
    return FBR_OK;
}

int fbr_result_data(fbr_pool_t* p, uint64_t seq, void** data) {
    if (!p || !data) return fail(FBR_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> g(p->mu);
    auto it = p->seqs.find(seq);
    if (it == p->seqs.end()) return fail(FBR_ENOENT, "unknown seq %llu", (unsigned long long)seq);
    *data = it->second->out;
    return FBR_OK;
}

int fbr_result_fetch(fbr_pool_t* p, uint64_t seq, uint64_t first, uint64_t count, void* host_dst) {
    if (!p || (!host_dst && count)) return fail(FBR_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> g(p->mu);
    auto it = p->seqs.find(seq);
    if (it == p->seqs.end()) return fail(FBR_ENOENT, "unknown seq %llu", (unsigned long long)seq);
    SeqState& st = *it->second;
    if (!(st.flags & FBR_RESULTS_ON_DEVICE)) return fail(FBR_EINVAL, "seq %llu does not keep its results on the device", (unsigned long long)seq);
    if (first + count > st.n_tasks) return fail(FBR_EINVAL, "range out of bounds");
    const uint64_t R = st.result_bytes;
    for (auto& part : st.parts) {
        const uint64_t lo = std::max(first, part.first), hi = std::min(first + count, part.first + part.count);
        if (lo >= hi) continue;
        Worker& w = p->workers[part.worker];
        CK(cudaSetDevice(w.device));
        CK(cudaEventSynchronize(part.done));
        CK(cudaMemcpyAsync((uint8_t*)host_dst + (lo - first) * R, part.cx.window_base + (lo - part.first) * R, (hi - lo) * R,
                           cudaMemcpyDeviceToHost, w.s_out));
        p->stats.d2h_bytes += (hi - lo) * R;
    }
    for (auto& part : st.parts) {
        CK(cudaSetDevice(p->workers[part.worker].device));
        CK(cudaStreamSynchronize(p->workers[part.worker].s_out));
    }
    return FBR_OK;
}

int fbr_result_release(fbr_pool_t* p, uint64_t seq) {
    if (!p) return fail(FBR_EINVAL, "NULL pool");
    std::lock_guard<std::mutex> g(p->mu);
    auto it = p->seqs.find(seq);
    if (it == p->seqs.end()) return fail(FBR_ENOENT, "unknown seq %llu", (unsigned long long)seq);
    if (it->second->waiters > 0) {        // another thread is blocked on this map's events: it frees the seq when it leaves
        it->second->release_pending = true;
        return FBR_OK;
    }
    harvest(p, *it->second);  // keeps the timing statistics of maps released without a wait
    free_seq(p, *it->second);
    p->seqs.erase(it);
    return FBR_OK;
}

int fbr_host_alloc(fbr_pool_t* p, uint64_t bytes, void** ptr) {
    if (!p || !ptr) return fail(FBR_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> g(p->mu);
    return pinned_acquire(p, bytes, ptr);
}

int fbr_host_free(fbr_pool_t* p, void* ptr) {
    if (!p) return fail(FBR_EINVAL, "NULL pool");
    std::lock_guard<std::mutex> g(p->mu);
    pinned_release(p, ptr);
    return FBR_OK;
}

int fbr_device_alloc(fbr_pool_t* p, int worker, uint64_t bytes, void** dptr) {
    if (!p || !dptr || worker < 0 || worker >= (int)p->workers.size()) return fail(FBR_EINVAL, "bad arguments");
    CK(cudaSetDevice(p->workers[worker].device));
    CK(cudaMalloc(dptr, bytes));
    return FBR_OK;
}

int fbr_device_free(fbr_pool_t* p, int worker, void* dptr) {
    if (!p || worker < 0 || worker >= (int)p->workers.size()) return fail(FBR_EINVAL, "bad arguments");
    CK(cudaSetDevice(p->workers[worker].device));
    CK(cudaFree(dptr));
    return FBR_OK;
}

int fbr_memcpy_h2d(fbr_pool_t* p, int worker, void* dptr, const void* src, uint64_t bytes) {
    if (!p || worker < 0 || worker >= (int)p->workers.size()) return fail(FBR_EINVAL, "bad arguments");
    Worker& w = p->workers[worker];
    CK(cudaSetDevice(w.device));
    CK(cudaMemcpyAsync(dptr, src, bytes, cudaMemcpyHostToDevice, w.s_in));
    CK(cudaStreamSynchronize(w.s_in));
    return FBR_OK;
}

int fbr_memcpy_d2h(fbr_pool_t* p, int worker, void* dst, const void* dptr, uint64_t bytes) {
    if (!p || worker < 0 || worker >= (int)p->workers.size()) return fail(FBR_EINVAL, "bad arguments");
    Worker& w = p->workers[worker];
    CK(cudaSetDevice(w.device));
    CK(cudaStreamSynchronize(w.s_comp));
    CK(cudaMemcpyAsync(dst, dptr, bytes, cudaMemcpyDeviceToHost, w.s_out));
    CK(cudaStreamSynchronize(w.s_out));
    return FBR_OK;
}

int fbr_payload_fill_device(fbr_pool_t* p, int worker, void* dptr, uint64_t t0, uint64_t n) {
    if (!p || !dptr || worker < 0 || worker >= (int)p->workers.size()) return fail(FBR_EINVAL, "bad arguments");
    std::lock_guard<std::mutex> g(p->mu);
    Worker& w = p->workers[worker];
    CK(cudaSetDevice(w.device));
    const uint64_t n_vec = n * (kPayloadBytes / 16);
    const int grid = (int)std::max<uint64_t>(1, std::min<uint64_t>((n_vec + kThreads - 1) / kThreads, (uint64_t)w.sm_count * w.occ_fill));
    payload_fill_kernel<<<grid, kThreads, 0, w.s_comp>>>((uint4*)dptr, t0, n_vec);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(w.s_comp));
    p->stats.fill_launches++;
    return FBR_OK;
}

int fbr_pool_stats(fbr_pool_t* p, fbr_stats_t* s) {
    if (!p || !s) return fail(FBR_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> g(p->mu);
    *s = p->stats;
    return FBR_OK;
}

int fbr_pool_stats_reset(fbr_pool_t* p) {
    if (!p) return fail(FBR_EINVAL, "NULL pool");
    std::lock_guard<std::mutex> g(p->mu);
    memset(&p->stats, 0, sizeof p->stats);
    return FBR_OK;
}

}  // extern "C"
