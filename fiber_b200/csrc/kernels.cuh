// kernels.cuh -- the sm_100a kernels of the Pool.map hot path.
//
//   dispatch_*_kernel  : persistent CTAs claim fixed-layout task records from the device task ring
//                        by atomic ticket, run the mapped body, and write the unit's results plus a
//                        16 B header into the paired slot of the result ring.
//                        Replaces _handle_tasks + PUSH/PULL + zpool_worker_core
//                        (fiber/pool.py:952-963, 783-824).
//   gather_ordered_kernel : result ring -> ordered output by index placement, optional sum
//                        epilogue.  Replaces result_conn.send xN + _res_get + Inventory.get
//                        (fiber/pool.py:814-824, 968-973, 666-679).
//   payload_fill_kernel : synthetic 4 KB records for BASELINE.json config 4.
//
// Everything here is HBM-bound byte/integer work (no dense contraction => no tensor cores):
// 16 B vector accesses, fully coalesced, grids sized as (SM count x resident CTAs).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include <type_traits>

#include "bodies.cuh"

namespace fbr {

constexpr int kThreads = 256;

// One claim unit = `count` consecutive tasks of one map.  32 B, written by the host into the
// pinned task ring and copied to the device ring with cudaMemcpyAsync.  It is the fixed-layout
// stand-in for the reference's pickled task tuple (seq, batch_start, func, chunk, starmap)
// (fiber/pool.py:1181).
struct TaskRecord {
    uint32_t seq;       // map id (Inventory seq, fiber/pool.py:659-664), low 32 bits
    uint32_t count;     // tasks in this unit
    uint64_t first;     // index of the unit's first task inside the map (the reference's `batch`)
    uint64_t arg_off;   // byte offset of the unit's first argument record in the wave's arg ring
    uint32_t func_id;
    uint32_t attempt;   // re-dispatch count (resilient pool)
};
static_assert(sizeof(TaskRecord) == 32, "task record layout is part of the ABI");

// Header of a result-ring slot: the fixed-layout stand-in for the reference's per-item result
// message (seq, batch, batch + i, res) (fiber/pool.py:814,821), one per unit instead of per item.
struct SlotHeader {
    uint32_t seq;
    uint32_t count;     // bit 31: unit lost (its worker "died"), must be re-dispatched
    uint64_t first;
};
static_assert(sizeof(SlotHeader) == 16, "slot header layout is part of the ABI");
constexpr uint32_t kUnitLost = 0x80000000u;

struct WaveParams {
    const TaskRecord* records;  // device task ring window of this wave; nullptr: the wave is a contiguous,
                                // unshuffled block and unit t's record is computed from the syn_* fields below
                                // (an arithmetic progression needs no 32 B/unit of PCIe traffic)
    SlotHeader* headers;        // result ring headers (paired with records by ticket); nullptr: direct placement --
                                // `ring` IS the ordered output window and slot t lands at its final index, no gather
    uint8_t* ring;              // result ring payload arena (or the ordered output window, see headers)
    uint32_t* ticket;           // device counter, zero at launch
    uint32_t n_units;
    uint32_t slot_stride;       // bytes, multiple of 16
    const uint8_t* args;        // device argument ring window (arg_off is relative to it)
    uint32_t arg_stride;        // 0 => implicit index arguments
    int64_t index_start, index_step;
    uint64_t index_base;        // global index of the map's task 0
    const uint8_t* shared;      // broadcast argument block
    uint64_t shared_bytes;
    unsigned long long* err_word;
    uint32_t resilient;         // lost units are re-dispatched by the host (else a fault is an error)
    long long* sum;             // fold sum(results) here (nullptr: no fold); done where the values are in registers.
                                // 8-byte results: sum of the LOW 32-bit halves (as unsigned) ...
    long long* sum_hi;          // ... and sum of the high halves (arithmetic >> 32) here: the exact, unbounded sum
                                // is sum_hi * 2^32 + sum, whatever the int64 total would have wrapped to
    // synthesised records (records == nullptr): unit t = tasks [syn_first + t*syn_unit, ...) of map syn_seq
    uint64_t syn_first;         // map index of the wave's first task
    uint64_t syn_tasks;         // tasks in the wave
    uint64_t syn_arg_off;       // arg_off of unit 0
    uint32_t syn_unit;          // tasks per unit
    uint32_t syn_seq;
    uint32_t syn_func;
    uint32_t syn_attempt;       // re-dispatch count of the whole wave (a dead worker's block re-run elsewhere)
    uint64_t n_items;           // bodies whose task consumes several argument items (bit-packed bool twins: 8 per
                                // task): number of items of the whole map, items at or past it are not read
};

// Task record of ticket t: from the device task ring, or computed (contiguous wave).
__device__ __forceinline__ TaskRecord wave_record(const WaveParams& wp, uint32_t t) {
    if (wp.records != nullptr) return wp.records[t];
    const uint64_t off = (uint64_t)t * wp.syn_unit;
    const uint64_t left = wp.syn_tasks - off;
    TaskRecord r;
    r.seq = wp.syn_seq;
    r.count = left < (uint64_t)wp.syn_unit ? (uint32_t)left : wp.syn_unit;
    r.first = wp.syn_first + off;
    r.arg_off = wp.syn_arg_off + off * (uint64_t)wp.arg_stride;
    r.func_id = wp.syn_func;
    r.attempt = wp.syn_attempt;
    return r;
}
__device__ __forceinline__ void put_header(const WaveParams& wp, uint32_t t, const SlotHeader& h) {
    if (wp.headers != nullptr) wp.headers[t] = h;
}

// ------------------------------------------------------------------------------------------------
// streaming 16 B accesses
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 ld_stream(const void* p) { return __ldcs(reinterpret_cast<const uint4*>(p)); }
__device__ __forceinline__ void st_vec(void* p, const uint4& v) { *reinterpret_cast<uint4*>(p) = v; }

// Ticket claim with prefetch: thread 0 holds the next ticket while the CTA works on the current
// one, so the ~700-cycle L2 atomic round trip is off the critical path.
struct TicketClaimer {
    uint32_t* counter;
    uint32_t next;  // valid in thread 0 only
    __device__ __forceinline__ void prime() {
        if (threadIdx.x == 0) next = atomicAdd(counter, 1u);
    }
    // returns the ticket for this iteration (uniform across the CTA) and prefetches the following one
    __device__ __forceinline__ uint32_t claim(uint32_t* s_slot) {
        __syncthreads();  // previous iteration's readers of *s_slot are done
        if (threadIdx.x == 0) {
            *s_slot = next;
            next = atomicAdd(counter, 1u);
        }
        __syncthreads();
        return *s_slot;
    }
    // Re-arm the counter for the wave that uses it next.  Every CTA draws exactly two tickets >= n_units (the
    // one that ends its loop and the one prefetched behind it), so n_units + 2*gridDim.x atomics happen in
    // all, and the highest value is always a prefetched, unused one: its holder knows every other atomic
    // has been performed and zeroes the counter (no memset node, no gather kernel needed for it).
    __device__ __forceinline__ void rearm(uint32_t n_units) {
        if (threadIdx.x == 0 && next == n_units + 2u * gridDim.x - 1u) *counter = 0u;
    }
    // one-barrier variant: `s_slots[2]` is indexed by iteration parity (see dispatch_thread_kernel)
    __device__ __forceinline__ uint32_t claim_db(uint32_t* s_slots, uint32_t iter) {
        if (threadIdx.x == 0) {
            s_slots[iter & 1] = next;
            next = atomicAdd(counter, 1u);
        }
        __syncthreads();
        return s_slots[iter & 1];
    }
};

// Fold one value per thread into a global accumulator: warp shuffle, then one atomic per warp (no
// block barrier: a __syncthreads() after the persistent loop made ptxas restructure the whole loop,
// +15 % instructions on the pi body).
// (unsigned arithmetic throughout: two's-complement wrap-around is defined, signed overflow is not)
__device__ __forceinline__ void warp_add(unsigned long long v, long long* target) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0 && v != 0) atomicAdd(reinterpret_cast<unsigned long long*>(target), v);
}

// ================================================================================================
// dispatch: ThreadBody -- one thread per task, V = 16/sizeof(Res) consecutive tasks per thread so
// each thread emits one 16 B store; a warp writes 512 contiguous bytes of the ring slot.
// ================================================================================================
// The slice of one unit that thread `vt` (0..kThreads-1) of the unit's thread grid owns: vectors
// vt, vt + kThreads, ...  Adds the slice's results to unit_acc / unit_acc32.
template <class B, bool kIndex>
__device__ __forceinline__ void run_unit_slice(const WaveParams& wp, const TaskRecord& rec, uint8_t* slot, uint32_t vt,
                                               const ErrSink& es, unsigned long long& unit_acc, unsigned long long& unit_hi,
                                               uint32_t& unit_acc32) {
    using Arg = typename B::Arg;
    using Res = typename B::Res;
    constexpr int V = (sizeof(Res) >= 16) ? 1 : (16 / (int)sizeof(Res));
    const uint8_t* uargs = wp.args + rec.arg_off;
    for (uint32_t base = vt * V; base < rec.count; base += kThreads * V) {
        // implicit range() argument: one multiply per thread, then strength-reduced adds
        // (keeps the integer-multiply pipe for the body: Philox needs 18 IMAD.WIDE per task)
        int64_t a_idx = 0;
        if constexpr (kIndex) a_idx = wp.index_start + (int64_t)(rec.first + base) * wp.index_step;
        const uint64_t gidx0 = wp.index_base + rec.first + base;
        uint8_t* dst = slot + (size_t)base * sizeof(Res);
        if (base + V <= rec.count) {
            // full vector: no per-task bounds checks (a branch per task cost 6 instructions and
            // serialised the tasks' dependency chains); results are packed into one 16 B
            // register vector (no local-memory staging)
            uint32_t pk[4] = {0u, 0u, 0u, 0u};
            if constexpr (kIndex && B::kVecIndex) {
                B::template run_index_vec<V>(a_idx, wp.index_step, pk);
            } else {
#pragma unroll
                for (int v = 0; v < V; ++v) {
                    Arg a;
                    if constexpr (kIndex) { a = (Arg)a_idx; a_idx += wp.index_step; }
                    else a = *reinterpret_cast<const Arg*>(uargs + (size_t)(base + v) * wp.arg_stride);
                    const Res r = B::run(a, gidx0 + v, es, rec.attempt);
                    if constexpr (sizeof(Res) == 1) {
                        pk[v >> 2] |= (uint32_t)(uint8_t)r << ((v & 3) * 8);
                    } else if constexpr (sizeof(Res) == 8) {
                        unsigned long long bits;
                        memcpy(&bits, &r, 8);
                        unit_acc += bits & 0xffffffffull;
                        unit_hi += (unsigned long long)((long long)bits >> 32);
                        pk[2 * v] = (uint32_t)bits;
                        pk[2 * v + 1] = (uint32_t)(bits >> 32);
                    } else {
                        static_assert(sizeof(Res) == 1 || sizeof(Res) == 8, "add a packing rule for this result size");
                    }
                }
            }
            if constexpr (sizeof(Res) == 1) {     // byte results: fold the packed words with dp4a
                uint32_t s4 = __dp4a(pk[0], 0x01010101u, 0u);
                s4 = __dp4a(pk[1], 0x01010101u, s4);
                s4 = __dp4a(pk[2], 0x01010101u, s4);
                s4 = __dp4a(pk[3], 0x01010101u, s4);
                unit_acc32 += s4;
            }
            st_vec(dst, make_uint4(pk[0], pk[1], pk[2], pk[3]));
        } else {
            // the unit's partial tail vector (at most one per unit): one task at a time, kept
            // rolled so the kernel holds a single copy of the unrolled body
#pragma unroll 1
            for (uint32_t i = base; i < rec.count; ++i) {
                Arg a;
                if constexpr (kIndex) { a = (Arg)a_idx; a_idx += wp.index_step; }
                else a = *reinterpret_cast<const Arg*>(uargs + (size_t)i * wp.arg_stride);
                const Res r = B::run(a, gidx0 + (i - base), es, rec.attempt);
                if constexpr (sizeof(Res) == 1) unit_acc32 += (uint32_t)(uint8_t)r;
                else if constexpr (sizeof(Res) == 8) {
                    unsigned long long bits;
                    memcpy(&bits, &r, 8);
                    unit_acc += bits & 0xffffffffull;
                    unit_hi += (unsigned long long)((long long)bits >> 32);
                }
                memcpy(dst + (size_t)(i - base) * sizeof(Res), &r, sizeof(Res));
            }
        }
    }
}

// kIndex: the task index itself is the argument (range()); a separate instantiation keeps each
// kernel to one copy of the unrolled body (the two-path version was 45 KB of SASS, beyond the 32 KB
// instruction cache level).
//
// One barrier per unit: the ticket slot (and, for bodies that can lose a unit, the fault flag) is
// double-buffered by iteration parity, so the write of iteration i+2 is ordered after the reads of
// iteration i by the barrier of iteration i+1.  (Three barriers per 4096-task unit were 5 % of the
// pi kernel's stall samples.  Tried and dropped: warp-granular claims with no barrier at all --
// 0.2689 ms against 0.2654 ms on the 1e8-task pi wave; the skew between a CTA's warps is not what
// limits this kernel.)
template <class B, bool kIndex>
__global__ void __launch_bounds__(kThreads) dispatch_thread_kernel(const WaveParams wp) {
    __shared__ uint32_t s_ticket[2];
    __shared__ int s_fault[2];
    if (threadIdx.x == 0) { s_fault[0] = 0; s_fault[1] = 0; }
    TicketClaimer tc{wp.ticket, 0u};
    tc.prime();
    unsigned long long acc = 0, acc_hi = 0;   // sums of this thread's results over every unit its CTA completed
    for (uint32_t iter = 0;; ++iter) {
        const uint32_t t = tc.claim_db(s_ticket, iter);
        if (t >= wp.n_units) break;
        int* const unit_fault = &s_fault[iter & 1];
        const ErrSink es{wp.err_word, unit_fault};
        const TaskRecord rec = wave_record(wp, t);
        unsigned long long unit_acc = 0, unit_hi = 0;
        uint32_t unit_acc32 = 0;
        run_unit_slice<B, kIndex>(wp, rec, wp.ring + (size_t)t * wp.slot_stride, threadIdx.x, es, unit_acc, unit_hi, unit_acc32);
        bool lost = false;
        if constexpr (B::kCanFault) {
            __syncthreads();      // every thread's fault reports for this unit are in
            lost = *unit_fault != 0;
            // re-arm the other flag for the next unit: its last readers ran before this barrier,
            // its next writers run after the next claim barrier
            if (threadIdx.x == 0) s_fault[(iter + 1) & 1] = 0;
        }
        if (!lost) {                                          // a lost unit is re-dispatched: never folded twice
            acc += unit_acc + unit_acc32;
            acc_hi += unit_hi;
        }
        if (threadIdx.x == 0) {
            // A dead worker loses its whole chunk.  ResilientZPool re-queues it; in the plain ZPool
            // the map would hang forever (fiber/pool.py:801-824 has no try/except) -- here it is
            // reported as a task error instead.
            if (lost && !wp.resilient)
                atomicMin(wp.err_word, (unsigned long long)(((wp.index_base + rec.first) << 8) | TASK_FAULT));
            put_header(wp, t, SlotHeader{rec.seq, rec.count | ((lost && wp.resilient) ? kUnitLost : 0u), rec.first});
        }
    }
    tc.rearm(wp.n_units);
    if (wp.sum != nullptr) {
        warp_add(acc, wp.sum);
        if constexpr (sizeof(typename B::Res) == 8) warp_add(acc_hi, wp.sum_hi);
    }
}

// ================================================================================================
// dispatch: pi_inside_bits8 -- task g is the 8 range() indices 8g..8g+7, its result one byte (bit k =
// is_inside(index 8g+k)).  A thread owns two consecutive bytes of the unit (16 indices, the same
// Philox vector as the byte-result kernel) and stores them as one uint16; a warp writes 64
// contiguous bytes.  Algorithmic bytes per index: 0 read + 1/8 written.
// ================================================================================================
__global__ void __launch_bounds__(kThreads) dispatch_pi_bits_kernel(const WaveParams wp) {
    __shared__ uint32_t s_ticket[2];
    TicketClaimer tc{wp.ticket, 0u};
    tc.prime();
    unsigned long long acc = 0;
    for (uint32_t iter = 0;; ++iter) {
        const uint32_t t = tc.claim_db(s_ticket, iter);
        if (t >= wp.n_units) break;
        const TaskRecord rec = wave_record(wp, t);
        uint8_t* slot = wp.ring + (size_t)t * wp.slot_stride;
        for (uint32_t b = threadIdx.x * 2; b < rec.count; b += kThreads * 2) {
            const int64_t a0 = wp.index_start + (int64_t)((rec.first + b) * 8ull) * wp.index_step;
            const uint32_t bits = PiInsideDet::run_index_bits16(a0, wp.index_step);
            if (b + 2 <= rec.count) {
                *reinterpret_cast<uint16_t*>(slot + b) = (uint16_t)bits;
                acc += __popc(bits);
            } else {                                  // odd byte count: the unit's last byte
                slot[b] = (uint8_t)bits;
                acc += __popc(bits & 0xffu);
            }
        }
        if (threadIdx.x == 0) put_header(wp, t, SlotHeader{rec.seq, rec.count, rec.first});
    }
    tc.rearm(wp.n_units);
    if (wp.sum != nullptr) warp_add(acc, wp.sum);
}

// ================================================================================================
// dispatch: bit-packed twin of ANY bool ThreadBody: 8 items per byte-task, items being explicit argument
// records (B::Arg, kIndex = false) or range() indices (kIndex = true: item i is index_start + i*index_step,
// no argument bytes).  A warp takes 512 consecutive items per pass: lane l evaluates items l, l+32, ...
// (each load instruction reads 32 consecutive records: fully coalesced), and the ballot of pass j IS word j
// of the warp's 64 output bytes (bit l = lane l's result = item 32j + l) -- no shuffles, no transposes.
// Lanes 0..15 store the 16 words: 64 contiguous bytes per warp.  Items at or past wp.n_items are not
// evaluated and leave zero bits.  Algorithmic bytes per item: sizeof(Arg) read + 1/8 written.
// ================================================================================================
template <class B, bool kIndex = false>
__global__ void __launch_bounds__(kThreads) dispatch_bits_items_kernel(const WaveParams wp) {
    using Arg = typename B::Arg;
    static_assert(!B::kCanFault, "bit-packed twins are for bodies that cannot lose a unit");
    __shared__ uint32_t s_ticket[2];
    __shared__ int s_fault;
    TicketClaimer tc{wp.ticket, 0u};
    tc.prime();
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const ErrSink es{wp.err_word, &s_fault};
    unsigned long long acc = 0;
    for (uint32_t iter = 0;; ++iter) {
        const uint32_t t = tc.claim_db(s_ticket, iter);
        if (t >= wp.n_units) break;
        const TaskRecord rec = wave_record(wp, t);
        uint8_t* slot = wp.ring + (size_t)t * wp.slot_stride;
        const uint8_t* uargs = wp.args + rec.arg_off;
        const uint64_t item0 = rec.first * 8ull;                       // map-level index of the unit's first item
        const uint32_t n_it = rec.count * 8u;                          // items covered by this unit's bytes
        for (uint32_t base = warp * 512u; base < n_it; base += (kThreads / 32) * 512u) {
            uint32_t mine = 0u;                                        // word `lane` of this pass block (lanes 0..15)
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const uint32_t i = base + 32u * j + lane;
                bool r = false;
                if (i < n_it && item0 + i < wp.n_items) {
                    Arg a;
                    if constexpr (kIndex) a = (Arg)(wp.index_start + (int64_t)(item0 + i) * wp.index_step);
                    else a = *reinterpret_cast<const Arg*>(uargs + (size_t)i * sizeof(Arg));
                    r = B::run(a, wp.index_base + item0 + i, es, rec.attempt) != 0;
                }
                const uint32_t word = __ballot_sync(0xffffffffu, r);
                if (lane == (uint32_t)j) mine = word;
            }
            if (lane < 16) {
                const uint32_t byte0 = (base >> 3) + lane * 4u;            // this word's first byte inside the slot
                if (byte0 + 4u <= rec.count) {
                    *reinterpret_cast<uint32_t*>(slot + byte0) = mine;
                } else {
                    for (uint32_t b = byte0; b < rec.count; ++b) slot[b] = (uint8_t)(mine >> ((b - byte0) * 8u));
                }
                acc += __popc(mine);
            }
        }
        if (threadIdx.x == 0) put_header(wp, t, SlotHeader{rec.seq, rec.count, rec.first});
    }
    tc.rearm(wp.n_units);
    if (wp.sum != nullptr) warp_add(acc, wp.sum);
}

// ================================================================================================
// dispatch: payload_map_4k -- a CTA streams its unit's 4 KB records: thread j owns the j-th 16 B
// column of every record, 4 records in flight per thread (16 KB per CTA in flight).
//   out[w] = in[w] * 2654435761 + t   (u32 wrap), t = global task index.
// Algorithmic bytes per task: 4096 read + 4096 written.
// ================================================================================================
__global__ void __launch_bounds__(kThreads) dispatch_payload_map_kernel(const WaveParams wp) {
    __shared__ uint32_t s_ticket;
    TicketClaimer tc{wp.ticket, 0u};
    tc.prime();
    constexpr int U = 4;
    for (;;) {
        const uint32_t t = tc.claim(&s_ticket);
        if (t >= wp.n_units) break;
        const TaskRecord rec = wave_record(wp, t);
        const uint8_t* src = wp.args + rec.arg_off + threadIdx.x * 16;
        uint8_t* dst = wp.ring + (size_t)t * wp.slot_stride + threadIdx.x * 16;
        const uint32_t tbase = (uint32_t)(wp.index_base + rec.first);
        uint32_t r = 0;
        for (; r + U <= rec.count; r += U) {
            uint4 v[U];
#pragma unroll
            for (int u = 0; u < U; ++u) v[u] = ld_stream(src + (size_t)(r + u) * wp.arg_stride);
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const uint32_t tt = tbase + r + u;
                v[u].x = v[u].x * kPayloadMul + tt;
                v[u].y = v[u].y * kPayloadMul + tt;
                v[u].z = v[u].z * kPayloadMul + tt;
                v[u].w = v[u].w * kPayloadMul + tt;
                st_vec(dst + (size_t)(r + u) * kPayloadBytes, v[u]);
            }
        }
        for (; r < rec.count; ++r) {
            uint4 v = ld_stream(src + (size_t)r * wp.arg_stride);
            const uint32_t tt = tbase + r;
            v.x = v.x * kPayloadMul + tt; v.y = v.y * kPayloadMul + tt;
            v.z = v.z * kPayloadMul + tt; v.w = v.w * kPayloadMul + tt;
            st_vec(dst + (size_t)r * kPayloadBytes, v);
        }
        if (threadIdx.x == 0) put_header(wp, t, SlotHeader{rec.seq, rec.count, rec.first});
    }
    tc.rearm(wp.n_units);
}

// ================================================================================================
// dispatch: payload_checksum_4k -- one warp per record, 8 coalesced 16 B loads per lane, shuffle
// reduce, lane 0 stores the u32.  Algorithmic bytes per task: 4096 read + 4 written.
// ================================================================================================
__global__ void __launch_bounds__(kThreads) dispatch_payload_checksum_kernel(const WaveParams wp) {
    __shared__ uint32_t s_ticket;
    TicketClaimer tc{wp.ticket, 0u};
    tc.prime();
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    unsigned long long acc = 0;
    for (;;) {
        const uint32_t t = tc.claim(&s_ticket);
        if (t >= wp.n_units) break;
        const TaskRecord rec = wave_record(wp, t);
        uint32_t* dst = reinterpret_cast<uint32_t*>(wp.ring + (size_t)t * wp.slot_stride);
        for (uint32_t r = warp; r < rec.count; r += kThreads / 32) {
            const uint8_t* src = wp.args + rec.arg_off + (size_t)r * wp.arg_stride + lane * 16;
            uint4 v[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) v[k] = ld_stream(src + k * 512);
            uint32_t s = 0;
#pragma unroll
            for (int k = 0; k < 8; ++k) s += v[k].x + v[k].y + v[k].z + v[k].w;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if (lane == 0) { dst[r] = s; acc += s; }
        }
        if (threadIdx.x == 0) put_header(wp, t, SlotHeader{rec.seq, rec.count, rec.first});
    }
    tc.rearm(wp.n_units);
    if (wp.sum != nullptr) warp_add(acc, wp.sum);
}

// ================================================================================================
// dispatch: parzen -- a CTA per task: every thread tests samples j, j+256, ... against the window
// (samples are read from the broadcast block, L2-resident after the first task), block-reduce the
// count, thread 0 emits (h, (k/n)/h**power).  Algorithmic bytes per task: n*dims*sizeof(T) read
// (from L2), 16 written.
// ================================================================================================
template <typename T>
__global__ void __launch_bounds__(kThreads) dispatch_parzen_kernel(const WaveParams wp) {
    __shared__ uint32_t s_ticket;
    __shared__ uint32_t s_warp[kThreads / 32];
    TicketClaimer tc{wp.ticket, 0u};
    tc.prime();
    const ParzenShared sh = *reinterpret_cast<const ParzenShared*>(wp.shared);
    const T* samples = reinterpret_cast<const T*>(wp.shared + sizeof(ParzenShared));
    for (;;) {
        const uint32_t t = tc.claim(&s_ticket);
        if (t >= wp.n_units) break;
        const TaskRecord rec = wave_record(wp, t);
        double* dst = reinterpret_cast<double*>(wp.ring + (size_t)t * wp.slot_stride);
        for (uint32_t i = 0; i < rec.count; ++i) {
            const double h = *reinterpret_cast<const double*>(wp.args + rec.arg_off + (size_t)i * wp.arg_stride);
            const T hT = (T)h;
            uint32_t k = 0;
            if (sh.dims == 2) {
                // 4 independent sample loads in flight per thread (the block is L2-resident: ~40 dependent
                // L2 round trips per task otherwise), then the divides
                constexpr int U = 4;
                using V2 = typename std::conditional<sizeof(T) == 4, float2, double2>::type;
                const V2* s2 = reinterpret_cast<const V2*>(samples);
                uint32_t j = threadIdx.x;
                for (; j + (U - 1) * kThreads < sh.n_samples; j += U * kThreads) {
                    V2 v[U];
#pragma unroll
                    for (int u = 0; u < U; ++u) v[u] = s2[j + u * kThreads];
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        const T row[2] = {v[u].x, v[u].y};
                        k += parzen_inside<T>(row, sh, hT) ? 1u : 0u;
                    }
                }
                for (; j < sh.n_samples; j += kThreads) {
                    const V2 v = s2[j];
                    const T row[2] = {v.x, v.y};
                    k += parzen_inside<T>(row, sh, hT) ? 1u : 0u;
                }
            } else {
                for (uint32_t j = threadIdx.x; j < sh.n_samples; j += kThreads)
                    k += parzen_inside<T>(samples + (size_t)j * sh.dims, sh, hT) ? 1u : 0u;
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) k += __shfl_xor_sync(0xffffffffu, k, o);
            if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = k;
            __syncthreads();
            if (threadIdx.x == 0) {
                uint32_t kn = 0;
                for (int w = 0; w < kThreads / 32; ++w) kn += s_warp[w];
                // (k_n / len(x_samples)) / (h ** point_x.shape[1]), float64 like the reference
                double hp = 1.0;
                for (uint32_t e = 0; e < sh.power; ++e) hp = __dmul_rn(hp, h);
                dst[2 * i] = h;
                dst[2 * i + 1] = __ddiv_rn(__ddiv_rn((double)kn, (double)sh.n_samples), hp);
            }
            __syncthreads();
        }
        if (threadIdx.x == 0) put_header(wp, t, SlotHeader{rec.seq, rec.count, rec.first});
    }
    tc.rearm(wp.n_units);
}

// ================================================================================================
// gather_ordered: result ring -> ordered output by index placement (fiber/pool.py:672).  The ring
// holds one slot per claim unit in task-record (arrival) order; each slot's header says which
// tasks it carries.  Three kernels, picked per wave by the host:
//
//   gather_bulk_kernel     TMA path (cp.async.bulk, UBLKCP in SASS) for slots of >= 4 KB whose units
//                          are all valid: one elected thread per CTA pipelines
//                          ring --bulk load--> shared stage --bulk store--> output; no payload byte
//                          touches a register.  8.2 GB payload wave: 104 % of the measured HBM copy
//                          peak with ONE CTA of one warp per SM.
//   gather_rows_kernel     slots made of whole 4 KB rows, any unit state (lost units skipped and
//                          listed for re-dispatch, partial tail vector copied byte-wise).
//   gather_ordered_kernel  flat per-vector kernel for small or unaligned slots.
//
// The sum(results) fold lives in the dispatch kernels (where the values are in registers).
// Algorithmic bytes per task: R read + R written.
// ================================================================================================
struct LostUnit { uint64_t first; uint32_t count; uint32_t pad; };

struct GatherParams {
    const SlotHeader* headers;
    const uint8_t* ring;
    uint32_t n_units;
    uint32_t slot_stride;     // bytes, multiple of 16
    uint32_t result_bytes;    // R
    uint32_t pad;
    uint8_t* out;             // ordered output window
    uint64_t win_first;       // map index of out[0]
    uint32_t* ticket_to_reset;  // dispatch ticket of this wave, zeroed for its next use
    uint32_t* lost_count;     // device: number of lost units appended so far (nullable)
    LostUnit* lost_units;     // device: (first, count) of every lost unit, for re-dispatch
    uint32_t lost_capacity;
};

__device__ __forceinline__ SlotHeader ld_header(const SlotHeader* p) {
    const uint4 r = __ldg(reinterpret_cast<const uint4*>(p));
    SlotHeader h;
    h.seq = r.x; h.count = r.y; h.first = ((uint64_t)r.w << 32) | (uint64_t)r.z;
    return h;
}

__device__ __forceinline__ void copy_tail_bytes(uint8_t* dst, const uint4& data, uint32_t nb) {
    const uint32_t w[4] = {data.x, data.y, data.z, data.w};
    for (uint32_t b = 0; b < nb; ++b) dst[b] = (uint8_t)(w[b >> 2] >> ((b & 3) * 8));
}

// housekeeping shared by the gather kernels: re-arm the wave's dispatch ticket, list lost units
__device__ __forceinline__ void gather_epilogue(const GatherParams& gp, uint32_t tid, uint32_t nthreads) {
    if (tid == 0 && gp.ticket_to_reset) *gp.ticket_to_reset = 0u;
    if (gp.lost_count != nullptr) {
        for (uint32_t s = tid; s < gp.n_units; s += nthreads) {
            const SlotHeader h = gp.headers[s];
            if (h.count & kUnitLost) {
                const uint32_t k = atomicAdd(gp.lost_count, 1u);
                if (k < gp.lost_capacity) gp.lost_units[k] = LostUnit{h.first, h.count & ~kUnitLost, 0u};
            }
        }
    }
}

// ---- flat: one 16 B vector per thread-iteration ------------------------------------------------
__global__ void __launch_bounds__(kThreads) gather_ordered_kernel(const GatherParams gp) {
    // slot_stride == vps * 16, so ring vector v lives at ring + 16*v: the slot number is only
    // needed to find the header (destination), never for the source address.
    const uint32_t vps = gp.slot_stride >> 4;                   // vectors per slot
    const uint32_t total = gp.n_units * vps;                    // host guarantees < 2^32
    const int sh = (vps & (vps - 1)) == 0 ? (31 - __clz(vps)) : -1;
    constexpr int U = 4;
    constexpr uint32_t kTile = kThreads * U;                    // 16 KB of ring per CTA iteration

    // Resolve the destination while the data load is still in flight: per vector we keep only the
    // destination pointer and the number of valid bytes (0 = skip: lost unit / beyond the tail).
    auto resolve = [&](uint32_t v, uint8_t*& dst) -> uint32_t {
        const uint32_t slot = sh >= 0 ? (v >> sh) : (v / vps);
        const uint32_t within = v - slot * vps;
        const SlotHeader h = ld_header(gp.headers + slot);
        const uint64_t valid = (uint64_t)(h.count & ~kUnitLost) * gp.result_bytes;
        const uint64_t off = (uint64_t)within << 4;
        dst = gp.out + (h.first - gp.win_first) * gp.result_bytes + off;
        if ((h.count & kUnitLost) || off >= valid) return 0u;
        const uint32_t nb = (valid - off) < 16 ? (uint32_t)(valid - off) : 16u;
        // an unaligned destination takes the byte path as well (flagged in bit 8)
        return nb | (((reinterpret_cast<uintptr_t>(dst) & 15) != 0) ? 0x100u : 0u);
    };

    for (uint32_t base = blockIdx.x * kTile; base < total; base += gridDim.x * kTile) {
        uint4 data[U];
        uint8_t* dst[U];
        uint32_t nbf[U];
        const uint32_t v0 = base + threadIdx.x;
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint32_t v = v0 + u * kThreads;
            nbf[u] = 0u;
            if (v < total) {
                data[u] = ld_stream(gp.ring + ((size_t)v << 4));
                nbf[u] = resolve(v, dst[u]);
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (nbf[u] == 16u) st_vec(dst[u], data[u]);
            else if (nbf[u] != 0u) copy_tail_bytes(dst[u], data[u], nbf[u] & 0xffu);
        }
    }
    gather_epilogue(gp, blockIdx.x * kThreads + threadIdx.x, gridDim.x * kThreads);
}

// ---- rows: a CTA claims ~128 KB of ring by ticket and streams it as 4 KB rows ---------------------
// Thread j owns the j-th 16 B column of every row, 4 rows in flight.  Measured on the 8.2 GB payload
// wave: 99.8 % of the HBM copy peak (the flat kernel: 92 %).
__global__ void __launch_bounds__(kThreads) gather_rows_kernel(const GatherParams gp, uint32_t* ticket, uint32_t group_slots, bool reverse) {
    __shared__ uint32_t s_ticket;
    TicketClaimer tc{ticket, 0u};
    tc.prime();
    constexpr int U = 4;
    const uint32_t rps = gp.slot_stride >> 12;                          // 4 KB rows per slot
    const int sh = (rps & (rps - 1)) == 0 ? (31 - __clz(rps)) : -1;
    const uint32_t n_groups = (gp.n_units + group_slots - 1) / group_slots;

    auto place = [&](const uint4& data, uint32_t slot, uint32_t row_in_slot) {
        const SlotHeader h = ld_header(gp.headers + slot);
        const uint64_t valid = (uint64_t)(h.count & ~kUnitLost) * gp.result_bytes;
        const uint64_t off = ((uint64_t)row_in_slot << 12) + threadIdx.x * 16;
        if ((h.count & kUnitLost) || off >= valid) return;
        uint8_t* dst = gp.out + (h.first - gp.win_first) * gp.result_bytes + off;
        if (off + 16 <= valid) st_vec(dst, data);
        else copy_tail_bytes(dst, data, (uint32_t)(valid - off));
    };

    for (;;) {
        const uint32_t gt = tc.claim(&s_ticket);
        if (gt >= n_groups) break;
        // newest slots first: the dispatch kernel filled the ring in ticket order just before this
        // launch, so its tail is still in the 126 MB L2 while its head has been written back
        const uint32_t g = reverse ? n_groups - 1 - gt : gt;
        const uint32_t slot0 = g * group_slots;
        const uint32_t nslots = min(group_slots, gp.n_units - slot0);
        const uint32_t nrows = nslots * rps;
        const uint8_t* src = gp.ring + (size_t)slot0 * gp.slot_stride + threadIdx.x * 16;
        uint32_t r = 0;
        for (; r + U <= nrows; r += U) {
            uint4 v[U];
#pragma unroll
            for (int u = 0; u < U; ++u) v[u] = ld_stream(src + ((size_t)(r + u) << 12));
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const uint32_t row = r + u;
                const uint32_t s = sh >= 0 ? (row >> sh) : (row / rps);
                place(v[u], slot0 + s, row - s * rps);
            }
        }
        for (; r < nrows; ++r) {
            const uint4 v = ld_stream(src + ((size_t)r << 12));
            const uint32_t s = sh >= 0 ? (r >> sh) : (r / rps);
            place(v, slot0 + s, r - s * rps);
        }
    }
    gather_epilogue(gp, blockIdx.x * kThreads + threadIdx.x, gridDim.x * kThreads);
}

// ---- bulk: TMA pipeline -------------------------------------------------------------------------------
namespace bulk {
constexpr uint32_t kChunk = 16384;     // bytes per bulk copy (a slot smaller than this is one chunk)
constexpr int kStages = 6;             // 96 KB of shared memory per CTA
constexpr int kLag = 4;                // loads run this many chunks ahead of their store
constexpr uint32_t kGroup = 32;        // slots per ticket: their headers are prefetched by the 32 lanes

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bulk_store(void* gdst, const void* smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(smem_src)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
}  // namespace bulk

// Requirements checked by the host: slot_stride % 16 == 0 and >= 4 KB, slot_stride <= kChunk or a
// multiple of kChunk, R % 16 == 0 or every unit full, output window 16 B aligned, no lost units.
__global__ void __launch_bounds__(32) gather_bulk_kernel(const GatherParams gp, uint32_t* ticket, uint32_t stage_stride,
                                                         uint32_t group_slots /* <= kGroup */) {
    using namespace bulk;
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint64_t full[kStages];
    __shared__ SlotHeader s_hdr[kGroup];
    __shared__ uint32_t s_group;
    const uint32_t lane = threadIdx.x;
    if (lane == 0) {
        for (int s = 0; s < kStages; ++s) mbar_init(&full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();

    const uint32_t chunk = gp.slot_stride < kChunk ? gp.slot_stride : kChunk;
    const uint32_t n_groups = (gp.n_units + group_slots - 1) / group_slots;
    uint32_t it = 0, st = 0;                             // chunks loaded / stored so far (lane 0)
    uint8_t* pend_dst[kStages] = {};
    uint32_t pend_bytes[kStages] = {};

    auto store_one = [&]() {
        const int sg = st % kStages;
        mbar_wait(&full[sg], (st / kStages) & 1);
        bulk_store(pend_dst[sg], smem + (size_t)sg * stage_stride, pend_bytes[sg]);
        ++st;
    };

    for (;;) {
        if (lane == 0) s_group = atomicAdd(ticket, 1u);
        __syncwarp();
        const uint32_t g = s_group;
        if (g >= n_groups) break;
        const uint32_t slot0 = g * group_slots;
        const uint32_t nslots = min(group_slots, gp.n_units - slot0);
        if (lane < nslots) s_hdr[lane] = ld_header(gp.headers + slot0 + lane);   // one coalesced 512 B read
        __syncwarp();
        if (lane == 0) {
            for (uint32_t s = 0; s < nslots; ++s) {
                const SlotHeader h = s_hdr[s];
                const uint32_t valid = (h.count & ~kUnitLost) * gp.result_bytes;   // < 4 GiB by construction
                const uint8_t* src = gp.ring + (size_t)(slot0 + s) * gp.slot_stride;
                uint8_t* dst = gp.out + (h.first - gp.win_first) * gp.result_bytes;
                // a tail unit whose byte count is not a multiple of 16: the last <16 bytes go by hand
                const uint32_t valid16 = valid & ~15u;
                for (uint32_t b = valid16; b < valid; ++b) dst[b] = src[b];
                for (uint32_t off = 0; off < valid16; off += chunk) {
                    const uint32_t bytes = min(chunk, valid16 - off);
                    const int sg = it % kStages;
                    // the stage was last used by chunk it-kStages, whose store was issued at least
                    // kStages-kLag-1 groups ago: wait until it has finished reading shared memory
                    if (it >= (uint32_t)kStages) bulk_wait_read<kStages - kLag - 1>();
                    pend_dst[sg] = dst + off;
                    pend_bytes[sg] = bytes;
                    mbar_expect_tx(&full[sg], bytes);
                    bulk_load(smem + (size_t)sg * stage_stride, src + off, bytes, &full[sg]);
                    ++it;
                    while (it - st > (uint32_t)kLag) store_one();
                }
            }
        }
        __syncwarp();
    }
    if (lane == 0) {
        while (st < it) store_one();
        asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    }
    gather_epilogue(gp, blockIdx.x * 32 + lane, gridDim.x * 32);
}

// ================================================================================================
// dispatch: payload_map_4k, TMA-staged (warp-specialised).  Same contract as
// dispatch_payload_map_kernel, for contiguous argument records (arg_stride == 4096):
//   warp 0 (one elected lane)  claims units by ticket, writes their slot headers, and bulk-loads the
//                              records in 16 KB chunks into shared-memory IN stages (mbarrier
//                              complete_tx); it waits on the stage's EMPTY barrier before reuse;
//   warps 1-4 (128 threads)    wait for a FULL stage, read it (LDS.128), apply out = in*K + t and
//                              write an OUT stage (STS.128); after a proxy fence + named barrier one
//                              of them bulk-stores the OUT stage into the result ring.
// Payload bytes cross registers only between two shared-memory stages; global traffic is TMA only.
// ================================================================================================
namespace tma_map {
constexpr uint32_t kMapChunk = 16384;
constexpr int kConsumers = 128;
struct ChunkDesc { uint8_t* dst; uint32_t bytes; uint32_t tbase; };
constexpr size_t smem_bytes(int in_stages, int out_stages) { return (size_t)(in_stages + out_stages) * kMapChunk; }
constexpr size_t kSmemBytes = smem_bytes(3, 2);      // the default instantiation: 80 KB, two CTAs per SM
}  // namespace tma_map

// <3 IN, 2 OUT> stages, 2 CTAs/SM: local HBM (96 KB of loads in flight per SM).  <6, 3>, 1 CTA/SM: the same bytes
// in flight from ONE producer per SM -- for records that live in a peer GPU's memory (NVLink round trips are ~4x
// longer and the link prefers fewer, deeper request streams).
template <int kInStages, int kOutStages>
__global__ void __launch_bounds__(160) dispatch_payload_map_tma_kernel(const WaveParams wp) {
    using namespace bulk;
    using namespace tma_map;
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint64_t full[kInStages], empty[kInStages];
    __shared__ ChunkDesc desc[kInStages];
    uint8_t* in_stage = smem;
    uint8_t* out_stage = smem + (size_t)kInStages * kMapChunk;
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < kInStages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], kConsumers); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (warp == 0) {
        if (lane != 0) return;
        // ---------------- producer ----------------
        uint32_t seq = 0;
        auto acquire_stage = [&]() -> int {
            const int sg = seq % kInStages;
            mbar_wait(&empty[sg], ((seq / kInStages) & 1) ^ 1);   // fresh barrier: passes immediately
            return sg;
        };
        for (;;) {
            const uint32_t t = atomicAdd(wp.ticket, 1u);
            if (t >= wp.n_units) {
                // no prefetch here: each CTA draws exactly one ticket >= n_units; the highest re-arms the counter
                if (t == wp.n_units + gridDim.x - 1u) *wp.ticket = 0u;
                break;
            }
            const TaskRecord rec = wave_record(wp, t);
            put_header(wp, t, SlotHeader{rec.seq, rec.count, rec.first});
            const uint8_t* src = wp.args + rec.arg_off;
            uint8_t* dst = wp.ring + (size_t)t * wp.slot_stride;
            const uint32_t total = rec.count * kPayloadBytes;
            const uint32_t tbase = (uint32_t)(wp.index_base + rec.first);
            for (uint32_t off = 0; off < total; off += kMapChunk) {
                const uint32_t bytes = min(kMapChunk, total - off);
                const int sg = acquire_stage();
                desc[sg] = ChunkDesc{dst + off, bytes, tbase + off / kPayloadBytes};
                mbar_expect_tx(&full[sg], bytes);
                bulk_load(in_stage + (size_t)sg * kMapChunk, src + off, bytes, &full[sg]);
                ++seq;
            }
        }
        const int sg = acquire_stage();                 // end marker
        desc[sg] = ChunkDesc{nullptr, 0u, 0u};
        asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&full[sg])) : "memory");
        return;
    }

    // ---------------- consumers (threads 32..159) ----------------
    const uint32_t ct = threadIdx.x - 32;               // 0..127
    for (uint32_t seq = 0;; ++seq) {
        const int sg = seq % kInStages, og = seq % kOutStages;
        mbar_wait(&full[sg], (seq / kInStages) & 1);
        const ChunkDesc d = desc[sg];
        if (d.bytes == 0) break;
        // the bulk store that last read OUT stage `og` (chunk seq-kOutStages) must be done with it
        if (ct == 0 && seq >= (uint32_t)kOutStages) bulk_wait_read<kOutStages - 1>();
        asm volatile("bar.sync 1, 128;" ::: "memory");
        const uint8_t* in = in_stage + (size_t)sg * kMapChunk;
        uint8_t* out = out_stage + (size_t)og * kMapChunk;
        const uint32_t nvec = d.bytes >> 4;
#pragma unroll
        for (uint32_t k = 0; k < kMapChunk / 16 / kConsumers; ++k) {
            const uint32_t v = ct + k * kConsumers;
            if (v < nvec) {
                uint4 x = *reinterpret_cast<const uint4*>(in + ((size_t)v << 4));
                const uint32_t tt = d.tbase + (v >> 8);   // 256 vectors per 4 KB record
                x.x = x.x * kPayloadMul + tt; x.y = x.y * kPayloadMul + tt;
                x.z = x.z * kPayloadMul + tt; x.w = x.w * kPayloadMul + tt;
                *reinterpret_cast<uint4*>(out + ((size_t)v << 4)) = x;
            }
        }
        // IN stage consumed; make the generic-proxy writes to the OUT stage visible to the async proxy
        asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&empty[sg])) : "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("bar.sync 1, 128;" ::: "memory");
        if (ct == 0) bulk_store(d.dst, out, d.bytes);
    }
    if (ct == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// ================================================================================================
// dispatch: record body -- a ThreadBody whose Arg and Res are trivially copyable records of 4..256 bytes
// (multiples of 4): floats, small structs, packed float3 points.  Explicit argument records only.
// A CTA stages each tile of its unit through shared memory:
//   1. cp.async copies the tile's argument words into an IN stage (one warp instruction = 128 consecutive
//      bytes of the wave's arguments, whatever the record size or alignment);
//   2. thread i runs B::run on record i of the stage and writes its Res into the OUT tile;
//   3. the CTA stores the OUT tile to the slot, one warp instruction = 128 consecutive bytes.
// The copy of tile k+1 is in flight while tile k computes (two IN stages).  Records sit in shared memory at an
// odd number of words apart, so the per-thread record reads and result writes are free of bank conflicts for
// every record size (a 64 B record at its natural stride would be a 16-way conflict).  Record bases need only be
// 4-byte aligned: an arg_stride of 12 at an odd record offset, a unit whose result bytes end mid-vector and the
// argument records of a strided layout (arg_stride > sizeof(Arg)) all take the same word path.
// Algorithmic bytes per task: sizeof(Arg) read + sizeof(Res) written.
// ================================================================================================
namespace rec {
__device__ __forceinline__ void cp_async4(void* s, const void* g) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(s)), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

constexpr uint32_t kStageBytes = 12288;     // shared memory of one IN stage (OUT tile: at most the same)
constexpr uint32_t odd_words(uint32_t bytes) { return (bytes / 4) | 1u; }   // padded record pitch in words

template <class B>
struct Layout {
    using Arg = typename B::Arg;
    using Res = typename B::Res;
    static constexpr uint32_t kArgWords = sizeof(Arg) / 4, kResWords = sizeof(Res) / 4;
    static constexpr uint32_t kArgPitch = odd_words(sizeof(Arg)), kResPitch = odd_words(sizeof(Res));   // words
    static constexpr uint32_t kMaxPitch = kArgPitch > kResPitch ? kArgPitch : kResPitch;
    static constexpr uint32_t kTasks = (kStageBytes / 4 / kMaxPitch) < 2048u ? (kStageBytes / 4 / kMaxPitch) : 2048u;   // per tile
    static constexpr uint32_t kInWords = kTasks * kArgPitch, kOutWords = kTasks * kResPitch;
    static_assert(std::is_trivially_copyable<Arg>::value && std::is_trivially_copyable<Res>::value,
                  "record bodies take and return trivially copyable records");
    static_assert(sizeof(Arg) % 4 == 0 && sizeof(Arg) >= 4 && sizeof(Arg) <= 256, "sizeof(Arg) must be a multiple of 4 in [4, 256]");
    static_assert(sizeof(Res) % 4 == 0 && sizeof(Res) >= 4 && sizeof(Res) <= 256, "sizeof(Res) must be a multiple of 4 in [4, 256]");
    static_assert((2 * kInWords + kOutWords) * 4 <= 48 * 1024, "static shared memory of the record kernel");
};

// Copy the argument words of tasks [0, cnt) of a tile (records `stride` bytes apart from `src`) into `stage`.
template <class L>
__device__ __forceinline__ void load_tile(uint32_t* stage, const uint8_t* src, uint32_t stride, uint32_t cnt) {
    const uint32_t total = cnt * L::kArgWords;
    for (uint32_t w = threadIdx.x; w < total; w += kThreads) {
        const uint32_t r = w / L::kArgWords, j = w - r * L::kArgWords;
        cp_async4(stage + r * L::kArgPitch + j, src + (size_t)r * stride + 4u * j);
    }
}
}  // namespace rec

template <class B>
__global__ void __launch_bounds__(kThreads) dispatch_record_kernel(const WaveParams wp) {
    using L = rec::Layout<B>;
    using Arg = typename B::Arg;
    using Res = typename B::Res;
    __shared__ uint32_t s_in[2 * L::kInWords];
    __shared__ uint32_t s_out[L::kOutWords];
    __shared__ uint32_t s_ticket[2];
    __shared__ int s_fault;
    if (threadIdx.x == 0) s_fault = 0;
    const ErrSink es{wp.err_word, &s_fault};
    TicketClaimer tc{wp.ticket, 0u};
    tc.prime();
    uint32_t iter = 0;
    uint32_t t = tc.claim_db(s_ticket, iter++);
    TaskRecord rc{};
    if (t < wp.n_units) {
        rc = wave_record(wp, t);
        rec::load_tile<L>(s_in, wp.args + rc.arg_off, wp.arg_stride, min(rc.count, L::kTasks));
    }
    rec::cp_async_commit();
    uint32_t tile = 0, buf = 0;
    while (t < wp.n_units) {
        // the tile to prefetch: the next one of this unit, or the first of the next unit claimed
        uint32_t nt = t, ntile = tile + 1;
        TaskRecord nrc = rc;
        const bool last = (uint64_t)ntile * L::kTasks >= rc.count;
        if (last) {
            nt = tc.claim_db(s_ticket, iter++);
            ntile = 0;
            if (nt < wp.n_units) nrc = wave_record(wp, nt);
        }
        if (nt < wp.n_units) {
            const uint32_t first = ntile * L::kTasks;
            rec::load_tile<L>(s_in + (buf ^ 1u) * L::kInWords, wp.args + nrc.arg_off + (size_t)first * wp.arg_stride,
                              wp.arg_stride, min(nrc.count - first, L::kTasks));
        }
        rec::cp_async_commit();
        rec::cp_async_wait<1>();      // this thread's copies of the current tile have landed ...
        __syncthreads();              // ... and everyone else's; the previous OUT tile has been stored

        const uint32_t first = tile * L::kTasks;
        const uint32_t cnt = min(rc.count - first, L::kTasks);
        const uint32_t* in = s_in + buf * L::kInWords;
        const uint64_t gidx0 = wp.index_base + rc.first + first;
        for (uint32_t i = threadIdx.x; i < cnt; i += kThreads) {
            uint32_t aw[L::kArgWords];
#pragma unroll
            for (uint32_t k = 0; k < L::kArgWords; ++k) aw[k] = in[i * L::kArgPitch + k];
            Arg a;
            memcpy(&a, aw, sizeof(Arg));
            const Res r = B::run(a, gidx0 + i, es, rc.attempt);
            uint32_t rw[L::kResWords];
            memcpy(rw, &r, sizeof(Res));
#pragma unroll
            for (uint32_t k = 0; k < L::kResWords; ++k) s_out[i * L::kResPitch + k] = rw[k];
        }
        __syncthreads();              // OUT tile complete, fault reports of the tile are in, IN stage `buf` is free

        uint32_t* dst = reinterpret_cast<uint32_t*>(wp.ring + (size_t)t * wp.slot_stride + (size_t)first * sizeof(Res));
        const uint32_t total = cnt * L::kResWords;
        for (uint32_t w = threadIdx.x; w < total; w += kThreads) {
            const uint32_t r = w / L::kResWords, j = w - r * L::kResWords;
            dst[w] = s_out[r * L::kResPitch + j];
        }
        if (last && threadIdx.x == 0) {
            bool lost = false;
            if constexpr (B::kCanFault) {
                lost = s_fault != 0;  // every report of this unit happened before the barrier above
                s_fault = 0;          // the next unit computes only after the next barrier
                if (lost && !wp.resilient)
                    atomicMin(wp.err_word, (unsigned long long)(((wp.index_base + rc.first) << 8) | TASK_FAULT));
            }
            put_header(wp, t, SlotHeader{rc.seq, rc.count | ((lost && wp.resilient) ? kUnitLost : 0u), rc.first});
        }
        t = nt;
        rc = nrc;
        tile = ntile;
        buf ^= 1u;
    }
    rec::cp_async_wait<0>();
    tc.rearm(wp.n_units);
}

// ================================================================================================
// payload_fill: w[t][j] = low32(splitmix64(SEED ^ (t*1024 + j))); each thread emits 16 B.
// ================================================================================================
__global__ void __launch_bounds__(kThreads) payload_fill_kernel(uint4* out, uint64_t t0, uint64_t n_vec) {
    const uint64_t gsize = (uint64_t)gridDim.x * kThreads;
    for (uint64_t v = (uint64_t)blockIdx.x * kThreads + threadIdx.x; v < n_vec; v += gsize) {
        const uint64_t w0 = t0 * kPayloadWords + v * 4;
        uint4 r;
        r.x = (uint32_t)splitmix64(kPayloadSeed ^ (w0 + 0));
        r.y = (uint32_t)splitmix64(kPayloadSeed ^ (w0 + 1));
        r.z = (uint32_t)splitmix64(kPayloadSeed ^ (w0 + 2));
        r.w = (uint32_t)splitmix64(kPayloadSeed ^ (w0 + 3));
        out[v] = r;
    }
}

}  // namespace fbr
