// fiber_b200_body.cuh -- what an OUT-OF-TREE device body is compiled against.
//
// The reference ships any Python callable to its workers (fiber/pool.py:961) and the worker calls it
// (fiber/pool.py:806,809,820).  A B200 worker runs device code, so a user function needs a device body;
// this header lets that body live outside libfiber_b200: write a ThreadBody struct, export it, build a
// shared object, register it.
//
//     #include "fiber_b200_body.cuh"
//     struct Collatz {                                   // steps of the Collatz iteration from x
//         using Arg = int64_t; using Res = int64_t;
//         static constexpr bool kIndexArg = true;        // may be mapped over a range() with no argument bytes
//         static constexpr bool kVecIndex = false;
//         static constexpr bool kCanFault = false;
//         __device__ static Res run(const Arg& a, uint64_t task_index, const fbr::ErrSink& es, uint32_t attempt) { ... }
//     };
//     FBR_EXPORT_THREAD_BODY(Collatz, "collatz_steps", collatz_entry, FBR_RES_I64, FBR_BODY_INDEX_ARG | FBR_BODY_SUMMABLE)
//
//     nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -shared -Xcompiler -fPIC \
//          -I<repo>/include -I<repo>/fiber_b200/csrc body.cu -o libbody.so
//     fbr_register_body("collatz_steps", "libbody.so", "collatz_entry", &func_id);
//
// (fiber_b200.device_body(name, source=...) does the last two steps from Python.)  The body is instantiated
// into the same persistent-CTA dispatch kernel template the compiled-in bodies use, so it gets the ticket
// claim, record synthesis, direct placement / result ring, sum fold and resilient re-dispatch for free.
//
// A function of floats or of a small struct is a RECORD body: Arg and Res are any trivially copyable types whose
// sizes are multiples of 4 bytes from 4 to 256 (a packed float3 is 12 B), exported with FBR_EXPORT_RECORD_BODY.
// Its tiles are staged through shared memory by dispatch_record_kernel (kernels.cuh), except for 8 B -> 8 B records,
// which run one thread per record in dispatch_thread_kernel, where they are faster; it takes explicit argument
// records only (no kIndexArg mode), and its results are opaque records (no device-side sum).
//
//     struct Norm3 {                                     // |p| of a packed float3, correctly rounded steps
//         using Arg = float3; using Res = float;
//         static constexpr bool kIndexArg = false;
//         static constexpr bool kVecIndex = false;
//         static constexpr bool kCanFault = false;
//         __device__ static Res run(const Arg& p, uint64_t, const fbr::ErrSink&, uint32_t) {
//             return __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(p.x, p.x), __fmul_rn(p.y, p.y)), __fmul_rn(p.z, p.z)));
//         }
//     };
//     FBR_EXPORT_RECORD_BODY(Norm3, "norm3", norm3_entry, 0)
//
//     @fiber_b200.device_body("norm3", source=SRC, entry="norm3_entry", args="3f4", result="f4")
#pragma once
#include "fiber_b200.h"
#include "kernels.cuh"      // fiber_b200/csrc: dispatch_thread_kernel, dispatch_record_kernel, WaveParams, ErrSink, TaskError

namespace fbr_body_export {
template <class B>
void launch(const void* wpv, int grid, void* sv) {
    const fbr::WaveParams& wp = *(const fbr::WaveParams*)wpv;
    cudaStream_t s = (cudaStream_t)sv;
    if constexpr (B::kIndexArg) {
        if (wp.arg_stride == 0) {
            fbr::dispatch_thread_kernel<B, true><<<grid, fbr::kThreads, 0, s>>>(wp);
            return;
        }
    }
    fbr::dispatch_thread_kernel<B, false><<<grid, fbr::kThreads, 0, s>>>(wp);
}
template <class B>
int occupancy(int index_mode) {
    int occ = 0;
    cudaError_t e;
    if constexpr (B::kIndexArg) {
        if (index_mode) {
            e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, (const void*)fbr::dispatch_thread_kernel<B, true>, fbr::kThreads, 0);
            if (e != cudaSuccess) { cudaGetLastError(); return 1; }
            return occ > 0 ? occ : 1;
        }
    }
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, (const void*)fbr::dispatch_thread_kernel<B, false>, fbr::kThreads, 0);
    if (e != cudaSuccess) { cudaGetLastError(); return 1; }
    return occ > 0 ? occ : 1;
}
}  // namespace fbr_body_export

namespace fbr_body_export {
// the bit-packed twin of a bool body: 8 items (explicit records or range() indices) per result byte
template <class B>
void launch_bits(const void* wpv, int grid, void* sv) {
    const fbr::WaveParams& wp = *(const fbr::WaveParams*)wpv;
    cudaStream_t s = (cudaStream_t)sv;
    if constexpr (B::kIndexArg) {
        if (wp.arg_stride == 0) {
            fbr::dispatch_bits_items_kernel<B, true><<<grid, fbr::kThreads, 0, s>>>(wp);
            return;
        }
    }
    fbr::dispatch_bits_items_kernel<B, false><<<grid, fbr::kThreads, 0, s>>>(wp);
}
template <class B>
int occupancy_bits(int index_mode) {
    int occ = 0;
    const void* k = (const void*)fbr::dispatch_bits_items_kernel<B, false>;
    if constexpr (B::kIndexArg) {
        if (index_mode) k = (const void*)fbr::dispatch_bits_items_kernel<B, true>;
    }
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k, fbr::kThreads, 0) != cudaSuccess) { cudaGetLastError(); return 1; }
    return occ > 0 ? occ : 1;
}
}  // namespace fbr_body_export

// A bool body (Res = uint8_t, 0/1) additionally exports its bit-packed twin "<name>_bits8" (result kind
// FBR_RES_BITS8, 8 items per task): register both and bool results travel one bit each.
#define FBR_EXPORT_BOOL_BODY_BITS(Body, twin_name, entry, body_flags)                                              \
    extern "C" const fbr_body_module_t* entry(void) {                                                            \
        static const fbr_body_module_t m = {FBR_BODY_MODULE_ABI, (uint32_t)sizeof(fbr::WaveParams), twin_name,   \
                                            8u * (uint32_t)sizeof(typename Body::Arg), 1u, (uint32_t)FBR_RES_BITS8, \
                                            (uint32_t)(body_flags), 512u,                                        \
                                            fbr_body_export::launch_bits<Body>, fbr_body_export::occupancy_bits<Body>}; \
        return &m;                                                                                               \
    }

namespace fbr_body_export {
// record bodies: the staged record kernel (static shared memory only, below 48 KB: no attribute to set per device)
template <class B>
void launch_staged(const void* wpv, int grid, void* sv) {
    fbr::dispatch_record_kernel<B><<<grid, fbr::kThreads, 0, (cudaStream_t)sv>>>(*(const fbr::WaveParams*)wpv);
}
template <class B>
int occupancy_staged(int) {
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, (const void*)fbr::dispatch_record_kernel<B>, fbr::kThreads, 0) != cudaSuccess) {
        cudaGetLastError();
        return 1;
    }
    return occ > 0 ? occ : 1;
}
// Layouts where one thread per record, reading it in place, is faster than staging tiles through shared memory.
// Measured (profiles/record_perf_b200.json): 8 B -> 8 B records, 0.263 ms per 1e8 tasks in dispatch_thread_kernel
// against 0.317 ms staged.  Wider arguments lose in place (64 B -> 8 B: 2.84 ms against 1.49 ms staged).
template <class B>
constexpr bool kPerThreadRecords = sizeof(typename B::Arg) == 8 && sizeof(typename B::Res) == 8;
// The per-thread kernel reads each Arg in place, so it needs 8-byte aligned records; a wave whose records are only
// 4-byte aligned (arg_stride 12, device arguments at an odd word) takes the staged kernel, which reads words.
template <class B>
void launch_record(const void* wpv, int grid, void* sv) {
    const fbr::WaveParams& wp = *(const fbr::WaveParams*)wpv;
    if constexpr (kPerThreadRecords<B>) {
        if (wp.arg_stride % 8 == 0 && (reinterpret_cast<uintptr_t>(wp.args) & 7) == 0) {
            fbr::dispatch_thread_kernel<B, false><<<grid, fbr::kThreads, 0, (cudaStream_t)sv>>>(wp);
            return;
        }
    }
    launch_staged<B>(wpv, grid, sv);
}
// Resident CTAs of the kernel the body's waves normally take (a staged wave of a per-thread layout may get a grid
// larger than its residency: its extra CTAs start as others finish and find the tickets drawn)
template <class B>
int occupancy_record(int index_mode) {
    if constexpr (kPerThreadRecords<B>) return occupancy<B>(index_mode);
    return occupancy_staged<B>(index_mode);
}
}  // namespace fbr_body_export

// Body: a ThreadBody whose Arg and Res are trivially copyable records, sizes multiples of 4 in [4, 256] (checked by
// fbr::rec::Layout).  flags: 0, or FBR_BODY_* bits other than SUMMABLE / INDEX_ARG / INDEX_ONLY / NEEDS_SHARED.
// The kernel follows from the record sizes (kPerThreadRecords): there is nothing to choose.
#define FBR_EXPORT_RECORD_BODY(Body, body_name, entry, body_flags)                                               \
    static_assert(((body_flags) & (FBR_BODY_SUMMABLE | FBR_BODY_INDEX_ARG | FBR_BODY_INDEX_ONLY | FBR_BODY_NEEDS_SHARED)) == 0, \
                  "record bodies are not summable and take explicit argument records only");                    \
    static_assert(!Body::kIndexArg, "record bodies have no range() index mode");                                 \
    static_assert(sizeof(fbr::rec::Layout<Body>) > 0, "record layout");                                          \
    extern "C" const fbr_body_module_t* entry(void) {                                                            \
        static const fbr_body_module_t m = {FBR_BODY_MODULE_ABI, (uint32_t)sizeof(fbr::WaveParams), body_name,   \
                                            (uint32_t)sizeof(typename Body::Arg), (uint32_t)sizeof(typename Body::Res), \
                                            (uint32_t)FBR_RES_BYTES, (uint32_t)(body_flags) | FBR_BODY_RECORD, 4096u, \
                                            fbr_body_export::launch_record<Body>, fbr_body_export::occupancy_record<Body>}; \
        return &m;                                                                                               \
    }

// Body: a ThreadBody (see bodies.cuh) whose Res is 1 or 8 bytes.  result_kind: FBR_RES_BOOL / FBR_RES_I64 / ...
#define FBR_EXPORT_THREAD_BODY(Body, body_name, entry, kind, body_flags)                                         \
    extern "C" const fbr_body_module_t* entry(void) {                                                            \
        static const fbr_body_module_t m = {FBR_BODY_MODULE_ABI, (uint32_t)sizeof(fbr::WaveParams), body_name,   \
                                            (uint32_t)sizeof(typename Body::Arg), (uint32_t)sizeof(typename Body::Res), \
                                            (uint32_t)(kind), (uint32_t)(body_flags), 4096u,                     \
                                            fbr_body_export::launch<Body>, fbr_body_export::occupancy<Body>};    \
        return &m;                                                                                               \
    }
