"""Record bodies defined OUTSIDE libfiber_b200: float and struct arguments and results (FBR_EXPORT_RECORD_BODY).

The CUDA source below is compiled once into a body module under ``fiber_b200/_lib/bodies/`` and every body in it
is registered with the engine at import time, with NumPy dtypes for its argument and result records.  The ``*_np``
functions restate each body over whole arrays; float bodies use correctly rounded single operations
(``__fadd_rn``, ``__fmul_rn``, ``__dmul_rn``, ...), so the restatements agree bit for bit, no tolerance needed.

Two bodies are exported twice, with FBR_EXPORT_THREAD_BODY (one thread per task, records read in place) and with
FBR_EXPORT_RECORD_BODY: ``poly_f64`` and ``dot_w64``.  FBR_EXPORT_RECORD_BODY stages ``dot_w64``'s tiles through
shared memory and runs the 8 B -> 8 B ``poly_f64`` one thread per record; ``poly_f64_staged`` is the same body forced
through the staged kernel.  Their outputs must be identical, and ``profiles/record_perf.py`` times the kernels against
each other.
"""
import numpy as np

import fiber_b200
from fiber_b200 import bodies, registry

RECORD_SRC = r'''
#include "fiber_b200_body.cuh"

#define RECORD_BODY_TRAITS                      \
    static constexpr bool kIndexArg = false;    \
    static constexpr bool kVecIndex = false;

// float3 (12 B) -> float: squared norm
struct Norm2F3 {
    using Arg = float3; using Res = float;
    RECORD_BODY_TRAITS
    static constexpr bool kCanFault = false;
    __device__ static __forceinline__ Res run(const Arg& p, uint64_t, const fbr::ErrSink&, uint32_t) {
        return __fadd_rn(__fadd_rn(__fmul_rn(p.x, p.x), __fmul_rn(p.y, p.y)), __fmul_rn(p.z, p.z));
    }
};
FBR_EXPORT_RECORD_BODY(Norm2F3, "norm2_f3", norm2_f3_entry, 0)

// float3 -> float3: (2x + y, y/2 - z, z + x)
struct AffineF3 {
    using Arg = float3; using Res = float3;
    RECORD_BODY_TRAITS
    static constexpr bool kCanFault = false;
    __device__ static __forceinline__ Res run(const Arg& p, uint64_t, const fbr::ErrSink&, uint32_t) {
        return make_float3(__fadd_rn(__fmul_rn(p.x, 2.0f), p.y), __fsub_rn(__fmul_rn(p.y, 0.5f), p.z), __fadd_rn(p.z, p.x));
    }
};
FBR_EXPORT_RECORD_BODY(AffineF3, "affine_f3", affine_f3_entry, 0)

// f64 -> f64: 1.5 x + 0.25, as a thread body and as a record body
struct PolyF64 {
    using Arg = double; using Res = double;
    RECORD_BODY_TRAITS
    static constexpr bool kCanFault = false;
    __device__ static __forceinline__ Res run(const Arg& x, uint64_t, const fbr::ErrSink&, uint32_t) {
        return __dadd_rn(__dmul_rn(x, 1.5), 0.25);
    }
};
FBR_EXPORT_THREAD_BODY(PolyF64, "poly_f64_thread", poly_f64_thread_entry, FBR_RES_BYTES, 0)
FBR_EXPORT_RECORD_BODY(PolyF64, "poly_f64", poly_f64_entry, 0)
// ... and forced through the staged kernel, which FBR_EXPORT_RECORD_BODY does not pick for 8 B -> 8 B records: the
// other side of that choice, for the tests and profiles/record_perf.py (a hand-written descriptor, not an option)
extern "C" const fbr_body_module_t* poly_f64_staged_entry(void) {
    static const fbr_body_module_t m = {FBR_BODY_MODULE_ABI, (uint32_t)sizeof(fbr::WaveParams), "poly_f64_staged", 8u, 8u,
                                        (uint32_t)FBR_RES_BYTES, FBR_BODY_RECORD, 4096u,
                                        fbr_body_export::launch_staged<PolyF64>, fbr_body_export::occupancy_staged<PolyF64>};
    return &m;
}

struct W64 { double v[8]; };                                     // 64 B argument record
struct Stats { double sum; int32_t n_neg; uint32_t low_xor; };    // 16 B mixed result record

// 64 B -> {f64, i32, u32}: left-to-right sum, count of negative values, xor of the low words
struct StatsW64 {
    using Arg = W64; using Res = Stats;
    RECORD_BODY_TRAITS
    static constexpr bool kCanFault = false;
    __device__ static __forceinline__ Res run(const Arg& a, uint64_t, const fbr::ErrSink&, uint32_t) {
        Stats r{0.0, 0, 0u};
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            r.sum = __dadd_rn(r.sum, a.v[k]);
            r.n_neg += a.v[k] < 0.0 ? 1 : 0;
            r.low_xor ^= (uint32_t)__double2loint(a.v[k]);
        }
        return r;
    }
};
FBR_EXPORT_RECORD_BODY(StatsW64, "stats_w64", stats_w64_entry, 0)

// 64 B -> f64: sum_k (k + 1) v[k], left to right, as a thread body and as a record body
struct DotW64 {
    using Arg = W64; using Res = double;
    RECORD_BODY_TRAITS
    static constexpr bool kCanFault = false;
    __device__ static __forceinline__ Res run(const Arg& a, uint64_t, const fbr::ErrSink&, uint32_t) {
        double s = 0.0;
#pragma unroll
        for (int k = 0; k < 8; ++k) s = __dadd_rn(s, __dmul_rn(a.v[k], (double)(k + 1)));
        return s;
    }
};
FBR_EXPORT_THREAD_BODY(DotW64, "dot_w64_thread", dot_w64_thread_entry, FBR_RES_BYTES, 0)
FBR_EXPORT_RECORD_BODY(DotW64, "dot_w64", dot_w64_entry, 0)

// 256 B -> 256 B at the size limit: out[k] = in[63 - k] * 2654435761 + k (u32 wrap-around)
struct U64w { uint32_t w[64]; };
struct Mix256 {
    using Arg = U64w; using Res = U64w;
    RECORD_BODY_TRAITS
    static constexpr bool kCanFault = false;
    __device__ static __forceinline__ Res run(const Arg& a, uint64_t, const fbr::ErrSink&, uint32_t) {
        Res r;
#pragma unroll
        for (int k = 0; k < 64; ++k) r.w[k] = a.w[63 - k] * 2654435761u + (uint32_t)k;
        return r;
    }
};
FBR_EXPORT_RECORD_BODY(Mix256, "mix_256", mix_256_entry, 0)

// float -> float: x / 2, a bad argument unless x >= 0
struct HalveNonneg {
    using Arg = float; using Res = float;
    RECORD_BODY_TRAITS
    static constexpr bool kCanFault = false;
    __device__ static __forceinline__ Res run(const Arg& x, uint64_t gidx, const fbr::ErrSink& es, uint32_t) {
        if (!(x >= 0.0f)) { es.report(fbr::TASK_BADARG, gidx); return 0.0f; }
        return __fmul_rn(x, 0.5f);
    }
};
FBR_EXPORT_RECORD_BODY(HalveNonneg, "halve_nonneg", halve_nonneg_entry, 0)

// {f32 x, i32 tag} -> f32: 3x; a task tagged 1 "kills its worker" on its first attempt (the unit is lost and,
// in a resilient pool, re-dispatched with attempt 1)
struct Tagged { float x; int32_t tag; };
struct TripleOrFault {
    using Arg = Tagged; using Res = float;
    RECORD_BODY_TRAITS
    static constexpr bool kCanFault = true;
    __device__ static __forceinline__ Res run(const Arg& a, uint64_t gidx, const fbr::ErrSink& es, uint32_t attempt) {
        if (attempt == 0u && a.tag == 1) es.report(fbr::TASK_FAULT, gidx);
        return __fmul_rn(a.x, 3.0f);
    }
};
FBR_EXPORT_RECORD_BODY(TripleOrFault, "triple_or_fault", triple_or_fault_entry, 0)

// Descriptors the engine must refuse, written by hand (FBR_EXPORT_RECORD_BODY's static_asserts reject them)
#define BAD_RECORD_MODULE(entry, name, ab, rb, fl)                                                                 \
    extern "C" const fbr_body_module_t* entry(void) {                                                            \
        static const fbr_body_module_t m = {FBR_BODY_MODULE_ABI, (uint32_t)sizeof(fbr::WaveParams), name, ab, rb, \
                                            (uint32_t)FBR_RES_BYTES, (uint32_t)(fl) | FBR_BODY_RECORD, 4096u,    \
                                            fbr_body_export::launch_record<Norm2F3>,                             \
                                            fbr_body_export::occupancy_record<Norm2F3>};                         \
        return &m;                                                                                               \
    }
BAD_RECORD_MODULE(bad_arg6_entry, "bad_arg6", 6u, 4u, 0u)
BAD_RECORD_MODULE(bad_arg260_entry, "bad_arg260", 260u, 4u, 0u)
BAD_RECORD_MODULE(bad_res2_entry, "bad_res2", 12u, 2u, 0u)
BAD_RECORD_MODULE(bad_summable_entry, "bad_summable", 12u, 4u, FBR_BODY_SUMMABLE)
BAD_RECORD_MODULE(bad_index_entry, "bad_index", 12u, 4u, FBR_BODY_INDEX_ARG)
'''

F3 = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4")])
W64 = np.dtype([("v", "<f8", (8,))])
STATS = np.dtype([("sum", "<f8"), ("n_neg", "<i4"), ("low_xor", "<u4")])
TAGGED = np.dtype([("x", "<f4"), ("tag", "<i4")])

# modules fbr_register_body refuses: body name -> entry
BAD_MODULES = {"bad_arg6": "bad_arg6_entry", "bad_arg260": "bad_arg260_entry", "bad_res2": "bad_res2_entry",
               "bad_summable": "bad_summable_entry", "bad_index": "bad_index_entry"}

# body name -> (entry, argument dtype, result dtype)
LAYOUTS = {
    "norm2_f3": ("norm2_f3_entry", F3, "<f4"),
    "affine_f3": ("affine_f3_entry", "3f4", "3f4"),
    "poly_f64": ("poly_f64_entry", "f8", "f8"),
    "poly_f64_thread": ("poly_f64_thread_entry", "f8", "f8"),
    "poly_f64_staged": ("poly_f64_staged_entry", "f8", "f8"),
    "stats_w64": ("stats_w64_entry", W64, STATS),
    "dot_w64": ("dot_w64_entry", W64, "<f8"),
    "dot_w64_thread": ("dot_w64_thread_entry", W64, "<f8"),
    "mix_256": ("mix_256_entry", "64u4", "64u4"),
    "halve_nonneg": ("halve_nonneg_entry", "<f4", "<f4"),
    "triple_or_fault": ("triple_or_fault_entry", TAGGED, "<f4"),
}

MODULE = bodies.compile_module("record_bodies", RECORD_SRC)
for _name, (_entry, _args, _result) in LAYOUTS.items():
    registry.register_module(_name, MODULE, _entry, args=_args, result=_result)


# ---- the callables (one per body; several names can share a definition) ------------------------------------------
def norm2_f3(x, y, z):
    return float(np.float32(np.float32(x * x) + np.float32(y * y)) + np.float32(z * z))


def affine_f3(x, y, z):
    return tuple(affine_f3_np(np.array([[x, y, z]], dtype=np.float32))[0].tolist())


def poly_f64(x):
    return x * 1.5 + 0.25


def stats_w64(v):
    return tuple(stats_w64_np(np.array([(v,)], dtype=W64))[0].tolist())


def dot_w64(v):
    return float(dot_w64_np(np.array([(v,)], dtype=W64))[0])


def mix_256(*w):
    return tuple(mix_256_np(np.array([w], dtype=np.uint32))[0].tolist())


def halve_nonneg(x):
    if not x >= 0:
        raise ValueError("halve_nonneg: bad argument")
    return x / 2


def triple_or_fault(x, tag):
    return float(np.float32(x) * np.float32(3))


for _name, _f in (("norm2_f3", norm2_f3), ("affine_f3", affine_f3), ("poly_f64", poly_f64), ("stats_w64", stats_w64),
                  ("dot_w64", dot_w64), ("mix_256", mix_256), ("halve_nonneg", halve_nonneg),
                  ("triple_or_fault", triple_or_fault)):
    fiber_b200.bind(_f, _name)


def poly_f64_thread(x):
    return poly_f64(x)


def dot_w64_thread(v):
    return dot_w64(v)


def poly_f64_staged(x):
    return poly_f64(x)


fiber_b200.bind(poly_f64_thread, "poly_f64_thread")
fiber_b200.bind(poly_f64_staged, "poly_f64_staged")
fiber_b200.bind(dot_w64_thread, "dot_w64_thread")


# ---- NumPy restatements (whole arrays, bit-exact) ---------------------------------------------------------------
def _f32_cols(p):
    p = np.asarray(p)
    if p.dtype.names:
        return p["x"], p["y"], p["z"]
    return p[:, 0], p[:, 1], p[:, 2]


def norm2_f3_np(p):
    x, y, z = _f32_cols(p)
    return (x * x + y * y) + z * z


def affine_f3_np(p):
    x, y, z = _f32_cols(p)
    return np.stack([x * np.float32(2) + y, y * np.float32(0.5) - z, z + x], axis=1)


def poly_f64_np(x):
    return np.asarray(x, dtype=np.float64) * 1.5 + 0.25


def stats_w64_np(a):
    v = np.asarray(a)["v"]
    out = np.zeros(len(v), dtype=STATS)
    s = np.zeros(len(v))
    for k in range(8):
        s = s + v[:, k]
    out["sum"] = s
    out["n_neg"] = (v < 0).sum(axis=1)
    out["low_xor"] = np.bitwise_xor.reduce((v.view(np.uint64) & np.uint64(0xFFFFFFFF)).astype(np.uint32), axis=1)
    return out


def dot_w64_np(a):
    v = np.asarray(a)["v"]
    s = np.zeros(len(v))
    for k in range(8):
        s = s + v[:, k] * float(k + 1)
    return s


def mix_256_np(w):
    w = np.asarray(w, dtype=np.uint32)
    with np.errstate(over="ignore"):
        return w[:, ::-1] * np.uint32(2654435761) + np.arange(64, dtype=np.uint32)


def halve_nonneg_np(x):
    return np.asarray(x, dtype=np.float32) * np.float32(0.5)


def triple_or_fault_np(a):
    return np.asarray(a)["x"] * np.float32(3)
