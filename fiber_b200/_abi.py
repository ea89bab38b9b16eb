"""ctypes binding of ``include/fiber_b200.h`` (libfiber_b200.so).

This file *is* the reference-side binding a fiber maintainer would add (INTEGRATION.md): plain
``ctypes``, no torch types.  There is no CPU fallback: if the shared library is missing or cannot be
loaded, importing the engine raises immediately.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_lib", "libfiber_b200.so")

FBR_ABI_VERSION = 2

# fbr_status
FBR_OK, FBR_EINVAL, FBR_ECUDA, FBR_ENOMEM, FBR_ESTATE, FBR_ETIMEOUT, FBR_ETASK, FBR_ENODEV, FBR_ENOENT = \
    0, -1, -2, -3, -4, -5, -6, -7, -8
# fbr_result_kind
FBR_RES_BYTES, FBR_RES_BOOL, FBR_RES_I64, FBR_RES_U32, FBR_RES_F64X2, FBR_RES_NONE, FBR_RES_BITS8 = range(7)
# body flags
FBR_BODY_INDEX_ARG, FBR_BODY_NEEDS_SHARED, FBR_BODY_SUMMABLE, FBR_BODY_INDEX_ONLY = 0x1, 0x2, 0x4, 0x8
FBR_BODY_RECORD = 0x10
# pool flags
FBR_POOL_TIMING, FBR_POOL_OVERLAP = 0x1, 0x2
# map flags
FBR_MAP, FBR_STARMAP, FBR_APPLY = 0x0, 0x1, 0x2
FBR_ARGS_DEVICE, FBR_OUT_DEVICE, FBR_WANT_SUM, FBR_SHUFFLE, FBR_FULL_WINDOW, FBR_SHARED_HANDLE, FBR_RESILIENT, \
    FBR_RESULTS_ON_DEVICE, FBR_VIA_RING, FBR_NO_ZERO_COPY = 0x10, 0x20, 0x40, 0x80, 0x100, 0x200, 0x400, 0x800, 0x1000, 0x2000
# fbr_task_error
FBR_TASK_OK, FBR_TASK_OVERFLOW, FBR_TASK_BADARG, FBR_TASK_FAULT = range(4)

# every symbol include/fiber_b200.h declares (tests check the .so exports each of them)
SYMBOLS = [
    "fbr_abi_version", "fbr_last_error", "fbr_device_count",
    "fbr_body_count", "fbr_body_info", "fbr_body_lookup", "fbr_register_body",
    "fbr_pool_create", "fbr_pool_close", "fbr_pool_terminate", "fbr_pool_join", "fbr_pool_destroy",
    "fbr_pool_n_workers", "fbr_pool_worker_device",
    "fbr_map_submit", "fbr_shared_put", "fbr_shared_drop", "fbr_plan_query",
    "fbr_result_wait", "fbr_result_poll", "fbr_result_data", "fbr_result_fetch", "fbr_result_release",
    "fbr_host_alloc", "fbr_host_free", "fbr_device_alloc", "fbr_device_free",
    "fbr_memcpy_h2d", "fbr_memcpy_d2h", "fbr_payload_fill_device",
    "fbr_pool_stats", "fbr_pool_stats_reset",
    "fbr_queue_last_error", "fbr_queue_create", "fbr_queue_open_writer", "fbr_queue_open_reader",
    "fbr_lane_send", "fbr_lane_recv", "fbr_lane_poll", "fbr_queue_put", "fbr_queue_get", "fbr_queue_stats",
    "fbr_queue_destroy", "fbr_process_start", "fbr_process_poll", "fbr_process_join", "fbr_process_terminate",
    "fbr_process_handled", "fbr_process_destroy",
    "fbr_express_last_error", "fbr_express_create", "fbr_express_submit", "fbr_express_wait", "fbr_express_discard", "fbr_express_stats",
    "fbr_express_destroy",
    "fbr_comm_last_error", "fbr_comm_load", "fbr_comm_unique_id", "fbr_comm_create", "fbr_comm_info", "fbr_comm_sync",
    "fbr_comm_broadcast", "fbr_comm_allgather", "fbr_comm_gather", "fbr_comm_scatter", "fbr_comm_allreduce",
    "fbr_comm_allreduce_timed", "fbr_comm_allreduce_i64", "fbr_comm_allreduce_i64_begin", "fbr_comm_allreduce_i64_end",
    "fbr_comm_device_alloc", "fbr_comm_device_free",
    "fbr_comm_memcpy_h2d", "fbr_comm_memcpy_d2h", "fbr_comm_destroy",
]

FBR_REC_NONE, FBR_REC_INT, FBR_REC_FLOAT, FBR_REC_BYTES, FBR_REC_STR = range(5)
FBR_PROC_QUEUE_WORKER, FBR_PROC_PUT_QUEUE, FBR_PROC_GET_QUEUE, FBR_PROC_WRITE_PIPE, FBR_PROC_PIPE_WORKER = range(1, 6)


class Record(ctypes.Structure):
    _fields_ = [("tag", ctypes.c_uint32), ("len", ctypes.c_uint32), ("payload", ctypes.c_uint8 * 56)]


class BodyInfo(ctypes.Structure):
    _fields_ = [("func_id", ctypes.c_int32), ("arg_bytes", ctypes.c_uint32), ("result_bytes", ctypes.c_uint32),
                ("result_kind", ctypes.c_uint32), ("flags", ctypes.c_uint32), ("unit_tasks", ctypes.c_uint32),
                ("name", ctypes.c_char * 40)]


class MapDesc(ctypes.Structure):
    _fields_ = [("func_id", ctypes.c_int32), ("flags", ctypes.c_uint32), ("n_tasks", ctypes.c_uint64),
                ("chunksize", ctypes.c_uint32), ("arg_stride", ctypes.c_uint32), ("args", ctypes.c_void_p),
                ("index_start", ctypes.c_int64), ("index_step", ctypes.c_int64),
                ("shared", ctypes.c_void_p), ("shared_bytes", ctypes.c_uint64), ("out", ctypes.c_void_p),
                ("task_index_base", ctypes.c_uint64), ("shuffle_seed", ctypes.c_uint64), ("n_items", ctypes.c_uint64),
                ("attempt", ctypes.c_uint32), ("pad", ctypes.c_uint32)]


class Plan(ctypes.Structure):
    _fields_ = [("unit_tasks", ctypes.c_uint32), ("slot_stride", ctypes.c_uint32), ("n_units", ctypes.c_uint64),
                ("block_first", ctypes.c_uint64), ("block_count", ctypes.c_uint64)]


class Result(ctypes.Structure):
    _fields_ = [("seq", ctypes.c_uint64), ("n_tasks", ctypes.c_uint64), ("result_bytes", ctypes.c_uint32),
                ("result_kind", ctypes.c_uint32), ("data", ctypes.c_void_p), ("sum", ctypes.c_int64),
                ("err_code", ctypes.c_uint32), ("n_waves", ctypes.c_uint32), ("err_task", ctypes.c_uint64),
                ("sum_lo", ctypes.c_uint64), ("sum_hi", ctypes.c_int64), ("sum_overflow", ctypes.c_uint32),
                ("pad", ctypes.c_uint32)]


class Stats(ctypes.Structure):
    _fields_ = [("tasks_submitted", ctypes.c_uint64), ("tasks_completed", ctypes.c_uint64),
                ("units_dispatched", ctypes.c_uint64), ("dispatch_launches", ctypes.c_uint64),
                ("gather_launches", ctypes.c_uint64), ("fill_launches", ctypes.c_uint64),
                ("h2d_bytes", ctypes.c_uint64), ("d2h_bytes", ctypes.c_uint64),
                ("dispatch_ms", ctypes.c_double), ("gather_ms", ctypes.c_double),
                ("gather_bytes", ctypes.c_uint64), ("dispatch_bytes", ctypes.c_uint64),
                ("units_redispatched", ctypes.c_uint64), ("records_copied", ctypes.c_uint64),
                ("direct_waves", ctypes.c_uint64), ("peer_push_bytes", ctypes.c_uint64), ("workers_lost", ctypes.c_uint64)]

    def as_dict(self):
        return {name: getattr(self, name) for name, _ in self._fields_}


class EngineError(RuntimeError):
    """A libfiber_b200 call failed (``status`` is the negative ``fbr_status``)."""

    def __init__(self, status, message):
        super().__init__("%s (fbr_status %d)" % (message, status))
        self.status = status


_lib = None


def load():
    """Load libfiber_b200.so.  Fails loudly: this package has no CPU or eager fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "fiber_b200: %s is missing -- build it with `python -m fiber_b200.build` "
            "(needs nvcc; there is no CPU fallback)" % LIB_PATH)
    # resident device processes (queues.cu) must never meet a lazily loaded kernel: prefer eager
    # module loading when this is the first CUDA user in the process
    os.environ.setdefault("CUDA_MODULE_LOADING", "EAGER")
    L = ctypes.CDLL(LIB_PATH)
    vp, u64, i32, u32 = ctypes.c_void_p, ctypes.c_uint64, ctypes.c_int, ctypes.c_uint32
    P = ctypes.POINTER
    sig = {
        "fbr_abi_version": (i32, []),
        "fbr_last_error": (ctypes.c_char_p, []),
        "fbr_device_count": (i32, [P(i32)]),
        "fbr_body_count": (i32, [P(i32)]),
        "fbr_body_info": (i32, [i32, P(BodyInfo)]),
        "fbr_body_lookup": (i32, [ctypes.c_char_p, P(i32)]),
        "fbr_register_body": (i32, [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_char_p, P(i32)]),
        "fbr_pool_create": (i32, [i32, P(i32), u64, u32, P(vp)]),
        "fbr_pool_close": (i32, [vp]),
        "fbr_pool_terminate": (i32, [vp]),
        "fbr_pool_join": (i32, [vp]),
        "fbr_pool_destroy": (i32, [vp]),
        "fbr_pool_n_workers": (i32, [vp, P(i32)]),
        "fbr_pool_worker_device": (i32, [vp, i32, P(i32)]),
        "fbr_map_submit": (i32, [vp, P(MapDesc), P(u64)]),
        "fbr_shared_put": (i32, [vp, vp, u64, P(u64)]),
        "fbr_shared_drop": (i32, [vp, u64]),
        "fbr_plan_query": (i32, [i32, u64, u32, u64, i32, i32, i32, P(Plan)]),
        "fbr_result_wait": (i32, [vp, u64, i32, P(Result)]),
        "fbr_result_poll": (i32, [vp, u64, P(u64)]),
        "fbr_result_data": (i32, [vp, u64, P(vp)]),
        "fbr_result_fetch": (i32, [vp, u64, u64, u64, vp]),
        "fbr_result_release": (i32, [vp, u64]),
        "fbr_host_alloc": (i32, [vp, u64, P(vp)]),
        "fbr_host_free": (i32, [vp, vp]),
        "fbr_device_alloc": (i32, [vp, i32, u64, P(vp)]),
        "fbr_device_free": (i32, [vp, i32, vp]),
        "fbr_memcpy_h2d": (i32, [vp, i32, vp, vp, u64]),
        "fbr_memcpy_d2h": (i32, [vp, i32, vp, vp, u64]),
        "fbr_payload_fill_device": (i32, [vp, i32, vp, u64, u64]),
        "fbr_pool_stats": (i32, [vp, P(Stats)]),
        "fbr_pool_stats_reset": (i32, [vp]),
        "fbr_queue_last_error": (ctypes.c_char_p, []),
        "fbr_queue_create": (i32, [P(vp)]),
        "fbr_queue_open_writer": (i32, [vp, P(vp)]),
        "fbr_queue_open_reader": (i32, [vp, P(vp)]),
        "fbr_lane_send": (i32, [vp, P(Record), i32]),
        "fbr_lane_recv": (i32, [vp, P(Record), i32]),
        "fbr_lane_poll": (i32, [vp, P(i32)]),
        "fbr_queue_put": (i32, [vp, P(Record), i32]),
        "fbr_queue_get": (i32, [vp, P(Record), i32]),
        "fbr_queue_stats": (i32, [vp, P(u64), P(u32), P(u32)]),
        "fbr_queue_destroy": (i32, [vp]),
        "fbr_process_start": (i32, [i32, i32, vp, vp, ctypes.c_int64, P(Record), P(Record), u32, i32, P(vp)]),
        "fbr_process_poll": (i32, [vp, P(i32), P(i32)]),
        "fbr_process_join": (i32, [vp, i32]),
        "fbr_process_terminate": (i32, [vp]),
        "fbr_process_handled": (i32, [vp, P(u64)]),
        "fbr_process_destroy": (i32, [vp]),
        "fbr_express_last_error": (ctypes.c_char_p, []),
        "fbr_express_create": (i32, [i32, i32, P(vp)]),
        "fbr_express_submit": (i32, [vp, i32, ctypes.c_char_p, u32, P(u64)]),
        "fbr_express_wait": (i32, [vp, u64, vp, P(u32), P(u32), i32]),
        "fbr_express_discard": (i32, [vp, u64]),
        "fbr_express_stats": (i32, [vp, P(u64), P(u64), P(i32)]),
        "fbr_express_destroy": (i32, [vp]),
        "fbr_comm_last_error": (ctypes.c_char_p, []),
        "fbr_comm_load": (i32, [ctypes.c_char_p, P(i32)]),
        "fbr_comm_unique_id": (i32, [vp]),
        "fbr_comm_create": (i32, [i32, i32, i32, ctypes.c_char_p, P(vp)]),
        "fbr_comm_info": (i32, [vp, P(i32), P(i32), P(i32)]),
        "fbr_comm_sync": (i32, [vp]),
        "fbr_comm_broadcast": (i32, [vp, vp, u64, i32]),
        "fbr_comm_allgather": (i32, [vp, vp, vp, u64]),
        "fbr_comm_gather": (i32, [vp, vp, vp, u64, i32]),
        "fbr_comm_scatter": (i32, [vp, vp, vp, u64, i32]),
        "fbr_comm_allreduce": (i32, [vp, vp, vp, u64, i32, i32]),
        "fbr_comm_allreduce_timed": (i32, [vp, vp, u64, i32, i32, i32, P(ctypes.c_float)]),
        "fbr_comm_allreduce_i64": (i32, [vp, P(ctypes.c_int64)]),
        "fbr_comm_allreduce_i64_begin": (i32, [vp, ctypes.c_int64]),
        "fbr_comm_allreduce_i64_end": (i32, [vp, P(ctypes.c_int64)]),
        "fbr_comm_device_alloc": (i32, [vp, u64, P(vp)]),
        "fbr_comm_device_free": (i32, [vp, vp]),
        "fbr_comm_memcpy_h2d": (i32, [vp, vp, vp, u64]),
        "fbr_comm_memcpy_d2h": (i32, [vp, vp, vp, u64]),
        "fbr_comm_destroy": (i32, [vp]),
    }
    assert sorted(sig) == sorted(SYMBOLS)
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    if L.fbr_abi_version() != FBR_ABI_VERSION:
        raise RuntimeError("fiber_b200: ABI mismatch, rebuild with `python -m fiber_b200.build --force`")
    _lib = L
    return L


def check(status):
    if status != FBR_OK:
        raise EngineError(status, load().fbr_last_error().decode("utf-8", "replace"))
    return status


def xcheck(status):
    """Status check for the express-lane entry points (express.cu keeps its own error string)."""
    if status != FBR_OK:
        raise EngineError(status, load().fbr_express_last_error().decode("utf-8", "replace"))
    return status


def qcheck(status):
    """Status check for the queue / process entry points (queues.cu keeps its own error string)."""
    if status != FBR_OK:
        raise EngineError(status, load().fbr_queue_last_error().decode("utf-8", "replace"))
    return status
