"""``fiber_b200.Pool`` -- the reference's ``ZPool`` / ``ResilientZPool`` surface
(fiber/pool.py:881-1422, 1425-1688) on the B200 engine.

Same constructor, method names, defaults and exceptions as the reference:

* ``Pool(processes=None, initializer=None, initargs=(), maxtasksperchild=None, error_handling=False)``
  (fiber/context.py:38-45); ``processes=None`` means 1 (fiber/pool.py:894);
* ``map / map_async / starmap / starmap_async / apply / apply_async / imap / imap_unordered /
  close / terminate / join / start_workers / wait_until_workers_up``;
* ``chunksize=None`` -> 32 (fiber/pool.py:1169-1170), ``imap`` default chunksize 1 (:1218);
* ``ValueError("Pool is not running")`` once closed (:1107-1108, 1166-1167, 1284-1285);
  ``NotImplementedError`` for ``error_callback`` (:1162-1164); ``RuntimeError`` when a function
  with different ``__fiber_meta__`` arrives after the workers started (:1128-1133);
* workers start lazily on the first submission (:1122-1137).

What differs, by construction: a worker is a CUDA device, the mapped callable must be bound to a
compiled-in device body (``fiber_b200.device_body``), results come back as a buffer-backed
``ResultArray`` (list-like; ``.tolist()`` materialises the reference's list) instead of 1e8 Python
objects, and nothing on this path executes tasks on the CPU.
"""
import collections.abc
import ctypes
import math
import threading
import time

import numpy as np

from . import _abi, registry

RUN, CLOSE, TERMINATE = 0, 1, 2
DEFAULT_CHUNKSIZE = 32


class _Engine:
    """Owner of one ``fbr_pool_t``.  Destroyed when the last Python reference (pool or result
    segment) goes away, so result buffers never dangle."""

    def __init__(self, n_workers, devices, ring_bytes, timing):
        self.lib = _abi.load()
        ids = (ctypes.c_int * n_workers)(*devices)
        handle = ctypes.c_void_p()
        _abi.check(self.lib.fbr_pool_create(n_workers, ids, ring_bytes, _abi.FBR_POOL_TIMING if timing else 0,
                                            ctypes.byref(handle)))
        self.handle = handle
        self.n_workers = n_workers
        self.devices = list(devices)
        self.lock = threading.Lock()

    def __del__(self):
        h, self.handle = getattr(self, "handle", None), None
        if h:
            self.lib.fbr_pool_destroy(h)


class _Segment:
    """Owner of one map's engine state (its seq: control slots, events, pinned result segment) from the
    moment it is submitted.  Once the map has finished, ``bind`` exposes the pinned segment through
    ``__array_interface__`` so NumPy views keep it (and through it the engine) alive.  Dropping the last
    reference -- a fetched result going away, but also a fire-and-forget ``map_async`` or an abandoned
    ``imap`` generator -- releases the seq (``self._inventory[job_seq] = None``, fiber/pool.py:677-679)."""

    def __init__(self, engine, seq):
        self.engine, self.seq, self.ptr, self.nbytes = engine, seq, None, 0

    def bind(self, ptr, nbytes):
        self.ptr, self.nbytes = ptr, nbytes
        self.__array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr or 0, False), "version": 3}
        return self

    def __del__(self):
        eng = getattr(self, "engine", None)
        if eng is not None and eng.handle:
            eng.lib.fbr_result_release(eng.handle, self.seq)


class _PinnedBlock:
    """Pinned host block from the engine's segment cache (``fbr_host_alloc``): NumPy views keep it
    alive, garbage collection returns it.  Arguments that live here are DMA'd straight to the device
    (no staging copy) -- the host end of the pinned task ring."""

    def __init__(self, engine, nbytes):
        self.engine = engine
        ptr = ctypes.c_void_p()
        _abi.check(engine.lib.fbr_host_alloc(engine.handle, max(1, nbytes), ctypes.byref(ptr)))
        self.ptr = ptr.value
        self.__array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (self.ptr, False), "version": 3}

    def __del__(self):
        eng = getattr(self, "engine", None)
        if eng is not None and eng.handle and getattr(self, "ptr", None):
            eng.lib.fbr_host_free(eng.handle, ctypes.c_void_p(self.ptr))


class ResultArray(collections.abc.Sequence):
    """Ordered results of one map, backed by the pinned result segment (no per-item Python
    objects).  Behaves like the list the reference returns: indexing, slicing, iteration, ``len``,
    ``==`` against lists; ``tolist()`` materialises it; ``sum()`` returns the device-side sum folded
    by ``gather_ordered`` when available.

    With ``Pool(results="device")`` the ordered results stay in HBM: ``sum()`` and ``len()`` cost
    nothing, indexing fetches just the requested range, and the full array crosses PCIe only when
    something needs all of it (``array``, ``tolist()``, iteration, ``==``)."""

    def __init__(self, spec, array, device_sum=None, n=None, fetch=None, bits=None):
        self._spec = spec
        self._arr = array
        self._sum = device_sum
        self._n = len(array) if array is not None else n
        self._fetch = fetch            # (lo, hi) -> ndarray, for device-resident results
        self._bits = bits              # Pool(results="bits"): uint8[ceil(n/8)], bit k of byte j = result 8j+k

    @property
    def _a(self):
        if self._arr is None:
            if self._bits is not None:
                self._arr = np.unpackbits(self._bits, count=self._n, bitorder="little").view(np.bool_)
            else:
                self._arr = self._fetch(0, self._n)
        return self._arr

    @property
    def packed(self):
        """The bit-packed results (``Pool(results="bits")``): zero-copy uint8 view of the pinned
        segment, result i at bit ``i & 7`` of byte ``i >> 3``; ``None`` for byte-per-result maps."""
        return self._bits

    @property
    def on_device(self):
        return self._arr is None and self._bits is None

    def __len__(self):
        return self._n

    def __getitem__(self, i):
        if self._arr is None and self._bits is not None:
            # bit-backed: single results and contiguous ranges are read straight from the packed bytes
            if isinstance(i, slice):
                lo, hi, step = i.indices(self._n)
                if step == 1:
                    hi = max(lo, hi)
                    part = np.unpackbits(self._bits[lo >> 3:(hi + 7) >> 3], bitorder="little")
                    return part[lo & 7:(lo & 7) + hi - lo].view(np.bool_).tolist()
            else:
                j = i + self._n if i < 0 else i
                if not 0 <= j < self._n:
                    raise IndexError("ResultArray index out of range")
                return bool((int(self._bits[j >> 3]) >> (j & 7)) & 1)
        elif self._arr is None:
            if isinstance(i, slice):
                lo, hi, step = i.indices(self._n)
                if step == 1:
                    return self._spec.rows_to_list(self._fetch(lo, max(lo, hi)))
            else:
                j = i + self._n if i < 0 else i
                if not 0 <= j < self._n:
                    raise IndexError("ResultArray index out of range")
                return self._spec.to_python(self._fetch(j, j + 1)[0])
        if isinstance(i, slice):
            return self._spec.rows_to_list(self._a[i])
        return self._spec.to_python(self._a[i])

    def __iter__(self):
        step = 1 << 16
        for s in range(0, self._n, step):
            yield from self[s:s + step]

    def __eq__(self, other):
        if isinstance(other, ResultArray):
            if self._bits is not None and other._bits is not None:
                return self._n == other._n and np.array_equal(self._bits, other._bits)
            return np.array_equal(self._a, other._a)
        if isinstance(other, (list, tuple)):
            return len(other) == len(self) and self.tolist() == list(other)
        return NotImplemented

    def __repr__(self):
        n = len(self)
        head = self[:6]
        return "ResultArray(%s%s, len=%d, body=%s%s)" % (head, "..." if n > 6 else "", n, self._spec.name,
                                                         ", bit-packed" if self._bits is not None else
                                                         ", on device" if self.on_device else "")

    def __array__(self, dtype=None, copy=None):
        a = self._a
        return a.astype(dtype) if dtype is not None else a

    @property
    def array(self):
        """Zero-copy NumPy view of the pinned result segment (fetches device-resident results)."""
        return self._a

    def tolist(self):
        return self._spec.rows_to_list(self._a)

    def sum(self):
        if self._sum is not None:
            return self._sum
        py_sum = getattr(self._spec, "py_sum", None)
        if py_sum is not None:          # record bodies: the builtin's sum of the list (floats left to right, tuples raise)
            return py_sum(self)
        if self._bits is not None:
            return int(np.unpackbits(self._bits).sum())   # the bits past n are zero
        if self._a.dtype.kind in "iu" and self._a.dtype.itemsize == 8:
            # int64 results: NumPy's sum wraps silently, Python's sum of the reference's list does not
            lo = int((self._a.view(np.uint64) & np.uint64(0xFFFFFFFF)).sum(dtype=np.uint64))
            hi = int((self._a.view(np.int64) >> np.int64(32)).sum(dtype=np.int64))
            return hi * (1 << 32) + lo
        return int(self._a.sum())

    def sort(self):
        raise TypeError("ResultArray is read-only; use sorted(result) or result.tolist()")


class MapResult:
    """Handle of an asynchronous map (fiber/pool.py:731-743)."""

    def __init__(self, pool, engine, spec, seq, n, keepalive):
        self._pool, self._engine, self._spec, self._seq, self._n = pool, engine, spec, seq, n
        self._keepalive = keepalive   # argument buffers must outlive the asynchronous H2D copies
        self._result = None
        self._exc = None              # a task error is raised again by every later get()
        self._segment = _Segment(engine, seq) if n else None   # owns the seq from submission on
        self._yielded = False
        self._n_items = None          # bit-packed maps: number of range() indices (n = ceil(n_items / 8) byte tasks)
        self._user_spec = spec

    # -- internal ----------------------------------------------------------------------------
    def _wait(self, timeout=None):
        if self._result is not None:
            return self._result
        if self._exc is not None:
            raise self._exc
        if self._n == 0:
            us = self._user_spec
            self._result = ResultArray(us, np.empty((0,) + us.result_dtype()[1], us.result_dtype()[0]), 0)
            return self._result
        res = _abi.Result()
        eng = self._engine
        tmo = -1 if timeout is None else int(timeout * 1000)
        rc = eng.lib.fbr_result_wait(eng.handle, self._seq, tmo, ctypes.byref(res))
        if rc == _abi.FBR_ETIMEOUT:
            raise TimeoutError("map %d not finished" % self._seq)
        if rc == _abi.FBR_ETASK:
            try:
                self._raise_task_error(res)
            except Exception as e:      # noqa: BLE001 -- remembered: later get() calls raise it without touching the engine
                self._exc = e
                raise
        _abi.check(rc)
        self._keepalive = None
        self._pool.recv_tasks += self._n if self._n_items is None else self._n_items
        dtype, sub = self._spec.result_dtype()
        # exact, unbounded sum: the device folds the two halves of int64 results separately (nothing wraps)
        dsum = (int(res.sum_hi) * (1 << 32) + int(res.sum_lo)) if (self._flags & _abi.FBR_WANT_SUM) else None
        self.n_waves = res.n_waves
        if self._flags & _abi.FBR_RESULTS_ON_DEVICE:
            seg = self._segment                              # owns the seq (device buffer) until GC
            rb, seq = res.result_bytes, self._seq

            def fetch(lo, hi, seg=seg):
                block = _PinnedBlock(eng, max(1, (hi - lo) * rb))
                if hi > lo:
                    _abi.check(eng.lib.fbr_result_fetch(eng.handle, seq, lo, hi - lo, ctypes.c_void_p(block.ptr)))
                return np.asarray(block)[: (hi - lo) * rb].view(dtype).reshape((hi - lo,) + sub)
            self._result = ResultArray(self._spec, None, dsum, n=int(res.n_tasks), fetch=fetch)
            return self._result
        seg = self._segment.bind(res.data, res.n_tasks * res.result_bytes)
        arr = np.asarray(seg).view(dtype).reshape((res.n_tasks,) + sub)
        if self._n_items is not None:
            # bit-packed map (pi_inside_bits8): `arr` holds ceil(n/8) bytes.  The body evaluated all 8
            # indices of the last byte; the ones past the end of the range are dropped here, from the
            # byte and from the folded count.
            n, extra = self._n_items, (-self._n_items) % 8
            if extra:
                last = int(arr[-1])
                keep = last & (0xFF >> extra)
                if dsum is not None:
                    dsum -= bin(last ^ keep).count("1")
                arr[-1] = keep
            self._result = ResultArray(self._user_spec, None, dsum, n=n, bits=arr)
            return self._result
        self._result = ResultArray(self._spec, arr, dsum)
        return self._result

    def _raise_task_error(self, res):
        code, task = res.err_code, res.err_task
        name = getattr(self, "_user_spec", self._spec).name     # the body the caller mapped (not its bit-packed twin)
        if code == _abi.FBR_TASK_OVERFLOW:
            raise OverflowError("%s: result of task %d does not fit int64 (Python ints are unbounded; "
                                "the device body refuses to wrap)" % (name, task))
        if code == _abi.FBR_TASK_BADARG:
            raise ValueError("%s: bad argument in task %d" % (name, task))
        raise RuntimeError("%s: task %d failed with device error code %d" % (name, task, code))

    # -- reference surface -------------------------------------------------------------------
    def get(self, timeout=None):
        return self._wait(timeout)

    def _iter_ready(self):
        """Yield results as ordered prefixes become final (per-wave completion events)."""
        if self._n == 0:
            return
        if self._flags & _abi.FBR_RESULTS_ON_DEVICE:
            yield from self._wait()
            return
        eng = self._engine
        if self._n_items is not None:
            # bit-packed map: progress is counted in result bytes (8 tasks each); every byte of a finished
            # wave is a full byte, the (masked) last byte of the map only comes from _wait()
            done, emitted = ctypes.c_uint64(0), 0
            while emitted < self._n:
                _abi.check(eng.lib.fbr_result_poll(eng.handle, self._seq, ctypes.byref(done)))
                if done.value >= self._n:
                    break
                if done.value > emitted:
                    part = self._peek(emitted, done.value, np.dtype(np.uint8), ())
                    yield from np.unpackbits(part, bitorder="little").view(np.bool_).tolist()
                    emitted = done.value
                else:
                    time.sleep(0.0002)
            res = self._wait()
            if emitted * 8 < self._n_items:
                yield from res[emitted * 8:]
            return
        done = ctypes.c_uint64(0)
        emitted = 0
        dtype, sub = self._spec.result_dtype()
        # peek at the segment: results land in it wave by wave
        while emitted < self._n:
            _abi.check(eng.lib.fbr_result_poll(eng.handle, self._seq, ctypes.byref(done)))
            if done.value >= self._n:
                break
            if done.value > emitted:
                # an ordered prefix is final but the map is not: hand it out from the live segment
                part = self._peek(emitted, done.value, dtype, sub)
                yield from self._spec.rows_to_list(part)
                emitted = done.value
            else:
                time.sleep(0.0002)
        res = self._wait()
        if emitted < self._n:
            yield from self._spec.rows_to_list(res.array[emitted:])

    def _peek(self, lo, hi, dtype, sub):
        base = self._pool._segment_ptr(self._seq)
        rb = self._spec.result_bytes
        buf = (ctypes.c_char * ((hi - lo) * rb)).from_address(base + lo * rb)
        return np.frombuffer(buf, dtype=dtype).reshape((hi - lo,) + sub).copy()

    def iget_ordered(self):
        return self._iter_ready()

    def iget_unordered(self):
        # arrival order == ring order; ordered prefixes are a valid "unordered" stream
        return self._iter_ready()


class ApplyResult(MapResult):
    """fiber/pool.py:746-757: ``get()`` returns the single element."""

    def get(self, timeout=None):
        return self._wait(timeout)[0]


class _Express:
    """Owner of one ``fbr_express_t``: the doorbell lane of one device (resident one-warp kernel)."""
    BODIES = ("square_i64", "mul2_i64", "square_scale_i64", "identity_i64", "pi_inside_det", "sleep_f64")

    def __init__(self, device, idle_us):
        self.lib = _abi.load()
        h = ctypes.c_void_p()
        _abi.xcheck(self.lib.fbr_express_create(device, idle_us, ctypes.byref(h)))
        self.handle = h

    def stats(self):
        served, launches, resident = ctypes.c_uint64(), ctypes.c_uint64(), ctypes.c_int()
        _abi.xcheck(self.lib.fbr_express_stats(self.handle, ctypes.byref(served), ctypes.byref(launches), ctypes.byref(resident)))
        return {"served": served.value, "kernel_launches": launches.value, "resident": bool(resident.value)}

    def __del__(self):
        h, self.handle = getattr(self, "handle", None), None
        if h:
            self.lib.fbr_express_destroy(h)


class ExpressResult:
    """``ApplyResult`` (fiber/pool.py:746-757) of a task sent through the doorbell lane."""

    def __init__(self, pool, express, spec, ticket):
        self._pool, self._x, self._spec, self._ticket = pool, express, spec, ticket
        self._done, self._value, self._exc = False, None, None

    def __del__(self):
        # handle dropped without a get(): tell the lane to forget the response instead of parking it forever
        x = getattr(self, "_x", None)
        if x is not None and not getattr(self, "_done", True) and x.handle:
            x.lib.fbr_express_discard(x.handle, self._ticket)

    def get(self, timeout=None):
        if self._done:
            if self._exc is not None:
                raise self._exc
            return self._value
        buf = (ctypes.c_uint8 * 48)()
        nbytes, err = ctypes.c_uint32(), ctypes.c_uint32()
        rc = self._x.lib.fbr_express_wait(self._x.handle, self._ticket, buf, ctypes.byref(nbytes), ctypes.byref(err),
                                          -1 if timeout is None else int(timeout * 1000))
        if rc == _abi.FBR_ETIMEOUT:
            raise TimeoutError("apply %d not finished" % self._ticket)
        if rc == _abi.FBR_ETASK:
            self._done = True
            res = _abi.Result()
            res.err_code, res.err_task = err.value, 0
            try:
                MapResult._raise_task_error(self, res)
            except Exception as e:      # noqa: BLE001 -- remembered so that a second get() raises again
                self._exc = e
                raise
        _abi.xcheck(rc)
        self._value, self._done = self._spec.unpack_result(bytes(buf[: nbytes.value])), True
        self._pool.recv_tasks += 1
        return self._value


class Pool:
    """B200-native drop-in for ``fiber.Pool`` on the map/starmap/apply path."""

    def __init__(self, processes=None, initializer=None, initargs=(), maxtasksperchild=None,
                 error_handling=False, *, devices=None, ring_bytes=0, timing=False, results="host", express=True,
                 express_idle_us=2000, bind_cpu=False, isolation="thread"):
        self._processes = processes if processes is not None else 1   # fiber/pool.py:894
        if self._processes < 1:
            raise ValueError("Number of processes must be at least 1")
        if initializer is not None and getattr(initializer, "__fbr_init_body__", None) is None:
            # the reference runs initializer(*initargs) inside every worker process
            # (fiber/pool.py:858-859); a host callable cannot run inside a GPU worker.  What the idiom is
            # for -- giving every task the same large arguments once -- is the engine's broadcast block:
            # see fiber_b200.device_initializer.
            raise NotImplementedError("fiber_b200.Pool: Python initializers cannot run on GPU workers; bind the "
                                      "initializer with @fiber_b200.device_initializer(body) to upload initargs as "
                                      "the body's broadcast block")
        self._initializer, self._initargs = initializer, initargs
        self._init_block = None   # (body name, blob, handle): initargs uploaded once per worker at start
        self._maxtasksperchild = maxtasksperchild
        self._error_handling = bool(error_handling)
        self._devices = list(devices) if devices is not None else None
        self._ring_bytes = int(ring_bytes)
        self._timing = bool(timing)
        if results not in ("host", "bytes", "device", "bits"):
            raise ValueError("results must be 'host' (pinned result segment; bool results packed one bit each), "
                             "'bytes' (pinned result segment, one byte per bool), 'device' (stay in HBM, fetched "
                             "lazily) or 'bits' (same as 'host')")
        self._results_on_device = results == "device"
        # A bool needs one bit: bool bodies with a bit-packed twin run through it by default, so the ring, the
        # ordered output and the D2H copy move n/8 bytes.  ResultArray hides the layout; 'bytes' opts out.
        self._results_bits = results in ("host", "bits")
        self._use_express = bool(express) and not self._error_handling
        self._express_idle_us = int(express_idle_us)
        self._express = None
        if isolation not in ("thread", "process"):
            raise ValueError("isolation must be 'thread' (workers are devices of this process) or 'process' (one worker process "
                             "per GPU: the only fault domain CUDA offers -- see fiber_b200/procpool.py)")
        self._isolation = isolation
        self._proc = None                    # ProcessPool when isolation == "process"
        self._attempt = 0                    # re-dispatch count stamped on submitted blocks (set by process-pool workers)
        self._bind_cpu = bool(bind_cpu)      # one process per GPU: keep pinned segments on the GPU's NUMA node
        self.bound_cpus = []
        self._state = RUN
        self._engine = None
        self._worker_handler_started = False
        self._meta = None
        self._live = {}         # seq -> data pointer of the engine-owned segment (for imap peeks)
        self._shared_cache = collections.OrderedDict()
        self.sent_tasks = 0     # fiber/pool.py:902-903
        self.recv_tasks = 0

    def __repr__(self):
        return "<{}({}, {})>".format(type(self).__name__, self._processes,
                                     self._engine.devices if self._engine else None)

    # -- workers (fiber/pool.py:1118-1137, 1405-1422) ---------------------------------------------
    def start_workers(self):
        if self._isolation == "process":
            if self._proc is None:
                from .procpool import ProcessPool
                lib = _abi.load()
                n = ctypes.c_int(0)
                _abi.check(lib.fbr_device_count(ctypes.byref(n)))            # counts devices, creates no context
                if n.value == 0:
                    raise _abi.EngineError(_abi.FBR_ENODEV, "no CUDA device visible; fiber_b200 has no CPU fallback")
                devs = self._devices if self._devices is not None else list(range(n.value))
                self._proc = ProcessPool(self._processes, devs, results="bytes" if not self._results_bits else "host",
                                         redispatch=self._error_handling)
            self._proc.start()
            self._worker_handler_started = True
            return
        if self._engine is None:
            lib = _abi.load()
            n = ctypes.c_int(0)
            _abi.check(lib.fbr_device_count(ctypes.byref(n)))
            if self._devices is not None:
                devs = self._devices
            else:
                # one worker per GPU; more requested processes than GPUs fold onto the GPUs we have
                devs = list(range(min(self._processes, n.value)))
            if self._bind_cpu and len(devs) == 1:
                from .affinity import bind_to_device
                self.bound_cpus = bind_to_device(devs[0])
            self._engine = _Engine(len(devs), devs, self._ring_bytes, self._timing)
            if self._initializer is not None:
                # initializer(*initargs) in every worker (fiber/pool.py:858-859) == one broadcast block per device
                body = self._initializer.__fbr_init_body__
                blob = registry.spec(body).shared_block(*self._initargs)
                self._init_block = (body, blob, self._shared_handle(blob))
        self._worker_handler_started = True

    def lazy_start_workers(self, func):
        meta = getattr(func, "__fiber_meta__", None)
        if meta is not None and meta != self._meta:
            if self._worker_handler_started and self._meta is not None:
                raise RuntimeError(
                    "Cannot run function that has different resource "
                    "requirements acceptable by this pool. Try creating a "
                    "different pool for it.")
            self._meta = meta
        if not self._worker_handler_started:
            self.start_workers()

    def wait_until_workers_up(self):
        self.start_workers()
        if self._proc is not None:
            self._proc.wait_until_workers_up()

    @property
    def n_jobs(self):
        """Jobs the reference would start for this pool: ceil(processes / cpu_per_job)
        (fiber/pool.py:1405-1408)."""
        from . import config
        return n_jobs(self._processes, config.cpu_per_job)

    @property
    def n_workers(self):
        self.start_workers()
        return self._engine.n_workers

    # -- submission ----------------------------------------------------------------------------------
    def _check_running(self):
        if self._state != RUN:
            raise ValueError("Pool is not running")

    def _shared_handle(self, blob):
        # the very same bytes object as last time (the encoder's block cache): no need to fingerprint 80-160 KB again
        last = getattr(self, "_last_shared", None)
        if last is not None and last[0] is blob and last[1] in self._shared_cache:
            return self._shared_cache[last[1]]
        key = registry.fingerprint(blob)
        self._last_shared = (blob, key)
        hit = self._shared_cache.get(key)
        if hit is not None:
            self._shared_cache.move_to_end(key)
            return hit
        eng = self._engine
        buf = np.frombuffer(blob, dtype=np.uint8)
        h = ctypes.c_uint64(0)
        _abi.check(eng.lib.fbr_shared_put(eng.handle, buf.ctypes.data, buf.nbytes, ctypes.byref(h)))
        self._shared_cache[key] = h.value
        while len(self._shared_cache) > 8:
            _, old = self._shared_cache.popitem(last=False)
            eng.lib.fbr_shared_drop(eng.handle, old)
        return h.value

    def _submit(self, func, enc, kind, chunksize, cls=MapResult, want_sum=True, extra_flags=0, spec=None):
        spec = spec or registry.spec(registry.body_name_of(func))
        eng = self._engine
        d = _abi.MapDesc()
        d.func_id = spec.func_id
        flags = kind | extra_flags
        if self._results_on_device:
            flags |= _abi.FBR_RESULTS_ON_DEVICE
        if self._error_handling:
            # ResilientZPool (fiber/context.py:42-43): units whose worker dies are re-dispatched
            flags |= _abi.FBR_RESILIENT
        if want_sum and (spec.flags & _abi.FBR_BODY_SUMMABLE):
            flags |= _abi.FBR_WANT_SUM
        d.n_tasks = enc.n
        d.chunksize = chunksize
        d.arg_stride = enc.arg_stride
        keep = [enc.args]
        if enc.args is not None and enc.n:
            d.args = enc.args.ctypes.data
        d.index_start, d.index_step = enc.index_start, enc.index_step
        if enc.shared is not None:
            d.shared = self._shared_handle(enc.shared)
            d.shared_bytes = len(enc.shared)
            flags |= _abi.FBR_SHARED_HANDLE
        elif spec.flags & _abi.FBR_BODY_NEEDS_SHARED:
            # tasks without their own shared arguments read the block the pool's initializer uploaded
            if self._init_block is None or self._init_block[0] != spec.name:
                raise TypeError("%s: tasks carry no shared arguments and the pool has no initializer block for this "
                                "body (Pool(initializer=<@device_initializer(%r)>, initargs=...))" % (spec.name, spec.name))
            d.shared = self._shared_handle(self._init_block[1])
            d.shared_bytes = len(self._init_block[1])
            flags |= _abi.FBR_SHARED_HANDLE
        d.n_items = enc.n_items
        d.task_index_base = enc.task_index_base
        d.attempt = self._attempt
        d.flags = flags
        seq = ctypes.c_uint64(0)
        if enc.n:
            _abi.check(eng.lib.fbr_map_submit(eng.handle, ctypes.byref(d), ctypes.byref(seq)))
        self.sent_tasks += enc.n
        r = cls(self, eng, spec, seq.value, enc.n, keep)
        r._flags = flags
        return r

    def _segment_ptr(self, seq):
        # results are written into the engine-owned pinned segment wave by wave
        eng = self._engine
        ptr = ctypes.c_void_p()
        _abi.check(eng.lib.fbr_result_data(eng.handle, seq, ctypes.byref(ptr)))
        return ptr.value

    @staticmethod
    def _spec_of(func):
        return registry.spec(registry.body_name_of(func))

    def map_async(self, func, iterable, chunksize=None, callback=None, error_callback=None, _streaming=False):
        if error_callback:
            raise NotImplementedError
        self._check_running()
        if chunksize is None:
            chunksize = DEFAULT_CHUNKSIZE
        if not hasattr(iterable, "__len__"):
            iterable = list(iterable)
        spec = self._spec_of(func)
        self.lazy_start_workers(func)
        if self._proc is not None:
            return self._submit_proc(spec, "map", iterable, chunksize)
        enc = spec.encode_map(iterable)
        # imap wants ordered prefixes as they complete: results are staged and copied out wave by wave instead of being
        # stored straight into the pinned segment by one kernel (zero copy, final only when the whole block is)
        extra = _abi.FBR_NO_ZERO_COPY if _streaming else 0
        if self._results_bits and spec.name in registry.BITS_TWIN:
            return self._submit_bits(func, spec, enc, _abi.FBR_MAP, chunksize, extra)
        return self._submit(func, enc, _abi.FBR_MAP, chunksize, extra_flags=extra)

    def _submit_proc(self, spec, kind, items, chunksize, single=False):
        """Process-isolated workers: the map is cut into blocks that worker processes pull (procpool.py)."""
        if not isinstance(items, (range, list, np.ndarray)):
            items = list(items)
        if kind == "map" and len(items):
            spec.encode_map(items[:1] if not isinstance(items, range) else items)      # argument validation up front
        twin = registry.BITS_TWIN.get(spec.name) if (self._results_bits and kind != "apply") else None
        r = self._proc.submit(spec, twin, kind, items, chunksize, single)
        self.sent_tasks += len(items)
        return r

    def _submit_bits(self, func, spec, enc, kind, chunksize, extra_flags=0):
        """A bool needs one bit: the twin body evaluates 8 consecutive items (range() indices or argument
        records) per result byte, so the ring, the ordered output and the D2H copy move n/8 bytes."""
        twin = registry.spec(registry.BITS_TWIN[spec.name])
        n_items = enc.n
        r = self._submit(func, twin.from_encoded(enc), kind, max(1, chunksize // 8), spec=twin, extra_flags=extra_flags)
        r._n_items, r._user_spec = n_items, spec
        self.sent_tasks += n_items - r._n
        return r

    def map(self, func, iterable, chunksize=None):
        return self.map_async(func, iterable, chunksize).get()

    def starmap_async(self, func, iterable, chunksize=None, callback=None, error_callback=None):
        self._check_running()
        if chunksize is None:
            chunksize = DEFAULT_CHUNKSIZE
        if not hasattr(iterable, "__len__"):
            iterable = list(iterable)
        spec = self._spec_of(func)
        self.lazy_start_workers(func)
        if self._proc is not None:
            return self._submit_proc(spec, "starmap", list(iterable), chunksize)
        enc = spec.encode_starmap(iterable)
        if self._results_bits and spec.name in registry.BITS_TWIN:
            return self._submit_bits(func, spec, enc, _abi.FBR_STARMAP, chunksize)
        return self._submit(func, enc, _abi.FBR_STARMAP, chunksize)

    def starmap(self, func, iterable, chunksize=None):
        return self.starmap_async(func, iterable, chunksize).get()

    def apply_async(self, func, args=(), kwds={}, callback=None, error_callback=None):
        self._check_running()
        spec = self._spec_of(func)
        self.lazy_start_workers(func)
        if self._proc is not None:
            return self._submit_proc(spec, "apply", [(tuple(args), dict(kwds))], 1, single=True)
        if self._use_express and spec.name in _Express.BODIES:
            # one task whose record fits the doorbell lane: no kernel launch / copy on the round trip
            rec = spec.pack_apply(args, kwds)
            if self._express is None:
                self._express = _Express(self._engine.devices[0], self._express_idle_us)
            ticket = ctypes.c_uint64()
            _abi.xcheck(self._express.lib.fbr_express_submit(self._express.handle, spec.func_id, rec, len(rec),
                                                             ctypes.byref(ticket)))
            self.sent_tasks += 1
            return ExpressResult(self, self._express, spec, ticket.value)
        return self._submit(func, spec.encode_apply(args, kwds), _abi.FBR_APPLY, 1, cls=ApplyResult, want_sum=False)

    def apply(self, func, args=(), kwds={}):
        return self.apply_async(func, args, kwds).get()

    def imap(self, func, iterable, chunksize=1):
        r = self.map_async(func, iterable, chunksize, _streaming=True)
        return iter(r.get()) if self._proc is not None else r.iget_ordered()

    def imap_unordered(self, func, iterable, chunksize=1):
        r = self.map_async(func, iterable, chunksize, _streaming=True)
        return iter(r.get()) if self._proc is not None else r.iget_unordered()

    # -- shutdown (fiber/pool.py:1332-1403) -----------------------------------------------------------
    def close(self):
        if self._state == RUN:
            self._state = CLOSE
            if self._proc is not None:
                self._proc.close()
            if self._engine is not None:
                self._engine.lib.fbr_pool_close(self._engine.handle)

    def terminate(self):
        self._state = TERMINATE
        if self._proc is not None:
            self._proc.terminate()
        if self._engine is not None:
            self._engine.lib.fbr_pool_terminate(self._engine.handle)

    def join(self):
        assert self._state in (TERMINATE, CLOSE)
        if self._proc is not None:
            self._proc.join()
        if self._engine is not None:
            _abi.check(self._engine.lib.fbr_pool_join(self._engine.handle))

    # -- extras ------------------------------------------------------------------------------------------
    def pinned_empty(self, shape, dtype=np.uint8):
        """NumPy array in pinned host memory owned by this pool: argument records built in it are
        copied to the GPU by DMA without an intermediate staging copy."""
        self.start_workers()
        dtype = np.dtype(dtype)
        shape = (shape,) if isinstance(shape, int) else tuple(shape)
        nbytes = int(np.prod(shape, dtype=np.int64)) * dtype.itemsize
        block = _PinnedBlock(self._engine, nbytes)
        return np.asarray(block).view(dtype).reshape(shape)

    def stats(self):
        """``fbr_pool_stats`` as a dict (extends the reference's sent_tasks/recv_tasks counters)."""
        self.start_workers()
        if self._proc is not None:
            return dict(self._proc.stats)
        s = _abi.Stats()
        _abi.check(self._engine.lib.fbr_pool_stats(self._engine.handle, ctypes.byref(s)))
        d = s.as_dict()
        if self._express is not None:
            d["express"] = self._express.stats()
        return d

    def reset_stats(self):
        self.start_workers()
        _abi.check(self._engine.lib.fbr_pool_stats_reset(self._engine.handle))


def n_jobs(processes, cpu_per_job=1):
    """Number of job-backed workers the reference would start (fiber/pool.py:1405-1408)."""
    return math.ceil(float(processes) / cpu_per_job)
