"""Callable -> device-body registry and fixed-layout record encoders.

The reference ships the mapped callable to its workers by pickle reference and calls it there
(fiber/pool.py:961, 806-820).  A Python callable cannot execute on a GPU, so a callable has to be
*bound* to one of the device bodies compiled into libfiber_b200 (``fbr_body_lookup``).  The hook is
the one the reference already inspects when it starts workers: ``func.__fiber_meta__``
(fiber/meta.py:53-56, fiber/pool.py:1122-1137).  ``device_body`` / ``bind`` add ``__fbr_body__``.

An unbound callable raises ``TypeError`` -- there is no CPU fallback.

Encoders turn the Python-level task arguments (what the reference would pickle,
fiber/pool.py:1181,1297-1301,1112-1113) into fixed-layout argument records.
"""
import hashlib
import struct

import numpy as np

from . import _abi

_BOUND = {}  # callables that cannot carry attributes (builtins) -> body name


def device_body(name, source=None, entry="fbr_body_entry", args="i64", bits_entry=None, result=None, **meta):
    """Decorator: ``@device_body("pi_inside_det")`` binds ``func`` to the device body ``name`` and sets
    ``func.__fiber_meta__`` (``gpu=1`` unless overridden), like ``fiber.meta``.

    ``source=`` makes it an OUT-OF-TREE body: CUDA source of a translation unit that includes
    ``fiber_b200_body.cuh``, defines a ThreadBody and exports it with
    ``FBR_EXPORT_THREAD_BODY(Body, "<name>", <entry>, kind, flags)``.  It is compiled for sm_100a with
    nvcc (cached by content hash under ``fiber_b200/_lib/bodies/``) and registered with
    ``fbr_register_body`` -- the reference ships any callable to its workers (fiber/pool.py:961); this is
    how a callable that is not compiled into libfiber_b200 gets its device code there.  ``args`` names the
    argument record layout: ``"i64"`` (one int) or ``"i64x2"`` (two ints).  A bool body may also export its
    bit-packed twin (``FBR_EXPORT_BOOL_BODY_BITS(Body, "<name>_bits8", <bits_entry>, flags)``): pass ``bits_entry``
    and its results travel one bit each, like the compiled-in bool body's.

    A body of floats or small structs (``FBR_EXPORT_RECORD_BODY``) declares its records as NumPy dtypes:
    ``args=`` and ``result=`` take anything ``np.dtype()`` accepts -- ``"f8"``, ``"<f4"``, ``"i4"``, ``"3f4"`` (a packed
    float3) or a structured list of named fields -- and must match the module's ``arg_bytes`` / ``result_bytes``.
    Its tasks are encoded as records (``map``: one record per item, NumPy arrays of the record layout without a copy;
    ``starmap`` / ``apply``: the positional arguments are the fields in order, keywords name them) and its results
    decode to Python floats / ints, or tuples for multi-field records."""
    from .meta import VALID_META_KEYS
    for k in meta:
        assert k in VALID_META_KEYS, "Invalid meta argument \"{}\"".format(k)
    md = {"gpu": 1}
    md.update(meta)
    if source is not None:
        from . import bodies
        register_module(name, bodies.compile_module(name, source), entry, args, bits_entry, result)

    def decorator(func):
        bind(func, name, **md)
        return func
    return decorator


_MODULES = {}   # body name -> (module path, entry, argument layout, bits entry, result layout) of bodies registered
                # from their own module


def module_of(name):
    """Where an out-of-tree body came from (worker processes of a process-isolated pool register it themselves)."""
    return _MODULES.get(name)


def register_module(name, module_path, entry="fbr_body_entry", args="i64", bits_entry=None, result=None):
    """``fbr_register_body`` + the host-side encoder for the body's argument records (and, with ``bits_entry``, the
    body's bit-packed twin ``<name>_bits8``).  ``args`` is ``"i64"``, ``"i64x2"`` or ``"bits8"``, or -- with ``result``,
    and always for a record body (``FBR_BODY_RECORD``) -- a NumPy dtype of the argument record (see ``device_body``)."""
    import ctypes
    _MODULES[name] = (str(module_path), entry, args, bits_entry, result)
    if bits_entry is not None:
        twin = name + "_bits8"
        register_module(twin, module_path, bits_entry, "bits8")
        _MODULES.pop(twin, None)
        BITS_TWIN[name] = twin
    L = _abi.load()
    specs = _load_specs()      # before the body joins the engine's table: it is not listed as a plain BodySpec
    fid = ctypes.c_int(-1)
    _abi.check(L.fbr_register_body(name.encode(), str(module_path).encode(), entry.encode(), ctypes.byref(fid)))
    if name not in specs:
        info = _abi.BodyInfo()
        _abi.check(L.fbr_body_info(fid.value, ctypes.byref(info)))
        legacy = isinstance(args, str) and args in ("i64", "i64x2", "bits8")
        if result is not None or not legacy or (info.flags & _abi.FBR_BODY_RECORD):
            try:
                specs[name] = _Record(info, args, result)
            except (TypeError, ValueError):
                _MODULES.pop(name, None)
                raise
        elif args == "i64":
            specs[name] = _UnaryI64(info)
        elif args == "i64x2":
            specs[name] = _BinaryI64(info)
        elif args == "bits8":
            specs[name] = _Bits8(info)
        else:
            raise ValueError("unknown argument layout %r (have: i64, i64x2, bits8)" % (args,))
    return specs[name]


def device_initializer(body_name):
    """Bind a pool ``initializer`` to the broadcast block of device body ``body_name``.

    The reference runs ``initializer(*initargs)`` once in every worker process (fiber/pool.py:858-859),
    the idiom for giving all tasks the same large arguments without pickling them per task.  A host
    callable cannot run inside a GPU worker; what the idiom *means* maps exactly onto the engine's
    broadcast blocks: ``Pool(initializer=f, initargs=(...))`` with ``f`` decorated here uploads
    ``spec(body_name).shared_block(*initargs)`` once to every worker (``fbr_shared_put``), and tasks of that
    body submitted without their own shared arguments read it."""
    def decorator(func):
        spec(body_name)
        func.__fbr_init_body__ = body_name
        return func
    return decorator


def bind(func, name, **meta):
    """Bind an existing callable to device body ``name`` (see ``device_body``)."""
    from .meta import post_process
    spec(name)  # validate early: unknown names fail at bind time
    md = post_process(dict(meta) if meta else {"gpu": 1})
    try:
        func.__fbr_body__ = name
        func.__fiber_meta__ = md
    except (AttributeError, TypeError):
        _BOUND[func] = name
    return func


def body_name_of(func):
    name = getattr(func, "__fbr_body__", None)
    if name is None:
        try:
            name = _BOUND.get(func)
        except TypeError:
            name = None
    if name is None:
        raise TypeError(
            "fiber_b200.Pool: %r is not bound to a device body. Mapped functions execute on the GPU; "
            "bind one with @fiber_b200.device_body(name) or fiber_b200.bind(func, name) "
            "(available: %s). There is no CPU fallback." % (func, ", ".join(sorted(body_names()))))
    return name


# ------------------------------------------------------------------------------------------------
class Encoded:
    """Fixed-layout form of one map's arguments."""
    __slots__ = ("n", "args", "arg_stride", "index_start", "index_step", "shared", "task_index_base", "keepalive", "n_items")

    def __init__(self, n, args=None, arg_stride=0, index_start=0, index_step=1, shared=None, task_index_base=0, n_items=0):
        self.n, self.args, self.arg_stride = n, args, arg_stride
        self.index_start, self.index_step = index_start, index_step
        self.shared, self.task_index_base = shared, task_index_base
        self.n_items = n_items     # bit-packed twins: argument items of the whole map (8 per task, the last may be short)


def _as_i64(values, what):
    try:
        a = np.asarray(values)
    except OverflowError as e:
        raise OverflowError("%s: Python int too large for the int64 task record" % what) from e
    if a.size == 0:
        return np.zeros(a.shape if a.ndim else (0,), dtype=np.int64)
    if a.dtype == object:
        raise OverflowError("%s: arguments do not fit the int64 task record (got %r...)" % (what, values[:1]))
    if a.dtype.kind not in "iub":
        raise TypeError("%s: expected integer arguments, got dtype %s" % (what, a.dtype))
    if a.dtype.kind == "u" and a.dtype.itemsize == 8 and a.size and int(a.max()) > 2 ** 63 - 1:
        raise OverflowError("%s: argument exceeds int64" % what)
    return np.ascontiguousarray(a, dtype=np.int64)


class BodySpec:
    """One compiled-in device body plus the encoders for its argument records."""

    def __init__(self, info):
        self.name = info.name.decode()
        self.func_id = info.func_id
        self.arg_bytes = info.arg_bytes
        self.result_bytes = info.result_bytes
        self.result_kind = info.result_kind
        self.flags = info.flags

    # ---- argument encoders ---------------------------------------------------------------------
    def encode_map(self, items):
        """``map(func, items)``: one positional argument per task (fiber/pool.py:819-821)."""
        if self._fast_map_ok(items):
            return self._encode(items, fast=True)
        return self._encode([(it,) for it in items], fast=False)

    def encode_starmap(self, items):
        """``starmap(func, items)``: items are argument tuples (fiber/pool.py:807-809)."""
        return self._encode(list(items), fast=False)

    def encode_apply(self, args, kwds):
        """``apply_async(func, args, kwds)``: one task (fiber/pool.py:804-806)."""
        return self._encode([(tuple(args), dict(kwds))], fast=False, apply=True)

    def _fast_map_ok(self, items):
        return False

    def _encode(self, items, fast, apply=False):
        raise NotImplementedError

    @staticmethod
    def _split(item, apply):
        """-> (args tuple, kwds dict) of one starmap/apply item; mirrors the arity rules at
        fiber/pool.py:803-812."""
        if apply:
            return item
        if not isinstance(item, (tuple, list)):
            raise TypeError("starmap items must be argument tuples, got %r" % (item,))
        return tuple(item), {}

    # ---- single-record fast path (doorbell lane): no NumPy on the round trip ---------------------
    def pack_apply(self, args, kwds):
        """One task's argument record as bytes (default: through the array encoder)."""
        enc = self.encode_apply(args, kwds)
        return np.ascontiguousarray(enc.args).tobytes()

    def unpack_result(self, raw):
        k = self.result_kind
        if k == _abi.FBR_RES_NONE:
            return None
        if k == _abi.FBR_RES_BOOL:
            return raw[0] != 0
        if k == _abi.FBR_RES_I64:
            return struct.unpack_from("<q", raw)[0]
        if k == _abi.FBR_RES_U32:
            return struct.unpack_from("<I", raw)[0]
        if k == _abi.FBR_RES_F64X2:
            return struct.unpack_from("<dd", raw)
        return list(raw)

    # ---- result decoding -----------------------------------------------------------------------
    def result_dtype(self):
        k = self.result_kind
        if k == _abi.FBR_RES_BOOL:
            return np.dtype(np.bool_), ()
        if k == _abi.FBR_RES_I64:
            return np.dtype(np.int64), ()
        if k == _abi.FBR_RES_U32:
            return np.dtype(np.uint32), ()
        if k == _abi.FBR_RES_F64X2:
            return np.dtype(np.float64), (2,)
        if k == _abi.FBR_RES_NONE:
            return np.dtype(np.uint8), ()
        return np.dtype(np.uint8), (self.result_bytes,)

    def to_python(self, row):
        """One result element as the Python object the reference would have returned."""
        k = self.result_kind
        if k == _abi.FBR_RES_NONE:
            return None
        if k == _abi.FBR_RES_F64X2:
            return (float(row[0]), float(row[1]))
        if k == _abi.FBR_RES_BYTES:
            return row.tolist()
        return row.item()

    def rows_to_list(self, arr):
        k = self.result_kind
        if k == _abi.FBR_RES_NONE:
            return [None] * len(arr)
        if k == _abi.FBR_RES_F64X2:
            return [tuple(r) for r in arr.tolist()]
        return arr.tolist()


class _UnaryI64(BodySpec):
    """f(x) with one int argument: square_i64, identity_i64, pi_inside_det, fault_identity_i64."""

    def pack_apply(self, args, kwds):
        if len(args) != 1 or kwds or type(args[0]) is not int:
            return super().pack_apply(args, kwds)       # full validation / error messages
        try:
            return struct.pack("<q", args[0])
        except struct.error:
            raise OverflowError("%s: Python int too large for the int64 task record" % self.name) from None

    def _fast_map_ok(self, items):
        return True

    def _encode(self, items, fast, apply=False):
        if fast:
            if isinstance(items, range):
                # a range() chunk stays a range in the reference too (76 B pickled, BASELINE.md):
                # here it needs no argument records at all, the task index is the argument.
                if len(items) and not (-2 ** 63 <= items[0] <= 2 ** 63 - 1 and -2 ** 63 <= items[-1] <= 2 ** 63 - 1):
                    raise OverflowError("range() bounds exceed the int64 task record")
                return Encoded(len(items), index_start=items.start, index_step=items.step)
            a = _as_i64(items if isinstance(items, np.ndarray) else list(items), self.name)
            if a.ndim != 1:
                raise TypeError("%s: expected a flat sequence of ints" % self.name)
            return Encoded(len(a), args=a, arg_stride=8)
        xs = []
        for it in items:
            args, kwds = self._split(it, apply)
            if len(args) != 1 or kwds:
                raise TypeError("%s() takes exactly one positional argument" % self.name)
            xs.append(args[0])
        a = _as_i64(xs, self.name)
        return Encoded(len(a), args=a, arg_stride=8)


class _Bits8(BodySpec):
    """``pi_inside_bits8``: task g = items 8g..8g+7 (range() indices or int64 arguments), result = one byte
    (bit k = item 8g+k).  Not bound to a callable: ``Pool`` routes maps of the bool body here
    (``BITS_TWIN``) and presents the bytes as a bit-backed ``ResultArray``."""

    def from_encoded(self, enc):
        """Re-express the bool body's encoded map (one int64 record or range() index per task) as byte-tasks."""
        n = enc.n
        if enc.arg_stride == 0:
            return Encoded((n + 7) // 8, index_start=enc.index_start, index_step=enc.index_step, n_items=n)
        return Encoded((n + 7) // 8, args=enc.args, arg_stride=64, n_items=n)

    def result_dtype(self):
        return np.dtype(np.uint8), ()

    def encode_range(self, items):
        """``range`` of n indices -> ceil(n/8) byte tasks (the body walks the same start/step)."""
        if not isinstance(items, range):
            raise TypeError("%s takes range() arguments only" % self.name)
        if len(items) and not (-2 ** 63 <= items[0] <= 2 ** 63 - 1 and -2 ** 63 <= items[-1] + 7 * items.step <= 2 ** 63 - 1
                               and -2 ** 63 <= items[-1] <= 2 ** 63 - 1):
            raise OverflowError("range() bounds exceed the int64 task record")
        return Encoded((len(items) + 7) // 8, index_start=items.start, index_step=items.step, n_items=len(items))


# bool bodies that have a bit-packed twin: 8 consecutive range() indices per result byte
BITS_TWIN = {"pi_inside_det": "pi_inside_bits8"}


class _BinaryI64(BodySpec):
    """f(x, y) / f(x, y=default) with int arguments: mul2_i64, square_scale_i64."""

    def __init__(self, info, y_default=None):
        super().__init__(info)
        self.y_default = y_default

    def pack_apply(self, args, kwds):
        if not kwds and len(args) == 2 and type(args[0]) is int and type(args[1]) is int:
            try:
                return struct.pack("<qq", args[0], args[1])
            except struct.error:
                raise OverflowError("%s: Python int too large for the int64 task record" % self.name) from None
        return super().pack_apply(args, kwds)

    def _encode(self, items, fast, apply=False):
        rows = []
        for it in items:
            args, kwds = self._split(it, apply)
            vals = dict(zip(("x", "y"), args))
            if len(args) > 2:
                raise TypeError("%s() takes at most 2 positional arguments" % self.name)
            for k, v in kwds.items():
                if k not in ("x", "y") or k in vals:
                    raise TypeError("%s() got an unexpected or duplicate keyword argument %r" % (self.name, k))
                vals[k] = v
            if "y" not in vals and self.y_default is not None:
                vals["y"] = self.y_default
            if "x" not in vals or "y" not in vals:
                raise TypeError("%s() missing required arguments" % self.name)
            rows.append((vals["x"], vals["y"]))
        a = _as_i64(rows, self.name).reshape(len(rows), 2)
        return Encoded(len(rows), args=a, arg_stride=16)


class _SleepF64(BodySpec):
    def _fast_map_ok(self, items):
        return True

    def _encode(self, items, fast, apply=False):
        if fast:
            a = np.ascontiguousarray(list(items), dtype=np.float64)
        else:
            vals = []
            for it in items:
                args, kwds = self._split(it, apply)
                if len(args) != 1 or kwds:
                    raise TypeError("sleep body takes exactly one positional argument")
                vals.append(args[0])
            a = np.ascontiguousarray(vals, dtype=np.float64)
        return Encoded(len(a), args=a, arg_stride=8)


class _Parzen(BodySpec):
    """parzen_estimation(x_samples, point_x, h) (examples/parzen_estimation.py:6-15).

    ``x_samples`` and ``point_x`` are identical for every task of a map: they become the broadcast
    block (uploaded once per distinct array instead of pickled into every task message,
    SURVEY.md 3.2); the per-task record is ``h``."""
    HEADER = np.dtype([("n_samples", "<u4"), ("dims", "<u4"), ("power", "<u4"), ("elem_bytes", "<u4"),
                       ("point_x", "<f8", (8,))])

    def __init__(self, info, elem):
        super().__init__(info)
        self.elem = np.dtype(elem)

    def shared_block(self, x_samples, point_x):
        """The broadcast block for (x_samples, point_x).  The reference pickles both into every one of its task
        messages; the example submits 102 ``apply_async`` calls with the same arrays, so the last block is kept
        and reused when the arguments compare equal (an exact memcmp of 160 KB, ~10 us, instead of casting and
        serialising them again)."""
        xs = np.asarray(x_samples)
        px = np.asarray(point_x)
        last = getattr(self, "_last_block", None)
        if last is not None and last[0].shape == xs.shape and last[1].shape == px.shape and last[0].dtype == xs.dtype \
                and np.array_equal(last[0], xs) and np.array_equal(last[1], px):
            return last[2]
        blob = self._build_block(xs, px)
        self._last_block = (xs.copy(), px.copy(), blob)
        return blob

    def _build_block(self, xs, px):
        if xs.ndim != 2 or px.ndim != 2 or px.shape[0] != xs.shape[1]:
            raise TypeError("parzen_estimation: x_samples must be (n, d) and point_x (d, p)")
        if px.shape[0] > 8:
            raise TypeError("parzen_estimation: at most 8 dimensions are supported by the device body")
        if px.shape[1] != 1:
            # the reference evaluates `np.abs(row) > 1/2` on a length-p row, which raises for p != 1
            raise ValueError("The truth value of an array with more than one element is ambiguous")
        hdr = np.zeros((), dtype=self.HEADER)
        hdr["n_samples"], hdr["dims"], hdr["power"], hdr["elem_bytes"] = xs.shape[0], xs.shape[1], px.shape[1], self.elem.itemsize
        hdr["point_x"][: px.shape[0]] = px[:, 0].astype(np.float64)
        body = np.ascontiguousarray(xs, dtype=self.elem)  # the one cast to fp32 for parzen_f32
        return hdr.tobytes() + body.tobytes()

    def _fast_map_ok(self, items):
        # map(func, widths): the samples come from the pool's broadcast block (Pool(initializer=, initargs=))
        return True

    def _encode(self, items, fast, apply=False):
        if fast:
            return Encoded(len(items), args=np.ascontiguousarray(list(items), dtype=np.float64), arg_stride=8)
        hs, first = [], None
        for it in items:
            args, kwds = self._split(it, apply)
            if len(args) == 1 and not kwds:        # (h,): samples from the broadcast block
                if first is not None:
                    raise TypeError("parzen_estimation: mixed (h,) and (x_samples, point_x, h) items in one map")
                hs.append(float(args[0]))
                continue
            if hs and first is None:
                raise TypeError("parzen_estimation: mixed (h,) and (x_samples, point_x, h) items in one map")
            vals = dict(zip(("x_samples", "point_x", "h"), args))
            vals.update(kwds)
            if set(vals) != {"x_samples", "point_x", "h"}:
                raise TypeError("parzen_estimation(x_samples, point_x, h): bad arguments")
            if first is None:
                first = (vals["x_samples"], vals["point_x"])
            elif not (vals["x_samples"] is first[0] and vals["point_x"] is first[1]):
                if not (np.array_equal(vals["x_samples"], first[0]) and np.array_equal(vals["point_x"], first[1])):
                    raise ValueError("parzen_estimation: all tasks of one map must share x_samples and point_x")
            hs.append(float(vals["h"]))
        a = np.ascontiguousarray(hs, dtype=np.float64)
        enc = Encoded(len(a), args=a, arg_stride=8)
        enc.shared = self.shared_block(*first) if first is not None else None
        return enc


def _record_dtype(layout, what):
    """NumPy dtype of a record layout: anything ``np.dtype()`` takes, plus the names of the integer layouts."""
    if isinstance(layout, str) and layout in ("i64", "i64x2"):
        layout = "<i8" if layout == "i64" else "2<i8"
    try:
        return np.dtype(layout)
    except TypeError as e:
        raise ValueError("%s: %r is not a NumPy dtype (%s)" % (what, layout, e)) from None


def _leaves(dt, off=0):
    """(byte offset, scalar dtype) of every scalar of record dtype ``dt``, in memory order."""
    if dt.names:
        for n in dt.names:
            f, o = dt.fields[n][:2]
            yield from _leaves(f, off + o)
    elif dt.subdtype is not None:
        base, shape = dt.subdtype
        for i in range(int(np.prod(shape))):
            yield from _leaves(base, off + i * base.itemsize)
    else:
        yield off, dt


_MISSING = object()


class _Record(BodySpec):
    """A body whose argument and result records are NumPy dtypes (out-of-tree record bodies,
    ``FBR_EXPORT_RECORD_BODY``): ``f(x)`` of a scalar dtype, ``f(x, y, z)`` of a structured dtype's fields (or of the
    elements of a sub-array dtype such as ``"3f4"``).  The call rules follow the reference's task tuple
    (fiber/pool.py:803-821): ``map`` passes each item as the one argument -- a number, the value of a one-field record,
    or the tuple of field values --
    ``starmap`` its items as positional arguments, ``apply`` positional arguments then keywords by field name."""

    def __init__(self, info, args, result):
        super().__init__(info)
        if result is None:
            raise ValueError("%s: a record body needs result=<dtype> of its %d-byte result record" % (self.name, info.result_bytes))
        self.arg_dtype = _record_dtype(args, "%s args" % self.name)
        self.res_dtype = _record_dtype(result, "%s result" % self.name)
        for what, dt, nb in (("argument", self.arg_dtype, self.arg_bytes), ("result", self.res_dtype, self.result_bytes)):
            if dt.itemsize != nb:
                raise ValueError("%s: %s dtype %s has %d bytes, the module's %s record has %d"
                                 % (self.name, what, dt, dt.itemsize, what, nb))
        dt = self.arg_dtype
        self.fields = dt.names                      # keyword names (structured dtypes only)
        self.arity = len(dt.names) if dt.names else (int(np.prod(dt.subdtype[1])) if dt.subdtype is not None else 1)
        self._leaves = list(_leaves(dt))

    # ---- arguments ------------------------------------------------------------------------------
    def _row(self, args, kwds):
        """Positional arguments, then keywords by field name -> the record's field values in order."""
        n = self.arity
        if len(args) > n:
            raise TypeError("%s() takes %d positional argument%s but %d were given" % (self.name, n, "s" * (n != 1), len(args)))
        vals = list(args) + [_MISSING] * (n - len(args))
        for k, v in kwds.items():
            if not self.fields or k not in self.fields:
                raise TypeError("%s() got an unexpected keyword argument %r" % (self.name, k))
            i = self.fields.index(k)
            if vals[i] is not _MISSING:
                raise TypeError("%s() got multiple values for argument %r" % (self.name, k))
            vals[i] = v
        if any(v is _MISSING for v in vals):
            missing = [self.fields[i] if self.fields else str(i) for i, v in enumerate(vals) if v is _MISSING]
            raise TypeError("%s() missing required argument(s): %s" % (self.name, ", ".join(missing)))
        return vals

    def _records(self, rows):
        dt = self.arg_dtype
        if dt.names:
            return np.array([tuple(r) for r in rows], dtype=dt)
        if dt.subdtype is not None:
            base, shape = dt.subdtype
            return np.array(rows, dtype=base).reshape((len(rows),) + shape)
        return np.array([r[0] for r in rows], dtype=dt)

    def _array_records(self, a):
        """A NumPy array as argument records: itself when its rows already are the record layout (no copy)."""
        dt = self.arg_dtype
        if a.ndim == 1 and a.dtype == dt:
            return np.ascontiguousarray(a)
        if a.ndim == 2 and a.shape[1] == len(self._leaves) and a.shape[1] * a.itemsize == dt.itemsize and \
                all(b == a.dtype and off == i * a.itemsize for i, (off, b) in enumerate(self._leaves)):
            return np.ascontiguousarray(a)          # (n, k) rows of the record's k scalars
        if a.ndim == 1 and not dt.names and dt.subdtype is None and a.dtype.kind in "biuf":
            return np.ascontiguousarray(a, dtype=dt)
        if dt.names and a.dtype.names == dt.names and a.ndim == 1:
            return a.astype(dt)
        raise TypeError("%s: an array of dtype %s and shape %s does not hold %s records" % (self.name, a.dtype, a.shape, dt))

    def _fast_map_ok(self, items):
        return True

    def _encode(self, items, fast, apply=False):
        if fast:
            if isinstance(items, np.ndarray):
                a = self._array_records(items)
            elif self.arity == 1 and not self.fields and self.arg_dtype.subdtype is None:
                a = np.array(items if isinstance(items, list) else list(items), dtype=self.arg_dtype)
            elif self.arity == 1:
                a = self._records([(it,) for it in items])      # one field: the item is its value, f(item)
            else:
                rows = []
                for it in items:
                    if not isinstance(it, (tuple, list, np.ndarray, np.void)):
                        raise TypeError("%s: map() items must be tuples of the %d record fields, got %r" % (self.name, self.arity, it))
                    rows.append(self._row(tuple(it), {}))
                a = self._records(rows)
        else:
            a = self._records([self._row(*self._split(it, apply)) for it in items])
        return Encoded(len(a), args=a, arg_stride=self.arg_dtype.itemsize)

    # ---- results --------------------------------------------------------------------------------
    def result_dtype(self):
        dt = self.res_dtype
        if dt.subdtype is not None:
            return dt.subdtype[0], dt.subdtype[1]
        return dt, ()

    def to_python(self, row):
        if self.res_dtype.names or self.res_dtype.subdtype is not None:
            return self.rows_to_list(np.asarray(row)[None])[0]
        return row.item()

    def rows_to_list(self, arr):
        if self.res_dtype.subdtype is not None:
            return [tuple(r) for r in arr.tolist()]
        return arr.tolist()                          # structured rows: tuples of Python scalars

    def unpack_result(self, raw):
        return self.to_python(np.frombuffer(bytes(raw[:self.result_bytes]), dtype=self.res_dtype)[0])

    def py_sum(self, values):
        """``sum(results)`` exactly as the builtin computes it over the reference's list (the device does not fold
        record results): floats added left to right, and TypeError for tuples."""
        return sum(values.tolist())


class _Payload4K(BodySpec):
    """Synthetic 4 KB payload bodies.  ``map(func, records)`` with a ``(n, 1024)`` uint32 array, or
    ``starmap(func, [(t, rec), ...])`` with consecutive ``t`` (the task's global index)."""

    def _fast_map_ok(self, items):
        return isinstance(items, np.ndarray)

    def result_dtype(self):
        if self.result_kind == _abi.FBR_RES_BYTES:
            return np.dtype(np.uint32), (1024,)
        return super().result_dtype()

    def _encode(self, items, fast, apply=False):
        if fast:
            recs, base = items, 0
        else:
            ts, rows = [], []
            for it in items:
                args, kwds = self._split(it, apply)
                if len(args) != 2 or kwds:
                    raise TypeError("%s(t, rec): bad arguments" % self.name)
                ts.append(int(args[0]))
                rows.append(args[1])
            base = ts[0] if ts else 0
            if ts != list(range(base, base + len(ts))):
                raise ValueError("%s: task indices must be consecutive" % self.name)
            recs = np.asarray(rows, dtype=np.uint32)
        recs = np.ascontiguousarray(recs, dtype=np.uint32)
        if recs.ndim != 2 or recs.shape[1] != 1024:
            raise TypeError("%s: records must be (n, 1024) uint32" % self.name)
        return Encoded(recs.shape[0], args=recs, arg_stride=4096, task_index_base=base)


_SPECS = None


def _load_specs():
    global _SPECS
    if _SPECS is not None:
        return _SPECS
    import ctypes
    L = _abi.load()
    n = ctypes.c_int(0)
    _abi.check(L.fbr_body_count(ctypes.byref(n)))
    specs = {}
    for fid in range(n.value):
        info = _abi.BodyInfo()
        _abi.check(L.fbr_body_info(fid, ctypes.byref(info)))
        name = info.name.decode()
        if name in ("square_i64", "identity_i64", "pi_inside_det", "fault_identity_i64", "trap_identity_i64"):
            s = _UnaryI64(info)
        elif name == "mul2_i64":
            s = _BinaryI64(info)
        elif name == "square_scale_i64":
            s = _BinaryI64(info, y_default=1)
        elif name == "sleep_f64":
            s = _SleepF64(info)
        elif name == "parzen_f32":
            s = _Parzen(info, np.float32)
        elif name == "parzen_f64":
            s = _Parzen(info, np.float64)
        elif name in ("payload_map_4k", "payload_checksum_4k"):
            s = _Payload4K(info)
        elif name == "pi_inside_bits8":
            s = _Bits8(info)
        else:
            s = BodySpec(info)
        specs[name] = s
    _SPECS = specs
    return specs


def body_names():
    return list(_load_specs())


def spec(name):
    specs = _load_specs()
    if name not in specs:
        raise KeyError("no device body named %r is compiled into libfiber_b200 (have: %s)" % (name, ", ".join(sorted(specs))))
    return specs[name]


def fingerprint(buf):
    return hashlib.blake2b(buf, digest_size=16).digest()
