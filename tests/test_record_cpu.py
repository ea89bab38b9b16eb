"""CPU: record bodies (float / struct argument and result records, FBR_EXPORT_RECORD_BODY) without a device --
registration and its refusals, the host encoders and decoders, and the plans the engine makes for record maps."""
import ctypes

import numpy as np
import pytest

from fiber_b200 import _abi, registry
from fiber_b200.pool import ResultArray
from tests import record_bodies as RB
from tests.test_plan_cpu import FAKE_DEVICE_PTR, _desc, plan


def _info(name):
    info = _abi.BodyInfo()
    _abi.check(_abi.load().fbr_body_info(registry.spec(name).func_id, ctypes.byref(info)))
    return info


# ---- registration ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(RB.LAYOUTS))
def test_every_test_body_is_registered_with_its_layout(name):
    _, args, result = RB.LAYOUTS[name]
    info = _info(name)
    assert info.name.decode() == name and info.result_kind == _abi.FBR_RES_BYTES
    assert (info.arg_bytes, info.result_bytes) == (np.dtype(args).itemsize, np.dtype(result).itemsize)
    record = not name.endswith("_thread")
    assert bool(info.flags & _abi.FBR_BODY_RECORD) == record
    assert not info.flags & (_abi.FBR_BODY_SUMMABLE | _abi.FBR_BODY_INDEX_ARG | _abi.FBR_BODY_NEEDS_SHARED)
    assert isinstance(registry.spec(name), registry._Record)
    assert registry.module_of(name)[2:] == (args, None, result)     # what a worker process registers again


@pytest.mark.parametrize("name", sorted(RB.BAD_MODULES))
def test_engine_refuses_bad_record_layouts(name):
    """Sizes that are not whole words or exceed 256 bytes, and summable / range() record bodies."""
    L = _abi.load()
    fid = ctypes.c_int(-1)
    rc = L.fbr_register_body(name.encode(), RB.MODULE.encode(), RB.BAD_MODULES[name].encode(), ctypes.byref(fid))
    assert rc == _abi.FBR_EINVAL
    assert b"record body" in L.fbr_last_error()
    assert name not in registry.body_names()


def test_dtype_must_match_the_module():
    info = _info("norm2_f3")
    with pytest.raises(ValueError, match="12"):
        registry._Record(info, "f8", "f4")
    with pytest.raises(ValueError, match="result"):
        registry._Record(info, "3f4", "f8")
    with pytest.raises(ValueError):
        registry._Record(info, "3f4", None)             # a record body needs its result layout
    with pytest.raises(ValueError):
        registry._Record(info, "not a dtype", "f4")
    assert registry._Record(info, "3f4", "<i4").arity == 3


# ---- encoders ----------------------------------------------------------------------------------------------------
def test_map_uses_arrays_of_the_record_layout_without_a_copy():
    s = registry.spec("norm2_f3")
    rows = np.arange(30, dtype=np.float32).reshape(10, 3)
    for a in (rows, rows[1:], rows.view(RB.F3).reshape(-1), np.zeros(4, RB.F3)):
        enc = s.encode_map(a)
        assert enc.args.ctypes.data == a.ctypes.data and enc.arg_stride == 12 and enc.n == len(a)
    # one 12 B record into the array: 4-byte aligned, not 16-byte aligned
    assert s.encode_map(rows[1:]).args.ctypes.data % 16 != 0
    w = np.zeros((5, 8))
    assert registry.spec("dot_w64").encode_map(w).args is w
    assert registry.spec("mix_256").encode_map(np.zeros((3, 64), np.uint32)).arg_stride == 256
    with pytest.raises(TypeError):
        s.encode_map(np.zeros((4, 2), np.float32))      # rows of 8 bytes are not float3 records
    with pytest.raises(TypeError):
        s.encode_map(np.zeros((4, 3), np.float64))      # the right count of the wrong scalars


def test_map_of_sequences_encodes_one_record_per_item():
    p = registry.spec("poly_f64")
    assert p.encode_map([1, 2.5, -3]).args.tolist() == [1.0, 2.5, -3.0]
    assert p.encode_map(range(4)).args.tolist() == [0.0, 1.0, 2.0, 3.0]
    assert registry.spec("halve_nonneg").encode_map(np.arange(3.0)).args.dtype == np.float32   # a cast, by value
    s = registry.spec("norm2_f3")
    enc = s.encode_map([(1, 2, 3), [4, 5, 6]])
    assert enc.args.dtype == RB.F3 and enc.args.tolist() == [(1.0, 2.0, 3.0), (4.0, 5.0, 6.0)]
    with pytest.raises(TypeError):
        s.encode_map([1.0, 2.0])                        # a structured record takes the tuple of its fields
    with pytest.raises(TypeError):
        s.encode_map([(1, 2)])
    # a one-field record takes the field's value, as the reference calls f(item)
    v = [float(k) for k in range(8)]
    w = registry.spec("dot_w64").encode_map([v, np.arange(8.0)]).args
    assert w.dtype == RB.W64 and w["v"].tolist() == [v, v]
    with pytest.raises((TypeError, ValueError)):
        registry.spec("dot_w64").encode_map([v[:7]])
    t = registry.spec("triple_or_fault").encode_map([(1.5, 0), (2.5, 1)]).args
    assert t.dtype == RB.TAGGED and t["tag"].tolist() == [0, 1]


def test_starmap_and_apply_take_the_fields_as_arguments():
    s = registry.spec("norm2_f3")
    assert s.encode_starmap([(1, 2, 3), (4, 5, 6)]).args.tolist() == [(1.0, 2.0, 3.0), (4.0, 5.0, 6.0)]
    assert s.encode_apply((1,), {"z": 3, "y": 2}).args.tolist() == [(1.0, 2.0, 3.0)]
    assert s.encode_apply((), {"x": 1, "y": 2, "z": 3}).args.tolist() == [(1.0, 2.0, 3.0)]
    assert registry.spec("affine_f3").encode_starmap([(1, 2, 3)]).args.tolist() == [[1.0, 2.0, 3.0]]
    assert registry.spec("poly_f64").encode_apply((2.0,), {}).args.tolist() == [2.0]
    with pytest.raises(TypeError, match="takes 3 positional"):
        s.encode_apply((1, 2, 3, 4), {})
    with pytest.raises(TypeError, match="multiple values"):
        s.encode_apply((1,), {"x": 2, "y": 1, "z": 1})
    with pytest.raises(TypeError, match="missing"):
        s.encode_apply((1, 2), {})
    with pytest.raises(TypeError, match="unexpected keyword"):
        s.encode_apply((1, 2), {"w": 3})
    with pytest.raises(TypeError, match="unexpected keyword"):
        registry.spec("poly_f64").encode_apply((), {"x": 1.0})     # a scalar record has no field names
    with pytest.raises(TypeError):
        s.encode_starmap([1.0])                         # starmap items are argument tuples


# ---- decoders ----------------------------------------------------------------------------------------------------
def test_results_decode_to_python_scalars_and_tuples():
    f = registry.spec("norm2_f3")
    arr = np.array([1.5, 2.25], np.float32)
    r = ResultArray(f, arr)
    assert r.tolist() == [1.5, 2.25] and type(r[0]) is float and r.array is arr
    st = registry.spec("stats_w64")
    a = np.zeros(2, RB.STATS)
    a[1] = (2.5, -3, 7)
    r = ResultArray(st, a)
    assert r[1] == (2.5, -3, 7) and all(type(v) in (float, int) for v in r[1])
    assert r.tolist() == [(0.0, 0, 0), (2.5, -3, 7)] and r.array.dtype == RB.STATS
    af = registry.spec("affine_f3")
    assert af.result_dtype() == (np.dtype(np.float32), (3,))
    r = ResultArray(af, np.arange(6, dtype=np.float32).reshape(2, 3))
    assert r[1] == (3.0, 4.0, 5.0) and r.tolist() == [(0.0, 1.0, 2.0), (3.0, 4.0, 5.0)]
    assert st.unpack_result(a[1].tobytes()) == (2.5, -3, 7)


def test_sum_is_the_builtin_sum_of_the_list():
    vals = np.array([0.1, 0.2, 0.3, 1e16, -1e16, 0.7], np.float64)
    r = ResultArray(registry.spec("poly_f64"), vals)
    assert r.sum() == sum(vals.tolist()) and r.sum() != float(vals.sum())     # left to right, like the builtin
    with pytest.raises(TypeError):
        ResultArray(registry.spec("stats_w64"), np.zeros(3, RB.STATS)).sum()
    with pytest.raises(TypeError):
        sum(ResultArray(registry.spec("stats_w64"), np.zeros(3, RB.STATS)).tolist())


# ---- plans -------------------------------------------------------------------------------------------------------
def test_gcd_alignment_keeps_r12_units_16_byte_aligned():
    """R = 12: units are multiples of 4 tasks (16 / gcd(12, 16)), so full slots stay 16 B aligned and the map is
    placed directly.  A chunksize of 7 gives units of lcm(7, 4) * k = 4088 tasks, still aligned: still direct."""
    d = _desc("affine_f3", 10 ** 6, arg_stride=12, args=FAKE_DEVICE_PTR + 12)
    p = plan(d)
    assert p["paths"] == {"direct", "host_args"} and p["unit"] == 4096 and (p["unit"] * 12) % 16 == 0
    p = plan(_desc("affine_f3", 10 ** 6, chunksize=7, arg_stride=12, args=FAKE_DEVICE_PTR))
    assert p["paths"] == {"direct", "host_args"} and p["unit"] == 4088 and p["unit"] % 7 == 0
    p = plan(_desc("norm2_f3", 10 ** 6, chunksize=7, arg_stride=12, args=FAKE_DEVICE_PTR))   # R = 4: the same unit
    assert p["unit"] == 4088 and "direct" in p["paths"]


@pytest.mark.parametrize("flag", ["FBR_SHUFFLE", "FBR_VIA_RING", "FBR_RESILIENT"])
def test_record_maps_through_the_ring(flag):
    for chunksize in (32, 7):
        p = plan(_desc("affine_f3", 10 ** 6, getattr(_abi, flag), chunksize=chunksize, arg_stride=12, args=FAKE_DEVICE_PTR))
        assert "direct" not in p["paths"]


@pytest.mark.parametrize("ring", [0, 64 << 20, 4 << 20])
def test_256_byte_records_fit_the_ring(ring):
    ring_bytes = ring or (256 << 20)
    for flags in (0, _abi.FBR_VIA_RING):
        p = plan(_desc("mix_256", 10 ** 6, flags, arg_stride=256, args=FAKE_DEVICE_PTR), ring=ring)
        assert p["unit"] * 256 <= ring_bytes // 2
        assert p["wave_tasks"] * 256 <= ring_bytes and p["waves"] * p["wave_tasks"] >= 10 ** 6
    # the R = 16 and R = 8 bodies of the 64 B argument keep the existing 16 / R rule
    assert plan(_desc("stats_w64", 10 ** 6, arg_stride=64, args=FAKE_DEVICE_PTR))["unit"] == 4096
    assert plan(_desc("dot_w64", 10 ** 6, chunksize=7, arg_stride=64, args=FAKE_DEVICE_PTR))["unit"] == 4088
