"""GPU: record bodies (float / struct argument and result records, dispatch_record_kernel) against their NumPy
restatements, bit for bit, on every path a map can take: direct placement, the result ring with gather_ordered
(chunksize 7, FBR_SHUFFLE, FBR_VIA_RING), unaligned host records, device-resident arguments and output, imap,
device-resident results, several workers, resilient re-dispatch and worker processes."""
import ctypes

import numpy as np
import pytest

import fiber_b200
from fiber_b200 import _abi, registry
from tests import record_bodies as RB

pytestmark = pytest.mark.gpu

N = 1_000_003            # >= 1e6 tasks, and not a multiple of any unit or tile: every tail path runs


@pytest.fixture(scope="module")
def pool():
    p = fiber_b200.Pool(1)
    yield p
    p.terminate()
    p.join()


def _rng(seed=0):
    return np.random.default_rng(seed)


def _f3(n, seed=0):
    return _rng(seed).standard_normal((n, 3)).astype(np.float32) * np.float32(100)


def _w64(n, seed=0):
    return _rng(seed).standard_normal((n, 8)) * 1e3


def _args(name, n, seed=0):
    """Argument records of body `name` and the restated results."""
    if name in ("norm2_f3", "affine_f3"):
        a = _f3(n, seed)
    elif name.startswith("poly_f64"):
        a = _rng(seed).standard_normal(n) * 1e6
    elif name.startswith(("stats_w64", "dot_w64")):
        a = _w64(n, seed)
    elif name == "mix_256":
        a = _rng(seed).integers(0, 2 ** 32, (n, 64), dtype=np.uint32)
    elif name == "halve_nonneg":
        a = np.abs(_rng(seed).standard_normal(n).astype(np.float32))
    else:
        raise KeyError(name)
    return a, _expected(name, a)


def _expected(name, a):
    fn = getattr(RB, name.replace("_thread", "").replace("_staged", "") + "_np")
    return fn(a.view(RB.W64).reshape(-1) if name.startswith(("stats_w64", "dot_w64")) else a)


def _same(got, want):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape and got.dtype == want.dtype
    assert got.tobytes() == want.tobytes()          # bit for bit (NaN-safe, -0.0-safe)


def _f(name):
    return getattr(RB, name)


BODIES = ["norm2_f3", "affine_f3", "poly_f64", "poly_f64_thread", "poly_f64_staged", "stats_w64", "dot_w64", "dot_w64_thread", "mix_256",
          "halve_nonneg"]


@pytest.mark.parametrize("name", BODIES)
def test_body_matches_its_restatement_direct(pool, name):
    a, want = _args(name, N)
    r = pool.map_async(_f(name), a)
    res = r.get()
    _same(res.array, want)
    assert len(res) == N


def test_ten_million_tasks_in_several_waves():
    pool = fiber_b200.Pool(1, ring_bytes=64 << 20)
    try:
        n = 10_000_019
        a = _f3(n, 5)
        r = pool.map_async(RB.affine_f3, a)
        _same(r.get().array, RB.affine_f3_np(a))
        assert r.n_waves > 1
    finally:
        pool.terminate()
        pool.join()


@pytest.mark.parametrize("name", ["affine_f3", "norm2_f3", "stats_w64", "mix_256"])
def test_chunksize_7(pool, name):
    a, want = _args(name, N, 1)
    _same(pool.map(_f(name), a, chunksize=7).array, want)


def _submit_abi(pool, name, args, flags, n, arg_stride, out=None, chunksize=0):
    pool.start_workers()
    eng = pool._engine
    d = _abi.MapDesc()
    d.func_id, d.flags, d.n_tasks, d.chunksize, d.arg_stride = registry.spec(name).func_id, flags, n, chunksize, arg_stride
    d.args = args
    d.index_start, d.index_step, d.shuffle_seed = 0, 1, 11
    if out is not None:
        d.out = out
    seq = ctypes.c_uint64()
    rc = eng.lib.fbr_map_submit(eng.handle, ctypes.byref(d), ctypes.byref(seq))
    return rc, seq.value


def _wait_abi(pool, seq, nbytes):
    eng = pool._engine
    res = _abi.Result()
    _abi.check(eng.lib.fbr_result_wait(eng.handle, seq, -1, ctypes.byref(res)))
    out = np.frombuffer((ctypes.c_char * nbytes).from_address(res.data), dtype=np.uint8).copy()
    _abi.check(eng.lib.fbr_result_release(eng.handle, seq))
    return out


@pytest.mark.parametrize("flag", ["FBR_SHUFFLE", "FBR_VIA_RING"])
@pytest.mark.parametrize("name", ["affine_f3", "norm2_f3", "stats_w64", "mix_256", "poly_f64"])
def test_ring_and_gather_through_the_c_abi(pool, flag, name):
    a, want = _args(name, N, 2)
    for chunksize in (0, 7):
        rc, seq = _submit_abi(pool, name, a.ctypes.data, getattr(_abi, flag), N, a.nbytes // N, chunksize=chunksize)
        _abi.check(rc)
        got = _wait_abi(pool, seq, want.nbytes)
        assert got.tobytes() == np.ascontiguousarray(want).tobytes()


def test_records_at_a_4_byte_aligned_host_address(pool):
    rows = _f3(N + 1, 3)
    a = rows[1:]                                          # one 12 B record in: not 16-byte aligned
    assert a.ctypes.data % 16 != 0 and a.ctypes.data % 4 == 0
    _same(pool.map(RB.affine_f3, a).array, RB.affine_f3_np(a))
    _same(pool.map(RB.norm2_f3, a, chunksize=7).array, RB.norm2_f3_np(a))


@pytest.mark.parametrize("offset", [0, 12])
@pytest.mark.parametrize("name", ["affine_f3", "stats_w64"])
def test_device_resident_args_and_out(pool, name, offset):
    a, want = _args(name, N, 4)
    want = np.ascontiguousarray(want)
    pool.start_workers()
    eng, lib = pool._engine, pool._engine.lib
    din, dout = ctypes.c_void_p(), ctypes.c_void_p()
    _abi.check(lib.fbr_device_alloc(eng.handle, 0, a.nbytes + 16, ctypes.byref(din)))
    _abi.check(lib.fbr_device_alloc(eng.handle, 0, want.nbytes + 16, ctypes.byref(dout)))
    try:
        src, dst = din.value + offset, dout.value + offset
        _abi.check(lib.fbr_memcpy_h2d(eng.handle, 0, ctypes.c_void_p(src), a.ctypes.data, a.nbytes))
        rc, seq = _submit_abi(pool, name, src, _abi.FBR_ARGS_DEVICE | _abi.FBR_OUT_DEVICE, N, a.nbytes // N, out=dst)
        _abi.check(rc)
        res = _abi.Result()
        _abi.check(lib.fbr_result_wait(eng.handle, seq, -1, ctypes.byref(res)))
        _abi.check(lib.fbr_result_release(eng.handle, seq))
        got = np.empty_like(want)
        _abi.check(lib.fbr_memcpy_d2h(eng.handle, 0, got.ctypes.data, ctypes.c_void_p(dst), got.nbytes))
        _same(got, want)
    finally:
        lib.fbr_device_free(eng.handle, 0, din)
        lib.fbr_device_free(eng.handle, 0, dout)


def test_argument_stride_rules(pool):
    """Record bodies take any whole-word stride >= the record; other bodies keep their 8 / 16-byte rules."""
    a = np.zeros((16, 4), np.float32)                      # 16 B rows: a float3 record and 4 bytes of padding
    a[:, :3] = _f3(16, 6)
    rc, seq = _submit_abi(pool, "affine_f3", a.ctypes.data, 0, 16, 16)
    _abi.check(rc)
    got = _wait_abi(pool, seq, 16 * 12).view(np.float32).reshape(16, 3)
    _same(got, RB.affine_f3_np(np.ascontiguousarray(a[:, :3])))
    assert _submit_abi(pool, "affine_f3", a.ctypes.data, 0, 4, 14)[0] == _abi.FBR_EINVAL      # not whole words
    assert _submit_abi(pool, "affine_f3", a.ctypes.data, 0, 4, 8)[0] == _abi.FBR_EINVAL       # shorter than the record
    assert _submit_abi(pool, "affine_f3", a.ctypes.data + 2, 0, 4, 12)[0] == _abi.FBR_EINVAL  # not 4-byte aligned
    b = np.zeros(64)
    assert _submit_abi(pool, "poly_f64_thread", b.ctypes.data, 0, 4, 12)[0] == _abi.FBR_EINVAL   # thread body: 8 B rule
    w = np.zeros((5, 9))
    assert _submit_abi(pool, "dot_w64_thread", w.ctypes.data + 8, 0, 4, 72)[0] == _abi.FBR_EINVAL  # 16 B rule


def test_per_thread_layout_takes_the_staged_kernel_for_4_byte_aligned_records(pool):
    """FBR_EXPORT_RECORD_BODY runs 8 B -> 8 B records one thread per record, reading them in place; records that are
    only 4-byte aligned -- a 12 B stride, device arguments at an odd word -- go through the staged kernel instead."""
    x = _args("poly_f64", N, 14)[0]
    want = RB.poly_f64_np(x)
    padded = np.zeros((N, 3), np.float32)                  # each f64 in the first 8 bytes of a 12 B record
    padded[:, :2] = x.view(np.float32).reshape(N, 2)
    rc, seq = _submit_abi(pool, "poly_f64", padded.ctypes.data, 0, N, 12)
    _abi.check(rc)
    _same(_wait_abi(pool, seq, N * 8).view(np.float64), want)
    eng, lib = pool._engine, pool._engine.lib
    din, dout = ctypes.c_void_p(), ctypes.c_void_p()
    _abi.check(lib.fbr_device_alloc(eng.handle, 0, x.nbytes + 16, ctypes.byref(din)))
    _abi.check(lib.fbr_device_alloc(eng.handle, 0, x.nbytes + 16, ctypes.byref(dout)))
    try:
        for off in (4, 8):
            _abi.check(lib.fbr_memcpy_h2d(eng.handle, 0, ctypes.c_void_p(din.value + off), x.ctypes.data, x.nbytes))
            rc, seq = _submit_abi(pool, "poly_f64", din.value + off, _abi.FBR_ARGS_DEVICE | _abi.FBR_OUT_DEVICE, N, 8,
                                  out=dout.value + off)
            _abi.check(rc)
            res = _abi.Result()
            _abi.check(lib.fbr_result_wait(eng.handle, seq, -1, ctypes.byref(res)))
            _abi.check(lib.fbr_result_release(eng.handle, seq))
            got = np.empty_like(want)
            _abi.check(lib.fbr_memcpy_d2h(eng.handle, 0, got.ctypes.data, ctypes.c_void_p(dout.value + off), got.nbytes))
            _same(got, want)
    finally:
        lib.fbr_device_free(eng.handle, 0, din)
        lib.fbr_device_free(eng.handle, 0, dout)


def test_imap_streams_records(pool):
    a, want = _args("stats_w64", 300_001, 7)
    got = list(pool.imap(RB.stats_w64, a, chunksize=64))
    assert got == want.tolist()
    a, want = _args("affine_f3", 200_003, 7)
    assert list(pool.imap(RB.affine_f3, a)) == [tuple(r) for r in want.tolist()]


def test_device_resident_results_and_range_fetch():
    pool = fiber_b200.Pool(1, results="device")
    try:
        a, want = _args("stats_w64", N, 8)
        res = pool.map(RB.stats_w64, a)
        assert res.on_device and len(res) == N
        assert res[1000:1010] == want[1000:1010].tolist()
        assert res[N - 1] == tuple(want[N - 1].tolist())
        _same(res.array, want)
        x, fx = _args("poly_f64", 1000, 8)
        assert pool.map(RB.poly_f64, x).sum() == sum(fx.tolist())
    finally:
        pool.terminate()
        pool.join()


def test_starmap_apply_and_python_values(pool):
    pts = [(1.0, 2.0, 3.0), (0.5, -1.5, 2.25)]
    assert pool.starmap(RB.norm2_f3, pts) == [RB.norm2_f3(*p) for p in pts]
    assert pool.map(RB.norm2_f3, pts) == [RB.norm2_f3(*p) for p in pts]
    assert pool.apply(RB.norm2_f3, (1.0,), {"z": 3.0, "y": 2.0}) == 14.0
    assert pool.apply(RB.affine_f3, (1.0, 2.0, 3.0)) == (4.0, -2.0, 4.0)
    st = pool.apply(RB.stats_w64, ([1.0, -2.0, 3.0, -4.0, 5.0, 6.0, 7.0, 8.0],))
    assert st[:2] == (24.0, 2) and all(type(v) in (float, int) for v in st)
    assert pool.map(RB.poly_f64, range(5)) == [x * 1.5 + 0.25 for x in range(5)]
    with pytest.raises(TypeError):
        pool.apply(RB.norm2_f3, (1.0, 2.0))
    with pytest.raises(TypeError):
        pool.map(RB.stats_w64, _w64(4)).sum()            # like sum() over a list of tuples


def test_bad_argument_is_raised_from_get(pool):
    a = np.abs(_f3(N, 9)[:, 0])
    a[777_777] = -1.0
    a[900_001] = np.nan
    r = pool.map_async(RB.halve_nonneg, a)
    with pytest.raises(ValueError, match="task 777777"):
        r.get()
    with pytest.raises(ValueError, match="task 777777"):
        r.get()


def test_thread_and_record_twins_are_equal(pool):
    x = _args("poly_f64", N, 10)[0]
    _same(pool.map(RB.poly_f64, x).array, pool.map(RB.poly_f64_thread, x).array)
    _same(pool.map(RB.poly_f64_staged, x).array, pool.map(RB.poly_f64_thread, x).array)
    w = _w64(N, 10)
    _same(pool.map(RB.dot_w64, w).array, pool.map(RB.dot_w64_thread, w).array)


def _tagged(n, seed=11):
    t = np.zeros(n, RB.TAGGED)
    t["x"] = _rng(seed).standard_normal(n).astype(np.float32)
    t["tag"][_rng(seed + 1).choice(n, 40, replace=False)] = 1
    return t


def test_lost_units_are_redispatched_by_a_resilient_pool():
    t = _tagged(N)
    pool = fiber_b200.Pool(2, error_handling=True, ring_bytes=16 << 20)
    try:
        _same(pool.map(RB.triple_or_fault, t).array, RB.triple_or_fault_np(t))
        assert pool.stats()["units_redispatched"] >= 1
    finally:
        pool.terminate()
        pool.join()
    plain = fiber_b200.Pool(1)
    try:
        with pytest.raises(RuntimeError, match="error code 3"):
            plain.map(RB.triple_or_fault, t)
        t["tag"] = 0
        _same(plain.map(RB.triple_or_fault, t).array, RB.triple_or_fault_np(t))
    finally:
        plain.terminate()
        plain.join()


def test_two_workers_in_one_process():
    if fiber_b200.cpu_count() < 2:
        pytest.skip("needs 2 GPUs")
    pool = fiber_b200.Pool(2)
    try:
        for name in ("affine_f3", "stats_w64", "mix_256"):
            a, want = _args(name, N, 12)
            _same(pool.map(_f(name), a).array, want)
    finally:
        pool.terminate()
        pool.join()


def test_process_isolated_pool_registers_the_record_layout():
    pool = fiber_b200.Pool(2, isolation="process")
    try:
        pool.wait_until_workers_up()
        a, want = _args("stats_w64", 300_007, 13)
        _same(np.asarray(pool.map(RB.stats_w64, a)), want)
        pts = [(1.0, 2.0, 3.0), (4.0, 5.0, 6.0)]
        assert pool.starmap(RB.norm2_f3, pts) == [RB.norm2_f3(*p) for p in pts]
        assert pool.apply(RB.norm2_f3, (1.0, 2.0, 3.0)) == 14.0
    finally:
        pool.terminate()
        pool.join()
