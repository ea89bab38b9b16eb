"""CPU: the schedule the engine gives each worker's block of a map -- claim unit, data path, wave size and count --
computed by the library's host-side planner without a device.  Pins the plans of the maps that smoke(), the tests
and bench.py run, so a change to a path decision shows up here before it reaches a GPU."""
import ctypes

import pytest

from fiber_b200 import _abi, registry

# bit k of the planner's path flags (engine.cu, fbr_internal_plan_part)
PATHS = ("args_dev", "out_dev", "keep_on_device", "resilient", "peer_out", "peer_push", "zero_copy", "full_window",
         "host_args", "overlap", "direct")
FAKE_DEVICE_PTR = 1 << 40      # the planner only looks at the alignment of device pointers, it never dereferences them


def _planner():
    lib = _abi.load()
    fn = lib.fbr_internal_plan_part
    u32, u64, i32, P = ctypes.c_uint32, ctypes.c_uint64, ctypes.c_int, ctypes.POINTER
    fn.restype = i32
    fn.argtypes = [P(_abi.MapDesc), u64, u64, i32, i32, i32, u64, u32, i32, P(u32), P(u32), P(u32), P(u64), P(u64)]
    return fn


def _desc(body, n, flags=0, chunksize=32, arg_stride=0, n_items=0, args=None, out=None):
    d = _abi.MapDesc()
    d.func_id = registry.spec(body).func_id
    d.flags, d.n_tasks, d.chunksize, d.arg_stride, d.n_items = flags, n, chunksize, arg_stride, n_items
    d.index_start, d.index_step = 0, 1
    d.args, d.out = args, out
    return d


def plan(d, n_workers=1, worker=0, ring=0, pool_flags=0, has_out=None, root_alive=True):
    """The block of `worker` as fbr_map_submit cuts it (fbr_plan_query), then what the planner decides for it."""
    blk = _abi.Plan()
    _abi.check(_abi.load().fbr_plan_query(d.func_id, d.n_tasks, d.chunksize, ring, n_workers, worker, 148, ctypes.byref(blk)))
    if has_out is None:           # the caller's `out`, or else a pinned segment of the engine's
        has_out = not (d.flags & _abi.FBR_RESULTS_ON_DEVICE)
    unit, stride, flags = ctypes.c_uint32(), ctypes.c_uint32(), ctypes.c_uint32()
    cap, waves = ctypes.c_uint64(), ctypes.c_uint64()
    _abi.check(_planner()(ctypes.byref(d), blk.block_first, blk.block_count, worker, int(root_alive), 148, ring, pool_flags,
                          int(has_out), ctypes.byref(unit), ctypes.byref(stride), ctypes.byref(flags), ctypes.byref(cap),
                          ctypes.byref(waves)))
    # the planner's claim unit is the one fbr_plan_query reports for the same block
    assert (unit.value, stride.value) == (blk.unit_tasks, blk.slot_stride)
    return {"unit": unit.value, "paths": {p for k, p in enumerate(PATHS) if flags.value >> k & 1},
            "wave_tasks": cap.value, "waves": waves.value, "count": blk.block_count}


PI_BITS = dict(body="pi_inside_bits8", n=12_500_000, flags=_abi.FBR_WANT_SUM, n_items=10 ** 8)


def test_pi_map_bit_packed_results_are_stored_zero_copy_in_one_wave():
    # Pool(1).map(is_inside, range(1e8)): the bit-packed twin, chunksize 32 // 8
    p = plan(_desc(chunksize=4, **PI_BITS))
    assert p["paths"] == {"direct", "zero_copy", "full_window"}
    assert (p["unit"], p["waves"]) == (512, 1)


def test_pi_map_staged_for_imap_in_six_waves():
    # imap asks for staged waves (FBR_NO_ZERO_COPY); its default chunksize 1 gives 1 // 8 -> 1
    p = plan(_desc(chunksize=1, **dict(PI_BITS, flags=_abi.FBR_WANT_SUM | _abi.FBR_NO_ZERO_COPY)))
    assert p["paths"] == {"direct"}
    assert (p["unit"], p["waves"], p["wave_tasks"]) == (512, 6, 2_083_840)


def test_pi_map_byte_results_in_eight_waves():
    p = plan(_desc("pi_inside_det", 10 ** 8, _abi.FBR_WANT_SUM))
    assert p["paths"] == {"direct"}
    assert (p["unit"], p["waves"], p["wave_tasks"]) == (4096, 8, 12_500_992)


@pytest.mark.parametrize("flag", ["FBR_SHUFFLE", "FBR_VIA_RING", "FBR_RESILIENT"])
def test_pi_map_through_the_ring(flag):
    for d in (_desc("pi_inside_det", 10 ** 8, _abi.FBR_WANT_SUM | getattr(_abi, flag)),
              _desc(chunksize=4, **dict(PI_BITS, flags=_abi.FBR_WANT_SUM | getattr(_abi, flag)))):
        p = plan(d)
        assert "direct" not in p["paths"] and "zero_copy" not in p["paths"]
        assert ("resilient" in p["paths"]) == (flag == "FBR_RESILIENT")


def test_payload_map_streams_host_records_in_61_waves():
    p = plan(_desc("payload_map_4k", 10 ** 6, arg_stride=4096, args=FAKE_DEVICE_PTR))
    assert p["paths"] == {"direct", "host_args"}
    assert (p["unit"], p["waves"]) == (32, 61)


@pytest.mark.parametrize("ring, waves", [(0, 30), (64 << 20, 31)])
def test_root_resident_payload_map_on_two_workers(ring, waves):
    """Arguments and output on worker 0: worker 0 maps its block in place in one wave; worker 1's waves are pushed in
    by worker 0's copy engine and pushed back by its own (profiles/r02_peer_sweep.txt; bench.py runs a 64 MiB ring)."""
    d = _desc("payload_map_4k", 10 ** 6, _abi.FBR_ARGS_DEVICE | _abi.FBR_OUT_DEVICE, arg_stride=4096,
              args=FAKE_DEVICE_PTR, out=FAKE_DEVICE_PTR)
    root, other = plan(d, 2, 0, ring), plan(d, 2, 1, ring)
    assert root["paths"] == {"args_dev", "out_dev", "full_window", "direct"} and root["waves"] == 1
    assert other["paths"] == {"args_dev", "out_dev", "peer_out", "peer_push", "host_args", "direct"}
    assert other["waves"] == waves and root["count"] + other["count"] == 10 ** 6
    # with worker 0 gone there is no root to push the arguments
    assert "peer_push" not in plan(d, 2, 1, ring, root_alive=False)["paths"]


def test_results_kept_on_device_and_overlapped_gathers():
    p = plan(_desc("pi_inside_det", 10 ** 8, _abi.FBR_WANT_SUM | _abi.FBR_RESULTS_ON_DEVICE))
    assert p["paths"] == {"keep_on_device", "full_window", "direct"} and p["waves"] == 1
    p = plan(_desc("pi_inside_det", 10 ** 8, _abi.FBR_WANT_SUM | _abi.FBR_FULL_WINDOW | _abi.FBR_VIA_RING),
             pool_flags=_abi.FBR_POOL_OVERLAP)
    assert p["paths"] == {"full_window", "overlap"}


def test_planner_rejects_what_it_cannot_plan():
    fn, u32, u64 = _planner(), ctypes.c_uint32(), ctypes.c_uint64()
    out = [ctypes.byref(u32), ctypes.byref(u32), ctypes.byref(u32), ctypes.byref(u64), ctypes.byref(u64)]
    assert fn(ctypes.byref(_desc("pi_inside_det", 10)), 0, 0, 0, 1, 0, 0, 0, 1, *out) == _abi.FBR_EINVAL
    d = _desc("pi_inside_det", 10)
    d.func_id = 999
    assert fn(ctypes.byref(d), 0, 10, 0, 1, 0, 0, 0, 1, *out) == _abi.FBR_EINVAL


def test_environment_does_not_change_the_plan(monkeypatch):
    maps = [_desc(chunksize=4, **PI_BITS), _desc("pi_inside_det", 10 ** 8, _abi.FBR_WANT_SUM),
            _desc("payload_map_4k", 10 ** 6, arg_stride=4096, args=FAKE_DEVICE_PTR)]
    before = [plan(d) for d in maps]
    monkeypatch.setenv("FBR_UNIT_TASKS", "64")
    monkeypatch.setenv("FBR_WAVES", "3")
    monkeypatch.setenv("FBR_MIN_WAVE_KB", "64")
    assert [plan(d) for d in maps] == before
