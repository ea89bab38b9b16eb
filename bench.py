#!/usr/bin/env python
"""bench.py -- Pool.map tasks/sec on B200 (BASELINE.json metric), one JSON line on rank 0.

    python bench.py --gpus 1 --steps 10 --warmup 3            # this repo's arm
    python bench.py --impl reference --steps 3 --warmup 1     # CPU arm: the reference's own ZPool
    torchrun ... bench.py --gpus N ...                        # one rank per GPU

A "step" is one pass of the hot path over one batch of synthetic tasks:

* headline workload  ``pi_estimation 1e8 samples, 1 GPU persistent-kernel Pool, int result gather``
  (BASELINE.json configs[1]): ``Pool.map(is_inside_det, range(r*1e8, (r+1)*1e8))`` on rank r
  (weak scaling, the map shards by index block with no data-path collective; the scalar count is
  summed over ranks with one NCCL all-reduce per step when N > 1).
  - ``value``  : whole-job tasks/s with everything resident in HBM (index arguments need no input
                 bytes; ordered uint8 results + int64 count stay on the device).  A contiguous map is
                 placed directly at its final index by the dispatch kernel (one launch per step).
  - ``e2e``    : the same through the reference-facing call ``fiber_b200.Pool.map`` -- ordered results
                 D2H into the pinned result segment (bool results travel one bit each by default),
                 count read on the host -- all inside the timed region.
  - ``roofline``: the result-gather kernel the north-star names (gather_ordered), timed live with CUDA
                 events on the engine's compute stream (FBR_POOL_TIMING) in a leg where it has to run:
                 the same 1e8-task map with task records shuffled inside each wave, so ring (arrival)
                 order != index order and every unit is placed by its header.
* ``parzen``   : BASELINE.json configs[2] -- 102 window widths via apply_async (as the example) and via
                 starmap(chunksize=1), kernel time, L2 read rate, fp32 boundary mismatches, CPU time.
* ``payload4k``: ``synthetic 4 KB-payload map, 1e6 tasks`` (configs[3], per GPU): the HBM-bound kernels at
                 8.2 GB per launch (dispatch_payload_map_tma, gather_bulk).

``cpu_baseline`` / ``--impl reference`` time the UNMODIFIED reference pool on this box's host cores: its
``fiber`` package compiled to bytecode in ``oracle/_ref/fiber`` by ``__graft_entry__.build()``
(``oracle/ref_pyc.py``, git-ignored, with the one constant ``socket_lib = "nanomsg" -> "zmq"`` because nnpy
is not installable offline); if that build is missing or fails, the oracle port of ZPool
(``oracle/zpool_port.py``) stands in and the line says ``kind: "port"``.

``--steps K`` is the number of timed steps of every GPU leg (the CPU baseline arms keep fixed repetitions).  ``--dump-outputs DIR`` writes what the headline
leg's last timed step computed (see ``dump_pi_outputs``) as ``DIR/<name>.npy``; the inputs depend only on the
arguments, so two builds can be compared output for output.
"""
import argparse
import ctypes
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PI_TASKS = 10 ** 8
PAYLOAD_TASKS = 10 ** 6
CPU_SAMPLE_TASKS = 10 ** 6
REF_DIR = os.path.join(ROOT, "oracle", "_ref")


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return json.load(fh), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback (B200_PROFILING.md)"


def _newest(pattern):
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", pattern)))
    return files[-1] if files else None


def load_imad_peak():
    """Measured IMAD.WIDE.U32 rate of this GPU model (profiles/microbench/imad_peak.cu, committed summary)."""
    path = _newest("r*_imad_peak.json")
    try:
        with open(path) as fh:
            d = json.load(fh)
        best = max(v["Gops"] for k, v in d.items() if k.startswith("imad_wide_u32"))
        body = max(v["tasks_per_s"] for k, v in d.items() if k.startswith("pi_body_screened"))
        return {"gops": best, "source": os.path.relpath(path, ROOT) + " (measured)", "pi_body_screened_tasks_per_s": "%.3g" % body}
    except (OSError, ValueError, KeyError, TypeError):
        return {"gops": None, "source": "unavailable", "pi_body_screened_tasks_per_s": "n/a"}


def source_digest():
    """sha256 over the CUDA sources and headers of the library, in sorted order (same recipe as profiles/run_ncu.sh)."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "fiber_b200", "csrc", "*.cu")) + glob.glob(os.path.join(ROOT, "fiber_b200", "csrc", "*.cuh")) +
                   glob.glob(os.path.join(ROOT, "include", "*.h")) + glob.glob(os.path.join(ROOT, "include", "*.cuh")))
    h = hashlib.sha256()
    for f in files:
        with open(f, "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def load_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch (and the capture's commit) from the committed
    `ncu --set full` capture of profiles/prof_target.py (same kernels, same sizes); newest round wins."""
    path = _newest("r*_traffic.json")
    if not path:
        return {}, None
    with open(path) as fh:
        return json.load(fh), os.path.relpath(path, ROOT)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines, self.stamps, self.windows = gpu_index, None, [], [], []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())
            self.stamps.append(time.perf_counter())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        inside = [ln for ln, ts in zip(self.lines, self.stamps)
                  if any(a - 0.11 <= ts <= b + 0.11 for a, b in self.windows)]
        window = "timed regions (+-110 ms)"
        if len(inside) < 3:
            inside, window = self.lines, "whole bench run (timed regions are shorter than the 100 ms sampling period)"
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for nm, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "window": window,
                "reasons": sorted(reasons)}


class NvlinkCounters:
    """NVML per-GPU NVLink payload counters (KiB, all links): bytes sent / received by one GPU over a region."""

    def __init__(self, gpu_index):
        self.h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.read()
        except Exception:
            self.h = None

    def read(self):
        if self.h is None:
            return None
        nv = self.nv
        vals = nv.nvmlDeviceGetFieldValues(self.h, [(nv.NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_TX, 0xFFFFFFFF),
                                                    (nv.NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_RX, 0xFFFFFFFF)])
        out = []
        for v in vals:
            if v.nvmlReturn != 0:
                return None
            out.append(int(v.value.ullVal) * 1024)
        return tuple(out)     # (tx bytes, rx bytes)


# ------------------------------------------------------------------------------------------------
# distributed plumbing (torch.distributed is plumbing only: barrier, max-reduce, count all-reduce)
# ------------------------------------------------------------------------------------------------
class Dist:
    def __init__(self, want_gpus, backend="nccl"):
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.torch = None
        if self.world > 1:
            import torch
            import torch.distributed as dist
            self.torch, self.dist = torch, dist
            if backend == "nccl":
                torch.cuda.set_device(self.local_rank)
            # NCCL prints its version banner on stdout when the first communicator is created; rank 0's stdout
            # carries ONE JSON line, so fd 1 points at stderr until that has happened
            sys.stdout.flush()
            saved = os.dup(1)
            os.dup2(2, 1)
            try:
                dist.init_process_group(backend=backend)
                dist.barrier()
                if backend == "nccl":
                    torch.cuda.synchronize()
            finally:
                sys.stdout.flush()
                os.dup2(saved, 1)
                os.close(saved)
        if want_gpus != self.world and self.world > 1:
            raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (want_gpus, self.world))
        # the engine's own communicator (fbr_comm_* = NCCL behind the C ABI) carries every exchange step that
        # belongs to the path (count fold, scatter / gather of blocks); torch.distributed only bootstraps it
        # (its c10d store publishes the 128-byte id) and provides the barrier of the timing bracket
        self.comm = None
        self.comm_error = None
        if self.world > 1 and backend == "nccl":
            from fiber_b200 import comm as C
            try:
                self.comm = C.Comm.from_store(dist.distributed_c10d._get_default_store(), self.local_rank, self.world, self.rank)
            except Exception as e:      # noqa: BLE001 -- e.g. no loadable NCCL build: the exchanges fall back to torch.distributed
                self.comm, self.comm_error = None, "%s: %s" % (type(e).__name__, e)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
            if self.torch.cuda.is_available():
                self.torch.cuda.synchronize()

    def max(self, x):
        if self.world == 1:
            return x
        dev = "cuda" if self.dist.get_backend() == "nccl" else "cpu"
        t = self.torch.tensor([x], dtype=self.torch.float64, device=dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_i64(self, x):
        if self.world == 1:
            return x
        if self.comm is not None:
            return self.comm.allreduce_i64(x)          # ncclAllReduce(sum, int64) through the C ABI
        dev = "cuda" if self.dist.get_backend() == "nccl" else "cpu"
        t = self.torch.tensor([x], dtype=self.torch.int64, device=dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return int(t.item())

    def sum_i64_vector(self, xs):
        """Global element-wise sum of one int64 vector per rank (one ncclAllReduce through the C ABI)."""
        if self.world == 1:
            return list(xs)
        if self.comm is not None:
            import numpy as np
            from fiber_b200 import comm as C
            a = np.asarray(xs, dtype=np.int64)
            buf = self.comm.alloc(a.nbytes).upload(a)
            self.comm.allreduce(buf, buf, len(a), C.I64, C.SUM)
            self.comm.sync()
            out = buf.download(np.int64).tolist()
            buf.free()
            return out
        return [self.sum_i64(x) for x in xs]

    def sum_i64_begin(self, x):
        """Start the global fold of one int64 per rank; `sum_i64_end` collects it.  On the engine communicator the
        fold runs on its own stream and overlaps the next map (one fold in flight)."""
        if self.comm is not None:
            self.comm.allreduce_i64_begin(x)
            self._fold = None
        else:
            self._fold = self.sum_i64(x)

    def sum_i64_end(self):
        return self.comm.allreduce_i64_end() if (self.comm is not None and self._fold is None) else self._fold

    def all_true(self, flag):
        return self.sum_i64(0 if flag else 1) == 0

    def gather_objects(self, obj):
        """Every rank's picklable `obj`, in rank order, on every rank."""
        if self.world == 1:
            return [obj]
        out = [None] * self.world
        self.dist.all_gather_object(out, obj)
        return out

    def finish(self):
        if self.world > 1:
            if self.comm is not None:
                self.comm.destroy()
            self.dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------
# raw C-ABI steps with device-resident buffers (the `value` measurement)
# ------------------------------------------------------------------------------------------------
class RawEngine:
    def __init__(self, device, ring_bytes, flags=0):
        from fiber_b200 import _abi, registry
        self.abi, self.registry = _abi, registry
        self.lib = _abi.load()
        ids = (ctypes.c_int * 1)(device)
        self.h = ctypes.c_void_p()
        _abi.check(self.lib.fbr_pool_create(1, ids, ring_bytes, _abi.FBR_POOL_TIMING | flags, ctypes.byref(self.h)))
        self.deferred = []

    def dalloc(self, nbytes):
        p = ctypes.c_void_p()
        self.abi.check(self.lib.fbr_device_alloc(self.h, 0, nbytes, ctypes.byref(p)))
        return p

    def dfree(self, p):
        self.lib.fbr_device_free(self.h, 0, p)

    def d2h(self, dptr, nbytes, offset=0):
        import numpy as np
        host = np.empty(nbytes, dtype=np.uint8)
        self.abi.check(self.lib.fbr_memcpy_d2h(self.h, 0, host.ctypes.data, ctypes.c_void_p(dptr.value + offset), nbytes))
        return host

    def submit(self, body, n, out_dev, args_dev=None, arg_stride=0, index_start=0, task_base=0, want_sum=True, extra_flags=0, seed=0):
        a = self.abi
        spec = self.registry.spec(body)
        d = a.MapDesc()
        d.func_id = spec.func_id
        d.flags = a.FBR_OUT_DEVICE | (a.FBR_WANT_SUM if want_sum else 0) | (a.FBR_ARGS_DEVICE if args_dev else 0) | extra_flags
        d.n_tasks, d.chunksize, d.arg_stride = n, 0, arg_stride
        d.args = args_dev
        d.index_start, d.index_step = index_start, 1
        d.out = out_dev
        d.task_index_base = task_base
        d.shuffle_seed = seed
        seq = ctypes.c_uint64(0)
        a.check(self.lib.fbr_map_submit(self.h, ctypes.byref(d), ctypes.byref(seq)))
        return seq.value

    def wait(self, seq, release=True):
        res = self.abi.Result()
        self.abi.check(self.lib.fbr_result_wait(self.h, seq, -1, ctypes.byref(res)))
        out = (int(res.sum), int(res.n_waves))
        if release:
            self.abi.check(self.lib.fbr_result_release(self.h, seq))
        else:
            self.deferred.append(seq)
        return out

    def release_deferred(self):
        """Return finished maps' segments/events to the pool (host bookkeeping, outside timing)."""
        while self.deferred:
            self.abi.check(self.lib.fbr_result_release(self.h, self.deferred.pop()))

    def stats(self, reset=False):
        s = self.abi.Stats()
        self.abi.check(self.lib.fbr_pool_stats(self.h, ctypes.byref(s)))
        if reset:
            self.abi.check(self.lib.fbr_pool_stats_reset(self.h))
        return s.as_dict()

    def close(self):
        self.lib.fbr_pool_destroy(self.h)
        self.h = None


def timed_steps(dist, steps, warmup, step_fn, drain_fn=None, clock_windows=None):
    """W untimed steps, then exactly K steps between barrier+sync brackets; max over ranks."""
    for _ in range(warmup):
        step_fn()
    if drain_fn:
        drain_fn()
    dist.barrier()                 # every rank starts its K steps together (barrier + device sync)
    t0 = time.perf_counter()
    for _ in range(steps):
        step_fn()
    if drain_fn:
        drain_fn()                 # blocks until this rank's last step is complete on the device
    t1 = time.perf_counter()
    dist.barrier()                 # closing bracket; its own latency (an NCCL all-reduce) is not part of the K steps:
    if clock_windows is not None:  # the job's time is the slowest rank's, taken by the max below
        clock_windows.append((t0, t1))
    return dist.max(t1 - t0)


# ------------------------------------------------------------------------------------------------
# oracle helpers (checker only; never inside a timed region)
# ------------------------------------------------------------------------------------------------
def _threads(n_jobs):
    return max(1, min(n_jobs, (os.cpu_count() or 1) // 2, 32))


def _parallel(jobs):
    """Run callables on host threads (the C oracle releases the GIL) and return their results in order."""
    out = [None] * len(jobs)
    errs = []

    def run(i):
        try:
            out[i] = jobs[i]()
        except Exception as e:      # noqa: BLE001
            errs.append(e)
    nt = _threads(len(jobs))
    idx = list(range(len(jobs)))
    ths = [threading.Thread(target=lambda s=s: [run(i) for i in idx[s::nt]]) for s in range(nt)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    if errs:
        raise errs[0]
    return out


def oracle_payload_equal(got_u32, t0):
    """FULL comparison of mapped 4 KB records (rows of `got_u32`, task t0 + row) against the C oracle."""
    import numpy as np
    from oracle import cref
    n = got_u32.shape[0]
    step = 8192
    jobs = [(lambda a=a: bool(np.array_equal(got_u32[a:a + step], cref.payload_map(t0 + a, cref.payload_records(t0 + a, min(step, n - a))))))
            for a in range(0, n, step)]
    return all(_parallel(jobs))


def oracle_pi_equal(got_u8, first):
    """FULL comparison of ordered is_inside results (one byte each) against the C oracle."""
    import numpy as np
    from oracle import cref
    n = got_u8.shape[0]
    step = 1 << 24
    jobs = [(lambda a=a: bool(np.array_equal(got_u8[a:a + step], cref.pi_inside_range(first + a, min(step, n - a))[0])))
            for a in range(0, n, step)]
    return all(_parallel(jobs))


DUMP_SAMPLE = 1 << 20
DUMP_BLOCK = 10 ** 4


def dump_pi_outputs(out_dir, got_u8, first, total_count, dist):
    """Write what a caller of the headline map receives -- the ordered is_inside results of every rank's
    tasks [first, first + n) and the job's count -- as float64/float32 .npy files on rank 0 (about 12 MB
    in all; every rank calls this, its part travels to rank 0):
      pi_inside_index.npy  float64  a fixed sample of task indices (seed 0, sorted, unique; DUMP_SAMPLE / world
                                    draws per rank, ranks in order)
      pi_inside_sample.npy float32  the results at those indices (0 or 1)
      pi_block_counts.npy  float64  the number of true results in every block of DUMP_BLOCK consecutive tasks
      pi_count.npy         float64  [the count over all ranks]"""
    import numpy as np
    n = got_u8.shape[0]
    idx = np.unique(np.random.default_rng(0).integers(0, n, DUMP_SAMPLE // dist.world))
    blocks = np.add.reduceat(got_u8, np.arange(0, n, DUMP_BLOCK), dtype=np.int64)
    parts = dist.gather_objects((first, got_u8[idx], blocks))
    if dist.rank != 0:
        return
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in (("pi_inside_index", np.concatenate([f + idx for f, _, _ in parts]).astype(np.float64)),
                      ("pi_inside_sample", np.concatenate([s for _, s, _ in parts]).astype(np.float32)),
                      ("pi_block_counts", np.concatenate([b for _, _, b in parts]).astype(np.float64)),
                      ("pi_count", np.array([total_count], dtype=np.float64))):
        np.save(os.path.join(out_dir, name + ".npy"), arr)


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's own pool (oracle/_ref/fiber), or its oracle port, in a child process
# ------------------------------------------------------------------------------------------------
def _cpu_child(spec):
    """Runs in a fresh interpreter (`bench.py --cpu-child <json>`): the reference pool's workers re-import
    __main__ (spawn), so the arm lives in its own process, bounded by the parent's timeout."""
    kind, P, n, reps, warm = spec["kind"], spec["P"], spec["n"], spec["reps"], spec["warm"]
    from oracle import cref
    cref.lib()   # build/load the C body before the workers start
    if kind == "reference":
        import fiber
        assert os.path.realpath(fiber.__file__).startswith(os.path.realpath(REF_DIR)), fiber.__file__
        pool = fiber.Pool(P)
        impl = "%s (fiber %s, socket_lib=%s)" % (type(pool).__name__, getattr(fiber, "__version__", "?"), __import__("fiber.socket").socket.socket_lib)
    else:
        from oracle.zpool_port import PortPool
        pool = PortPool(P)
        impl = "oracle/zpool_port.PortPool"
    out = {"impl": impl}
    if spec["work"] == "pi":
        pool.map(cref.pi_inside_det_c, range(1000))          # excludes lazy worker start-up
        times, count = [], None
        for i in range(warm + reps):
            t0 = time.perf_counter()
            res = pool.map(cref.pi_inside_det_c, range(n))   # default chunksize 32, list in hand
            dt = time.perf_counter() - t0
            if i >= warm:
                times.append(dt)
            count = sum(res)
        out.update({"times": times, "count": count})
    else:   # parzen: exactly examples/parzen_estimation.py:22-40 (apply_async per width)
        from oracle import bodies as B
        xs, px, widths = B.parzen_example_inputs()
        pool.map(cref.pi_inside_det_c, range(1000))
        times = []
        for i in range(reps):
            t0 = time.perf_counter()
            handles = [pool.apply_async(B.parzen_estimation, args=(xs, px, w)) for w in widths]
            res = [h.get() for h in handles]
            times.append(time.perf_counter() - t0)
        res.sort()
        out.update({"times": times, "n_tasks": len(widths), "first": list(res[0]), "last": list(res[-1])})
    pool.terminate()
    pool.join()
    print("CPU_CHILD_RESULT " + json.dumps(out), flush=True)


def cpu_arm(work, P, n=CPU_SAMPLE_TASKS, reps=3, warm=1, timeout=420):
    """-> (result dict, kind).  Tries the real reference first, then the port; a port result that stands in
    for a failed reference arm says why in its ``impl``."""
    import tempfile
    kinds = ["reference", "port"] if os.path.isdir(os.path.join(REF_DIR, "fiber")) else ["port"]
    last_err = None
    for kind in kinds:
        env = dict(os.environ)
        paths = ([REF_DIR] if kind == "reference" else []) + [ROOT, env.get("PYTHONPATH", "")]
        env["PYTHONPATH"] = os.pathsep.join(p for p in paths if p)
        env.pop("RANK", None)
        spec = {"kind": kind, "P": P, "n": n, "reps": reps, "warm": warm, "work": work}
        try:
            # the reference logs to /tmp/fiber.log.<process> by default: a private directory keeps files another user
            # left there from failing the arm, and leaves nothing behind
            with tempfile.TemporaryDirectory(prefix="fbr_cpu_arm_") as logs:
                env["FIBER_LOG_FILE"] = os.path.join(logs, "fiber.log")
                cp = subprocess.run([sys.executable, os.path.abspath(__file__), "--cpu-child", json.dumps(spec)], env=env, cwd=ROOT,
                                    stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=timeout)
            for ln in cp.stdout.splitlines():
                if ln.startswith("CPU_CHILD_RESULT "):
                    res = json.loads(ln[len("CPU_CHILD_RESULT "):])
                    if last_err:
                        res["impl"] = "%s (standing in: %s)" % (res.get("impl"), last_err[-200:])
                    return res, kind
            last_err = "%s arm printed no result (rc %d): %s" % (kind, cp.returncode, cp.stderr[-300:])
        except subprocess.TimeoutExpired:
            last_err = "%s arm timed out after %d s" % (kind, timeout)
    raise RuntimeError(last_err)


def run_reference(args, dist):
    """--impl reference: the reference's own CPU implementation of the path on this box's host cores."""
    if dist.rank != 0:
        return
    cores = os.cpu_count() or 1
    try:
        res, kind = cpu_arm("pi", cores, reps=max(1, args.steps), warm=max(0, min(args.warmup, 1)),
                            timeout=max(420, 30 + 6 * max(1, args.steps)))
    except Exception as e:      # noqa: BLE001 -- neither the reference copy nor its port could run: say so, exit 0
        print(json.dumps({"impl": "reference", "unavailable": str(e)[:300]}), flush=True)
        return
    times = res["times"]
    total = sum(times)
    value = CPU_SAMPLE_TASKS * len(times) / total
    extra = {}
    try:        # examples/pi_estimation.py:15 uses Pool(processes=4): BASELINE.json configs[0]
        r4, k4 = cpu_arm("pi", 4, reps=2, warm=0)
        extra["pool4"] = {"value": CPU_SAMPLE_TASKS / min(r4["times"]), "unit": "tasks/s", "cores": 4, "kind": k4,
                          "sample": "best of 2 Pool(4).map over %d tasks (BASELINE.json configs[0])" % CPU_SAMPLE_TASKS}
    except Exception as e:      # noqa: BLE001
        extra["pool4"] = {"unavailable": str(e)[:200]}
    line = {
        "impl": "reference", "metric": "pool_map_tasks_per_sec", "value": value, "unit": "tasks/s",
        "n_gpus": args.gpus, "steps": len(times), "warmup": args.warmup,
        "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64->u8", "data": "synthetic",
        "config": {"workload": "pi_estimation Pool.map over 1e8 index tasks per GPU (BASELINE.json configs[1])",
                   "step_sample": "one Pool(processes=%d).map of %d tasks, default chunksize 32 (a rate: the CPU pool's tasks/s "
                                  "does not depend on the map length)" % (cores, CPU_SAMPLE_TASKS),
                   "tasks_per_step": CPU_SAMPLE_TASKS},
        "cpu_baseline": {"value": value, "unit": "tasks/s", "cores": cores, "kind": kind, "impl": res.get("impl"),
                         "sample": "%d maps of %d pi_inside_det tasks (C body via ctypes), %d worker processes"
                                   % (len(times), CPU_SAMPLE_TASKS, cores), **extra},
        "e2e": {"value": value, "unit": "tasks/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "check": {"count": res["count"]},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# multi-GPU sections
# ------------------------------------------------------------------------------------------------
def fused_peer_map(n_gpus, n_total, steps):
    """Root-resident 4 KB map over an in-process pool of `n_gpus` workers: inputs and ordered outputs
    stay on GPU 0; every worker's dispatch kernel bulk-loads its block from GPU 0 and bulk-stores its
    results at their final index on GPU 0 over NVLink peer memory, in the same kernel -- the scatter,
    the map and the gather are one launch per worker and the root's links run in both directions at once."""
    import numpy as np
    from fiber_b200 import _abi, registry
    lib = _abi.load()
    ids = (ctypes.c_int * n_gpus)(*range(n_gpus))
    h = ctypes.c_void_p()
    _abi.check(lib.fbr_pool_create(n_gpus, ids, 64 << 20, 0, ctypes.byref(h)))      # staging halves of 64 MiB = one wave
    try:
        din, dout = ctypes.c_void_p(), ctypes.c_void_p()
        _abi.check(lib.fbr_device_alloc(h, 0, n_total * 4096, ctypes.byref(din)))
        _abi.check(lib.fbr_device_alloc(h, 0, n_total * 4096, ctypes.byref(dout)))
        _abi.check(lib.fbr_payload_fill_device(h, 0, din, 0, n_total))
        d = _abi.MapDesc()
        d.func_id = registry.spec("payload_map_4k").func_id
        d.flags = _abi.FBR_ARGS_DEVICE | _abi.FBR_OUT_DEVICE
        d.n_tasks, d.arg_stride, d.args, d.out = n_total, 4096, din.value, dout.value
        res = _abi.Result()

        def step():
            seq = ctypes.c_uint64()
            _abi.check(lib.fbr_map_submit(h, ctypes.byref(d), ctypes.byref(seq)))
            _abi.check(lib.fbr_result_wait(h, seq.value, -1, ctypes.byref(res)))
            _abi.check(lib.fbr_result_release(h, seq.value))
        for _ in range(3):
            step()
        nvl = NvlinkCounters(0)
        c0 = nvl.read()
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        dt = time.perf_counter() - t0
        c1 = nvl.read()
        st = _abi.Stats()
        _abi.check(lib.fbr_pool_stats(h, ctypes.byref(st)))
        # FULL parity: every byte of the ordered output on GPU 0 against the C oracle
        got = np.empty((n_total, 1024), dtype=np.uint32)
        _abi.check(lib.fbr_memcpy_d2h(h, 0, got.ctypes.data, dout, got.nbytes))
        ok = oracle_payload_equal(got, 0)
        sha = hashlib.sha256(got.tobytes()).hexdigest()
        del got
        lib.fbr_device_free(h, 0, din)
        lib.fbr_device_free(h, 0, dout)
        link_bytes = n_total * 4096 * (n_gpus - 1) / n_gpus      # each way: peer loads out of / peer stores into GPU 0
        out = {"value": n_total * steps / dt, "unit": "tasks/s", "ms_per_step": 1e3 * dt / steps,
               "root_link_GBps_each_way": link_bytes / (dt / steps) / 1e9,
               "nvlink_ref_GBps": 770.0, "frac_of_peer_copy_ref": link_bytes / (dt / steps) / 1e9 / 770.0,
               "parity_full": ok, "checked_bytes": n_total * 4096, "sha256": sha,
               "direct_waves": int(st.direct_waves), "gather_launches": int(st.gather_launches),
               "note": "in-process Pool(%d): args/out on GPU 0; each wave of a non-root worker's block is pushed into its staging by "
                       "the root's copy engine, mapped locally, and pushed back into the root's output by the worker's copy engine "
                       "(posted writes both ways, 64 MB waves); FBR_PEER_PUSH=0 FBR_PEER_OUT=0 selects the single-kernel "
                       "variant with peer loads + stores" % n_gpus}
        if c0 and c1:
            out["nvml_gpu0_nvlink"] = {"tx_GBps": (c1[0] - c0[0]) / dt / 1e9, "rx_GBps": (c1[1] - c0[1]) / dt / 1e9,
                                      "source": "NVML NVLINK_THROUGHPUT_DATA_TX/RX (all links) around the timed steps"}
        return out
    finally:
        lib.fbr_pool_destroy(h)


def inprocess_pool_e2e(n_gpus, steps):
    """The literal drop-in usage: ONE process, `fiber_b200.Pool(processes=N)` over all N GPUs,
    `pool.map(is_inside, range(N * 1e8))` -> one pinned ResultArray (each GPU D2Hs its block) + count."""
    import numpy as np
    import fiber_b200
    from examples import workloads as W
    pool = fiber_b200.Pool(n_gpus)
    n = n_gpus * PI_TASKS
    counts = []

    def step():
        res = pool.map(W.is_inside, range(n))
        counts.append(res.sum())
        step.last = res
    for _ in range(3):
        step()
    k = steps
    t0 = time.perf_counter()
    for _ in range(k):
        step()
    dt = time.perf_counter() - t0
    # FULL parity of the last step's ordered results (bit-packed in the pinned segment) against the C oracle
    got = np.unpackbits(step.last.packed, count=n, bitorder="little")
    ok = oracle_pi_equal(got, 0) and counts[-1] == int(got.sum())
    step.last = None
    pool.terminate()
    pool.join()
    return {"value": n * k / dt, "unit": "tasks/s", "ms_per_step": 1e3 * dt / k, "tasks_per_step": n, "count": counts[-1],
            "parity_full": ok, "checked_tasks": n,
            "api": "fiber_b200.Pool(%d).map(is_inside_det, range(%d)) in one process -> pinned bit-packed ResultArray + count" % (n_gpus, n)}


def run_multi_gpu(args, dist, dev):
    """BASELINE.json configs[3] and [4] on N GPUs (torch.distributed/NCCL is the exchange plumbing;
    the map itself runs through the C ABI on torch-allocated device buffers):
      * payload4k_sharded: 1e6 tasks TOTAL, contiguous block per rank (strong scaling):
        (i) shard-resident, (ii) including NCCL scatter from rank 0 and gather to rank 0,
        (iii) root-resident with scatter+gather fused into the dispatch kernel over peer memory;
      * ring_allreduce: 256 MiB fp32 all-reduce across the ring (experimental.Ring's collective).
    Every path's output is compared IN FULL with the C oracle outside the timed loops."""
    import numpy as np
    import torch
    import torch.distributed as td
    from fiber_b200 import _abi, shard
    from fiber_b200.experimental import allreduce_bench

    rank, world = dist.rank, dist.world
    n_total = PAYLOAD_TASKS
    lo, hi = shard.block_of(n_total, rank, world)
    n_loc = hi - lo
    width = max(b - a for a, b in shard.blocks(n_total, world))
    cuda = torch.device("cuda", dev)
    eng = RawEngine(dev, 64 << 20)
    inp = torch.empty(width * 1024, dtype=torch.int32, device=cuda)
    out = torch.empty(width * 1024, dtype=torch.int32, device=cuda)
    _abi.check(eng.lib.fbr_payload_fill_device(eng.h, 0, ctypes.c_void_p(inp.data_ptr()), lo, n_loc))
    torch.cuda.synchronize()

    pend = []

    def submit_map():
        pend.append(eng.submit("payload_map_4k", n_loc, ctypes.c_void_p(out.data_ptr()), args_dev=ctypes.c_void_p(inp.data_ptr()),
                               arg_stride=4096, task_base=lo, want_sum=False))

    def drain_maps():
        while pend:
            eng.wait(pend.pop(0), release=False)

    def local_map():
        submit_map()
        drain_maps()

    for _ in range(3):
        local_map()
    eng.release_deferred()
    t_res = timed_steps(dist, args.steps, 0, submit_map, drain_maps)      # steps queue back to back
    eng.release_deferred()
    # (i) full parity of this rank's shard-resident block
    mine = out[: n_loc * 1024].cpu().numpy().view(np.uint32).reshape(n_loc, 1024)
    ok_shard = dist.all_true(oracle_payload_equal(mine, lo))
    del mine

    # (ii) scatter from rank 0 -> map -> gather to rank 0 (root-ingress bound over NVLink)
    full_in = full_out = None
    if rank == 0:
        full_in = torch.empty(world * width * 1024, dtype=torch.int32, device=cuda)
        full_out = torch.zeros(world * width * 1024, dtype=torch.int32, device=cuda)
        for r, (a, b) in enumerate(shard.blocks(n_total, world)):
            _abi.check(eng.lib.fbr_payload_fill_device(eng.h, 0, ctypes.c_void_p(full_in.data_ptr() + r * width * 4096), a, b - a))
        torch.cuda.synchronize()
    out.zero_()

    comm = dist.comm
    blk_bytes = width * 4096

    def scattered_map():
        # fan-out and fan-in of the reference's master sockets (fiber/pool.py:910-920) as grouped ncclSend/ncclRecv
        # issued by the engine's communicator; the map in between is the shard-resident one
        if comm is None:            # engine communicator unavailable (see Dist): same exchange through torch.distributed
            td.scatter(inp, list(full_in.chunk(world)) if rank == 0 else None, src=0)
            torch.cuda.synchronize()
            local_map()
            td.gather(out, list(full_out.chunk(world)) if rank == 0 else None, dst=0)
            torch.cuda.synchronize()
            return
        comm.scatter(full_in if rank == 0 else None, inp, blk_bytes, root=0)
        comm.sync()
        local_map()
        comm.gather(out, full_out if rank == 0 else None, blk_bytes, root=0)
        comm.sync()

    for _ in range(2):
        scattered_map()
    eng.release_deferred()
    t_sc = timed_steps(dist, args.steps, 0, scattered_map)
    eng.release_deferred()
    ok_gathered = True
    if rank == 0:       # full parity of the gathered output on rank 0, block by block
        for r, (a, b) in enumerate(shard.blocks(n_total, world)):
            blk = full_out[r * width * 1024: r * width * 1024 + (b - a) * 1024].cpu().numpy().view(np.uint32).reshape(b - a, 1024)
            ok_gathered &= oracle_payload_equal(blk, a)
            del blk
    eng.close()
    del inp, out, full_in, full_out
    torch.cuda.empty_cache()

    # (iii) the same root-resident map with scatter and gather FUSED into the dispatch kernel: one in-process
    # pool on rank 0 drives all N GPUs; arguments and ordered output live on GPU 0.
    fused = inproc = None
    # the other ranks wait on the HOST (store key), not in an NCCL barrier: a spinning NCCL kernel on
    # their GPUs would compete with the peer traffic being measured
    store = td.distributed_c10d._get_default_store()
    if rank == 0:
        try:
            fused = fused_peer_map(world, n_total, args.steps)
        except Exception as e:          # e.g. the launcher restricted CUDA_VISIBLE_DEVICES per rank
            fused = {"unavailable": "%s: %s" % (type(e).__name__, e)}
        try:
            inproc = inprocess_pool_e2e(world, args.steps)
        except Exception as e:
            inproc = {"unavailable": "%s: %s" % (type(e).__name__, e)}
        store.set("fbr_fused_done", "1")
    else:
        store.wait(["fbr_fused_done"])
    dist.barrier()
    from fiber_b200 import comm as C
    t_ok, t_algbw, t_busbw, t_ms = allreduce_bench(64 * 1024 * 1024, steps=args.steps, warmup=3, device=cuda)
    if comm is not None:
        ar_ok, algbw, busbw, ar_ms = C.allreduce_bench(comm, 64 * 1024 * 1024, steps=args.steps, warmup=3)
    else:
        ar_ok, algbw, busbw, ar_ms = t_ok, t_algbw, t_busbw, t_ms
    return {
        "payload4k_sharded": {
            "workload": "synthetic 4 KB-payload map, %d tasks TOTAL in contiguous blocks over %d GPUs (BASELINE.json configs[3])" % (n_total, world),
            "scaling": "strong",
            "shard_resident": {"value": n_total * args.steps / t_res, "unit": "tasks/s", "ms_per_step": 1e3 * t_res / args.steps,
                               "parity_full": ok_shard, "checked_bytes": n_total * 4096},
            "scatter_map_gather_root0": {"value": n_total * args.steps / t_sc, "unit": "tasks/s", "ms_per_step": 1e3 * t_sc / args.steps,
                                         "parity_full": ok_gathered, "checked_bytes": n_total * 4096,
                                         "note": "fbr_comm_scatter (grouped ncclSend/ncclRecv) from rank 0 + map + fbr_comm_gather to rank 0, "
                                                 "all through the C ABI; root link-bound"},
            "fused_peer_memory_root0": fused},
        "inprocess_pool_e2e": inproc,
        "ring_allreduce": {"workload": "all-reduce SUM of 64 Mi fp32 (256 MiB) per rank, %d ranks (BASELINE.json configs[4])" % world,
                           "bit_exact": ar_ok, "algbw_GBps": algbw, "busbw_GBps": busbw, "ms": ar_ms,
                           "api": "fbr_comm_allreduce (ncclAllReduce behind the C ABI, bootstrap id from the ring member table)"
                                  if comm is not None else "torch.distributed (engine communicator unavailable: %s)" % dist.comm_error,
                           "torch_distributed_same_buffer": {"bit_exact": t_ok, "busbw_GBps": t_busbw, "ms": t_ms},
                           "nvlink_ref": "measured refs: 725 GB/s all-reduce busbw @1 GiB, 770 GB/s peer copy (B200_PROFILING.md)"},
    }


# ------------------------------------------------------------------------------------------------
# parzen (BASELINE.json configs[2])
# ------------------------------------------------------------------------------------------------
def run_parzen(dev, traffic, with_cpu, steps):
    """102 window widths over the 10 000 x 2 sample set of examples/parzen_estimation.py:32-40 through
    apply_async (as the example) and starmap(chunksize=1); fp32 body = the north-star's path."""
    import numpy as np
    import fiber_b200
    from examples import workloads as W
    from oracle import bodies as B, cref
    xs, px, widths = B.parzen_example_inputs()
    n = len(xs)
    pool = fiber_b200.Pool(1, devices=[dev], timing=True)
    items = [(xs, px, w) for w in widths]

    def job_apply():
        hs = [pool.apply_async(W.parzen_estimation_f32, args=(xs, px, w)) for w in widths]
        return [h.get() for h in hs]

    def job_star():
        return pool.starmap(W.parzen_estimation_f32, items, 1)

    out = {"workload": "parzen_estimation: %d samples x %d dims (seed 123), %d widths, fp32 window test (BASELINE.json configs[2])"
                       % (n, xs.shape[1], len(widths))}
    for name, fn in (("apply_async_x102", job_apply), ("starmap_chunksize1", job_star)):
        for _ in range(2):
            res = fn()
        pool.reset_stats()
        t0 = time.perf_counter()
        for _ in range(steps):
            res = fn()
        dt = (time.perf_counter() - t0) / steps
        st = pool.stats()
        out[name] = {"ms_per_job": 1e3 * dt, "tasks_per_s": len(widths) / dt, "kernel_launches_per_job": st["dispatch_launches"] / steps,
                     "kernel_us_per_job": 1e3 * st["dispatch_ms"] / steps, "h2d_bytes_per_job": st["h2d_bytes"] // steps,
                     "d2h_bytes_per_job": st["d2h_bytes"] // steps}
    star = np.asarray(res)
    # parity: k_n vs the CPU fp32 restatement (exact) and vs fp64 (boundary samples only), density rtol 1e-6
    mism, ok = 0, True
    for (h, dens), w in zip(star.tolist(), widths):
        k_gpu = int(round(dens * h * n))
        k32 = cref.parzen_count(xs, px, w, np.float32)
        k64 = cref.parzen_count(xs, px, w, np.float64)
        ok &= (h == w) and (k_gpu == k32) and abs(k_gpu - k64) <= B.parzen_boundary_count(xs, px, w)
        if k_gpu == k64:
            want = (k64 / n) / h
            ok &= abs(dens - want) <= 1e-6 * abs(want)
        else:
            mism += 1
    f64 = pool.starmap(W.parzen_estimation, items, 1)
    ok64 = all((k == cref.parzen_count(xs, px, w, np.float64)) for (h, d), w, k in
               zip(f64.tolist(), widths, [int(round(d * h * n)) for h, d in f64.tolist()]))
    kern_us = out["starmap_chunksize1"]["kernel_us_per_job"]
    l2_bytes = len(widths) * n * xs.shape[1] * 4
    tr = traffic.get("dispatch_parzen_kernel<float>@prof_parzen", {})
    out.update({
        "value": out["starmap_chunksize1"]["tasks_per_s"], "unit": "tasks/s",
        "parity": {"k_n_equals_fp32_oracle_and_within_boundary_of_fp64": bool(ok), "fp32_vs_fp64_k_n_mismatches": mism,
                   "tolerance": "k_gpu == k_cpu(fp32) exactly; may differ from fp64 only on samples with ||x|/h - 0.5| <= 2^-22*max(1,|x|/h); "
                                "density rtol 1e-6 when k matches", "parzen_f64_k_n_bit_exact": bool(ok64)},
        "roofline": {"kernel": "dispatch_parzen_kernel<float> (one CTA per width, samples re-read from L2)", "bound": "l2",
                     "achieved": l2_bytes / (kern_us * 1e-6) / 1e9 if kern_us else None, "unit": "GB/s",
                     "algorithmic_bytes_per_launch": l2_bytes, "avg_launch_us": kern_us,
                     "lts_pct_of_peak": tr.get("lts_pct_of_peak"), "traffic": tr.get("dram_bytes_per_launch"),
                     "note": "102 CTAs x 80 KB from L2 = 8.2 MB per launch: the launch is latency-bound (a few us), far below any "
                             "bandwidth roof; lts_pct_of_peak comes from the committed ncu capture"},
    })
    pool.terminate()
    pool.join()
    if with_cpu:
        try:
            res_c, kind = cpu_arm("parzen", os.cpu_count() or 1, reps=2, timeout=300)
            best = min(res_c["times"])
            out["cpu_baseline"] = {"value": len(widths) / best, "unit": "tasks/s", "ms_per_job": 1e3 * best, "cores": os.cpu_count() or 1,
                                   "kind": kind, "impl": res_c.get("impl"),
                                   "sample": "best of 2: 102 apply_async calls of the reference's parzen_estimation (Python loops over "
                                             "10 000 samples, float64) through Pool(processes=%d), as examples/parzen_estimation.py:22-28" % (os.cpu_count() or 1),
                                   "first_result": res_c.get("first")}
        except Exception as e:      # noqa: BLE001
            out["cpu_baseline"] = {"unavailable": str(e)[:200]}
    return out


# ------------------------------------------------------------------------------------------------
def cref_count_first_1e6(first):
    """Oracle count of is_inside over [first, first + 1e6) (checker only)."""
    from oracle import cref
    return cref.pi_inside_range(first, 10 ** 6, want_array=False)[1]


def run_ours(args, dist):
    import numpy as np
    import fiber_b200
    from fiber_b200 import _abi
    from examples import workloads as W   # user-side function definitions bound to device bodies

    peaks, peak_src = load_peaks()
    hbm_peak = float(peaks["hbm_gbs"])
    traffic, traffic_src = load_traffic()
    traffic_commit = traffic.get("_meta", {}).get("commit")
    # is the committed ncu capture from the very sources being timed?  (nvcc output is not bit-reproducible, so the
    # build is identified by the digest of its sources, written by profiles/run_ncu.sh next to the captures)
    traffic_same_build = source_digest() == traffic.get("_meta", {}).get("src_sha256")

    def traffic_of(key):
        return traffic.get(key, {}).get("dram_bytes_per_launch")
    dev = dist.local_rank
    rank, world = dist.rank, dist.world
    my_first = rank * PI_TASKS

    clocks = ClockSampler(dev)
    if rank == 0:
        clocks.start()

    # ---------------- value: device-resident, raw C ABI ------------------------------------------
    eng = RawEngine(dev, 160 << 20)                       # (ring only used by the via-ring leg below)
    out_dev = eng.dalloc(PI_TASKS)
    pending = []
    leg = {"flags": 0, "seed": 1}

    def pi_step():
        leg["seed"] += 1
        pending.append(eng.submit("pi_inside_det", PI_TASKS, out_dev, index_start=my_first, task_base=my_first,
                                  extra_flags=leg["flags"], seed=leg["seed"]))

    counts = []

    def pi_drain():
        while pending:
            c, _ = eng.wait(pending.pop(0), release=False)   # the step's count is in hand here
            counts.append(c)

    # warm-up outside the stats window
    for _ in range(max(args.warmup, 3)):
        pi_step()
    pi_drain()
    eng.release_deferred()
    eng.stats(reset=True)
    t_value = timed_steps(dist, args.steps, 0, pi_step, pi_drain, clocks.windows)
    eng.release_deferred()
    st = eng.stats()
    my_count = counts[-1]
    total_count = dist.sum_i64(my_count)
    value = world * PI_TASKS * args.steps / t_value
    launches_value = st["dispatch_launches"] + st["gather_launches"]
    dispatch_ms = st["dispatch_ms"] / max(1, st["dispatch_launches"])
    # FULL parity of the device-resident ordered output of the last timed step (outside the timed loop)
    value_out = eng.d2h(out_dev, PI_TASKS)
    value_parity = dist.all_true(oracle_pi_equal(value_out, my_first))
    if args.dump_outputs:
        dump_pi_outputs(args.dump_outputs, value_out, my_first, total_count, dist)
    del value_out

    # ---- the gather leg: same map, task records shuffled inside each wave -> records + ring + gather_ordered
    leg["flags"] = _abi.FBR_SHUFFLE
    for _ in range(3):
        pi_step()
    pi_drain()
    eng.release_deferred()
    eng.stats(reset=True)
    t_ring = timed_steps(dist, args.steps, 0, pi_step, pi_drain, clocks.windows)
    eng.release_deferred()
    sr = eng.stats()
    ring_parity = dist.all_true(oracle_pi_equal(eng.d2h(out_dev, PI_TASKS), my_first) and counts[-1] == my_count)
    launches_ring = sr["dispatch_launches"] + sr["gather_launches"]
    gather_ms = sr["gather_ms"] / max(1, sr["gather_launches"])
    gather_bytes = sr["gather_bytes"] / max(1, sr["gather_launches"])
    roofline = {"kernel": "gather_rows_kernel (gather_ordered, 4 KB-row path; placement by index under shuffled arrival)", "bound": "hbm",
                "achieved": gather_bytes / (gather_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                "frac": gather_bytes / (gather_ms * 1e-3) / 1e9 / hbm_peak,
                "traffic": traffic_of("gather_rows_kernel@prof_pi"), "traffic_source": traffic_src, "traffic_capture_commit": traffic_commit,
                "traffic_capture_is_this_build": traffic_same_build,
                "peak_source": peak_src,
                "algorithmic_bytes_per_launch": gather_bytes, "avg_launch_ms": gather_ms,
                "step_ms_via_ring": 1e3 * t_ring / args.steps, "tasks_per_s_via_ring": world * PI_TASKS * args.steps / t_ring,
                "parity_full": ring_parity,
                "note": "2*R*N bytes (R=1 B) per launch, 1e8 tasks; the ring (100 MB) was just written by the dispatch kernel, so part "
                        "of it is still in the 126 MB L2 (`traffic` = DRAM bytes of the cold ncu capture); the DRAM-clean figures are "
                        "payload4k.roofline_dispatch / roofline_gather (8.2 GB per launch).  The headline `value` step does not "
                        "launch this kernel: a contiguous map is placed by the dispatch kernel itself"}
    # Philox4x32-10 + circle test: the bound is the SM's integer-multiply pipe (IMAD.WIDE.U32), not HBM
    # (1 B written per task).  Its peak is measured, not nominal: profiles/microbench/imad_peak.cu.
    wide_per_task = 18
    imad = load_imad_peak()
    wide_rate = wide_per_task * PI_TASKS / (dispatch_ms * 1e-3)
    roofline_dispatch = {"kernel": "dispatch_thread_kernel<PiInsideDet, index args> (+ sum fold, direct placement)", "bound": "alu (IMAD.WIDE.U32 pipe)",
                         "avg_launch_ms": dispatch_ms, "tasks_per_s": PI_TASKS / (dispatch_ms * 1e-3),
                         "hbm_gbs": PI_TASKS * 1 / (dispatch_ms * 1e-3) / 1e9,
                         "imad_wide_per_task": wide_per_task,
                         "achieved": wide_rate / 1e9, "peak": imad.get("gops"), "unit": "G IMAD.WIDE.U32/s",
                         "frac": (wide_rate / 1e9 / imad["gops"]) if imad.get("gops") else None,
                         "peak_source": imad.get("source"),
                         "note": "Philox4x32-10 on a (lo, hi, 0, 0) counter: 18 32x32->64 multiplies per task (round 1 has a "
                                 "zero word, round 2's M0*(hi^key) is shared by 16 tasks); circle test screened in fp32, "
                                 "float64 only within 2^-19 of the circle; the same body alone (no ring traffic) reaches "
                                 "%s tasks/s in the microbenchmark" % imad.get("pi_body_screened_tasks_per_s")}
    eng.dfree(out_dev)

    # ---------------- secondary: 4 KB payload map, device resident ----------------------------------
    payload = None
    launches_payload = 0
    if not args.skip_payload:
        eng.close()
        eng = RawEngine(dev, PAYLOAD_TASKS * 4096 + (1 << 20))
        t_base = rank * PAYLOAD_TASKS
        in_dev = eng.dalloc(PAYLOAD_TASKS * 4096)
        out2 = eng.dalloc(PAYLOAD_TASKS * 4096)
        _abi.check(eng.lib.fbr_payload_fill_device(eng.h, 0, in_dev, t_base, PAYLOAD_TASKS))
        pend2 = []
        pleg = {"flags": 0}

        def pl_step():
            pend2.append(eng.submit("payload_map_4k", PAYLOAD_TASKS, out2, args_dev=in_dev, arg_stride=4096,
                                    task_base=t_base, want_sum=False, extra_flags=pleg["flags"]))

        def pl_drain():
            while pend2:
                eng.wait(pend2.pop(0), release=False)
        for _ in range(3):
            pl_step()
        pl_drain()
        eng.release_deferred()
        eng.stats(reset=True)
        t_pl = timed_steps(dist, args.steps, 0, pl_step, pl_drain, clocks.windows)
        eng.release_deferred()
        sp = eng.stats()
        launches_payload = sp["dispatch_launches"] + sp["gather_launches"]
        d_ms = sp["dispatch_ms"] / max(1, sp["dispatch_launches"])
        d_bytes = sp["dispatch_bytes"] / max(1, sp["dispatch_launches"])
        # FULL parity of the last step's output against the C oracle (4.1 GB, outside the timed loop)
        got = eng.d2h(out2, PAYLOAD_TASKS * 4096).view(np.uint32).reshape(PAYLOAD_TASKS, 1024)
        ok = dist.all_true(oracle_payload_equal(got, t_base))
        del got
        # via-ring leg: the same map through task records + ring + gather_bulk (TMA), for the gather's HBM roofline
        pleg["flags"] = _abi.FBR_VIA_RING
        for _ in range(2):
            pl_step()
        pl_drain()
        eng.release_deferred()
        eng.stats(reset=True)
        k_ring = args.steps
        t_plr = timed_steps(dist, k_ring, 0, pl_step, pl_drain, clocks.windows)
        eng.release_deferred()
        spr = eng.stats()
        launches_payload += spr["dispatch_launches"] + spr["gather_launches"]
        g_ms = spr["gather_ms"] / max(1, spr["gather_launches"])
        g_bytes = spr["gather_bytes"] / max(1, spr["gather_launches"])
        host = eng.d2h(out2, 64 * 4096).view(np.uint32).reshape(64, 1024)
        from oracle import cref
        ok_ring = bool(np.array_equal(host, cref.payload_map(t_base, cref.payload_records(t_base, 64))))
        payload = {
            "workload": "synthetic 4 KB-payload map, %d tasks per GPU, inputs+outputs resident in HBM (4.1 GB each, >> L2)" % PAYLOAD_TASKS,
            "value": world * PAYLOAD_TASKS * args.steps / t_pl, "unit": "tasks/s", "ms_per_step": 1e3 * t_pl / args.steps,
            "roofline_dispatch": {"kernel": "dispatch_payload_map_tma_kernel (TMA-staged, warp-specialised, direct placement)", "bound": "hbm",
                                  "achieved": d_bytes / (d_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                  "frac": d_bytes / (d_ms * 1e-3) / 1e9 / hbm_peak, "avg_launch_ms": d_ms,
                                  "algorithmic_bytes_per_launch": d_bytes,
                                  "traffic": traffic_of("dispatch_payload_map_tma_kernel@prof_payload"), "traffic_capture_commit": traffic_commit},
            "roofline_gather": {"kernel": "gather_bulk_kernel (gather_ordered, TMA cp.async.bulk path; FBR_VIA_RING leg)", "bound": "hbm",
                                "achieved": g_bytes / (g_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                "frac": g_bytes / (g_ms * 1e-3) / 1e9 / hbm_peak, "avg_launch_ms": g_ms,
                                "algorithmic_bytes_per_launch": g_bytes, "step_ms_via_ring": 1e3 * t_plr / k_ring,
                                "traffic": traffic_of("gather_bulk_kernel@prof_payload"), "traffic_capture_commit": traffic_commit},
            "parity_full": ok, "checked_bytes": PAYLOAD_TASKS * 4096, "parity_spot_check_via_ring": ok_ring,
        }
        eng.dfree(in_dev)
        eng.dfree(out2)
    eng.close()

    # ---------------- N > 1: the sharded 4 KB map (config 4) and the ring all-reduce (config 5) ---------
    multi = None
    if world > 1 and not args.skip_payload:
        multi = run_multi_gpu(args, dist, dev)

    # ---------------- e2e: the public API with host buffers ---------------------------------------------
    pool = fiber_b200.Pool(1, devices=[dev], timing=False, bind_cpu=world > 1)   # N>1: NUMA-local pinned segments
    my_range = range(my_first, my_first + PI_TASKS)
    e2e_counts = []

    fold = {"local": []}

    def fold_count(c, sink):
        """Every step's own count is in hand on the host when the step ends; the job-wide counts of the K steps are
        folded by ONE ncclAllReduce(sum, int64[K]) when the region drains (inside the timed region).  A collective
        per step would make every rank wait for the slowest one K times for 8 bytes each -- measured at N=8: the
        per-step fold, even started asynchronously, stretched a 0.27 ms step to 0.96 ms -- while the map itself needs
        no data-path collective at all."""
        if world == 1:
            sink.append(c)
        else:
            fold["local"].append(c)

    def fold_drain(sink):
        if fold["local"]:
            sink.extend(dist.sum_i64_vector(fold["local"]))
            fold["local"] = []

    def e2e_step():
        res = pool.map(W.is_inside, my_range)             # blocks until the pinned result segment is final
        fold_count(res.sum(), e2e_counts)                 # count folded on the device, read on the host
        e2e_step.last = res

    for _ in range(max(args.warmup, 3)):
        e2e_step()
    fold_drain(e2e_counts)
    pool.reset_stats()
    t_e2e = timed_steps(dist, args.steps, 0, e2e_step, lambda: fold_drain(e2e_counts), clocks.windows)
    se = pool.stats()
    e2e_value = world * PI_TASKS * args.steps / t_e2e
    packed = e2e_step.last.packed
    e2e_parity = dist.all_true(oracle_pi_equal(np.unpackbits(packed, count=PI_TASKS, bitorder="little"), my_first))
    e2e = {"value": e2e_value, "unit": "tasks/s", "ms_per_step": 1e3 * t_e2e / args.steps,
           "h2d_bytes_per_step": se["h2d_bytes"] // args.steps, "d2h_bytes_per_step": se["d2h_bytes"] // args.steps,
           "api": "fiber_b200.Pool(1).map(is_inside_det, range(1e8)) -> pinned ResultArray (bool results one bit each, the default layout) + count",
           "packed_bytes": int(packed.nbytes), "parity_full": e2e_parity,
           "cpu_binding": ("%d GPU-local CPUs" % len(pool.bound_cpus)) if pool.bound_cpus else "none"}
    launches_e2e = se["dispatch_launches"] + se["gather_launches"]
    e2e_step.last = None
    del packed

    # secondary e2e: the same maps through map_async with two in flight (a user loop that submits step k+1 before it
    # reads step k): every step's bit-packed results still land in the pinned segment and its count is read on the host
    pipe_counts, inflight = [], []

    def e2e_pipe_step():
        inflight.append(pool.map_async(W.is_inside, my_range))
        if len(inflight) > 1:
            fold_count(inflight.pop(0).get().sum(), pipe_counts)

    def e2e_pipe_drain():
        while inflight:
            fold_count(inflight.pop(0).get().sum(), pipe_counts)
        fold_drain(pipe_counts)

    for _ in range(3):
        e2e_pipe_step()
    e2e_pipe_drain()
    pool.reset_stats()
    t_e2e_pipe = timed_steps(dist, args.steps, 0, e2e_pipe_step, e2e_pipe_drain, clocks.windows)
    sp_ = pool.stats()
    e2e["pipelined_map_async"] = {"value": world * PI_TASKS * args.steps / t_e2e_pipe, "unit": "tasks/s", "ms_per_step": 1e3 * t_e2e_pipe / args.steps,
                                  "d2h_bytes_per_step": sp_["d2h_bytes"] // args.steps, "count": pipe_counts[-1],
                                  "api": "fiber_b200.Pool(1).map_async(is_inside_det, range(1e8)) with two maps in flight, .get().sum() per step",
                                  "note": "secondary figure: the blocking Pool.map above is the headline"}
    launches_e2e += sp_["dispatch_launches"] + sp_["gather_launches"]

    # e2e of the 4 KB payload map: records in pinned host memory -> H2D -> map -> D2H (PCIe-bound)
    if payload is not None:
        from oracle import cref
        n_pl = PAYLOAD_TASKS
        recs = pool.pinned_empty((n_pl, 1024), np.uint32)
        # synthetic inputs: generated by the engine's fill kernel, copied into the pinned host array
        eng_l, eng_h = pool._engine.lib, pool._engine.handle
        tmp = ctypes.c_void_p()
        _abi.check(eng_l.fbr_device_alloc(eng_h, 0, recs.nbytes, ctypes.byref(tmp)))
        _abi.check(eng_l.fbr_payload_fill_device(eng_h, 0, tmp, rank * n_pl, n_pl))
        _abi.check(eng_l.fbr_memcpy_d2h(eng_h, 0, recs.ctypes.data, tmp, recs.nbytes))
        _abi.check(eng_l.fbr_device_free(eng_h, 0, tmp))

        def pl_e2e_step():
            r = pool.map(W.payload_map, recs)      # task t of the map is record t (t = row index)
            pl_e2e_step.last = r

        for _ in range(2):
            pl_e2e_step()
        pool.reset_stats()
        k_pl = args.steps
        t_pl_e2e = timed_steps(dist, k_pl, 0, pl_e2e_step, None, clocks.windows)
        sp2 = pool.stats()
        got = np.asarray(pl_e2e_step.last)
        ok2 = bool(np.array_equal(got[:32], cref.payload_map(0, recs[:32]))) and \
            bool(np.array_equal(got[-32:], cref.payload_map(n_pl - 32, recs[-32:])))
        payload["e2e"] = {"value": world * n_pl * k_pl / t_pl_e2e, "unit": "tasks/s", "ms_per_step": 1e3 * t_pl_e2e / k_pl,
                          "h2d_bytes_per_step": sp2["h2d_bytes"] // k_pl, "d2h_bytes_per_step": sp2["d2h_bytes"] // k_pl,
                          "pcie_GBps_each_way": n_pl * 4096 / (t_pl_e2e / k_pl) / 1e9, "steps": k_pl, "parity_spot_check": ok2,
                          "api": "fiber_b200.Pool(1).map(payload_map, pinned (1e6,1024) uint32) -> pinned ResultArray"}
        launches_e2e += sp2["dispatch_launches"] + sp2["gather_launches"]
        del recs, got
        pl_e2e_step.last = None
    # secondary e2e: same call on Pool(results="device") -- ordered results stay in HBM, only the
    # count (control block) crosses PCIe, as in `4.0 * pool.map(...).sum() / N`
    dpool = fiber_b200.Pool(1, devices=[dev], results="device")
    dev_counts = []

    def e2e_dev_step():
        res = dpool.map(W.is_inside, my_range)
        fold_count(res.sum(), dev_counts)
        del res

    for _ in range(3):
        e2e_dev_step()
    fold_drain(dev_counts)
    dpool.reset_stats()
    t_e2e_dev = timed_steps(dist, args.steps, 0, e2e_dev_step, lambda: fold_drain(dev_counts), clocks.windows)
    sd = dpool.stats()
    e2e["results_on_device"] = {"value": world * PI_TASKS * args.steps / t_e2e_dev, "unit": "tasks/s",
                                "ms_per_step": 1e3 * t_e2e_dev / args.steps,
                                "h2d_bytes_per_step": sd["h2d_bytes"] // args.steps, "d2h_bytes_per_step": sd["d2h_bytes"] // args.steps + 32,
                                "api": "fiber_b200.Pool(1, results='device').map(is_inside_det, range(1e8)).sum()",
                                "count": dev_counts[-1],
                                "note": "secondary figure: results are fetched lazily, only the folded count is read on the host"}
    launches_e2e += sd["dispatch_launches"] + sd["gather_launches"]
    dpool.terminate()
    dpool.join()
    # secondary e2e: same call on Pool(results="bytes") -- one BYTE per bool through the ordered output and PCIe
    # (100 MB D2H per step: the PCIe floor of the byte layout)
    bpool = fiber_b200.Pool(1, devices=[dev], results="bytes", bind_cpu=world > 1)
    byte_counts = []

    def e2e_bytes_step():
        res = bpool.map(W.is_inside, my_range)
        fold_count(res.sum(), byte_counts)
        e2e_bytes_step.last = res

    for _ in range(3):
        e2e_bytes_step()
    fold_drain(byte_counts)
    bpool.reset_stats()
    t_e2e_bytes = timed_steps(dist, args.steps, 0, e2e_bytes_step, lambda: fold_drain(byte_counts), clocks.windows)
    sb = bpool.stats()
    arr = np.asarray(e2e_bytes_step.last).view(np.uint8)
    e2e["results_byte_per_bool"] = {"value": world * PI_TASKS * args.steps / t_e2e_bytes, "unit": "tasks/s",
                                    "ms_per_step": 1e3 * t_e2e_bytes / args.steps,
                                    "h2d_bytes_per_step": sb["h2d_bytes"] // args.steps, "d2h_bytes_per_step": sb["d2h_bytes"] // args.steps,
                                    "api": "fiber_b200.Pool(1, results='bytes').map(is_inside_det, range(1e8)) -> pinned uint8 ResultArray + count",
                                    "count": byte_counts[-1],
                                    "parity_spot_check": bool(int(arr[:10 ** 6].sum()) == cref_count_first_1e6(my_first)),
                                    "note": "secondary figure: the opt-out layout, one byte per bool (PCIe-bound: 100 MB per step)"}
    launches_e2e += sb["dispatch_launches"] + sb["gather_launches"]
    e2e_bytes_step.last = None
    del arr
    bpool.terminate()
    bpool.join()

    # T_list at 1e6: Python list in hand, the reference's own end point (SURVEY.md 8(d))
    t0 = time.perf_counter()
    lst = pool.map(W.is_inside, range(10 ** 6)).tolist()
    t_list = time.perf_counter() - t0
    assert len(lst) == 10 ** 6
    pool.terminate()
    pool.join()
    clk = clocks.stop() if rank == 0 else None

    # ---------------- parzen (config 3) and the CPU baseline (rank 0, N=1) -------------------------------------
    parzen = cpu = None
    if rank == 0 and not args.skip_parzen:
        parzen = run_parzen(dev, traffic, with_cpu=(world == 1 and not args.skip_cpu), steps=args.steps)
    if rank == 0 and world == 1 and not args.skip_cpu:
        cores = os.cpu_count() or 1
        try:
            res_c, kind = cpu_arm("pi", cores, reps=3, warm=1)
            best = min(res_c["times"])
            cpu = {"value": CPU_SAMPLE_TASKS / best, "unit": "tasks/s", "cores": cores, "kind": kind, "impl": res_c.get("impl"),
                   "sample": "best of 3 Pool(processes=%d).map over %d pi_inside_det tasks (C body via ctypes), default chunksize 32, "
                             "after a 1000-task warm-up map" % (cores, CPU_SAMPLE_TASKS),
                   "mean_tasks_per_s": CPU_SAMPLE_TASKS * len(res_c["times"]) / sum(res_c["times"]),
                   "count_matches_oracle": res_c["count"] == cref_count_first_1e6(0)}
        except Exception as e:      # noqa: BLE001 -- the GPU line must not be lost to a hiccup of the CPU arm
            cpu = {"value": None, "unit": "tasks/s", "cores": cores, "kind": "unavailable", "sample": str(e)[:300]}
        try:
            if cpu["value"] is None:
                raise RuntimeError("CPU arm unavailable")
            r4, k4 = cpu_arm("pi", 4, reps=2, warm=0)
            cpu["pool4"] = {"value": CPU_SAMPLE_TASKS / min(r4["times"]), "unit": "tasks/s", "cores": 4, "kind": k4,
                            "sample": "best of 2 Pool(4).map over %d tasks (examples/pi_estimation.py:15, BASELINE.json configs[0])" % CPU_SAMPLE_TASKS}
        except Exception as e:      # noqa: BLE001
            cpu["pool4"] = {"unavailable": str(e)[:200]}

    if rank == 0:
        line = {
            "metric": "pool_map_tasks_per_sec", "value": value, "unit": "tasks/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": 1e3 * t_value / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64->u8", "data": "synthetic",
            "config": {"workload": "pi_estimation Pool.map over 1e8 index tasks per GPU (BASELINE.json configs[1]), ordered uint8 results + int64 count",
                       "tasks_per_gpu": PI_TASKS, "chunksize": 32, "parallelism": "index blocks per rank, no data-path collective",
                       "l2": "ordered output (100 MB per step) + the via-ring leg's result ring (100 MB) exceed the 126 MB L2; payload4k streams 8.2 GB per step",
                       "cpu_arm_sample_tasks": CPU_SAMPLE_TASKS},
            "e2e": e2e, "gpu_launches": int(launches_value + launches_ring + launches_payload + launches_e2e),
            "gpu_launches_detail": {"pi_value_per_step": launches_value / args.steps, "pi_via_ring_per_step": launches_ring / args.steps,
                                    "payload_total": launches_payload, "e2e_paths_total": launches_e2e,
                                    "note": "dispatch + gather launches of this repo's kernels inside the timed regions"},
            "parity_full": {"value_leg": value_parity, "via_ring_leg": ring_parity, "e2e": e2e_parity,
                            "payload4k": payload["parity_full"] if payload else None,
                            "note": "every byte/bit of the last timed step's output compared with the C oracle, outside the timed loops"},
            "roofline": roofline, "roofline_dispatch": roofline_dispatch, "payload4k": payload, "parzen": parzen,
            "multi_gpu": multi, "cpu_baseline": cpu, "clocks": clk,
            "check": {"pi_count_all_ranks": total_count, "pi_estimate": 4.0 * total_count / (world * PI_TASKS),
                      "e2e_count": e2e_counts[-1]},
            "t_list_1e6": {"tasks_per_s": 1e6 / t_list, "note": "Pool.map(...).tolist(): Python list in hand at 1e6 tasks"},
        }
        print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of every GPU leg (the CPU baseline arms keep their own fixed repetitions)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--skip-payload", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-parzen", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the headline map's last timed step (sampled results, block counts, count) as DIR/<name>.npy")
    ap.add_argument("--cpu-child", default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.cpu_child:
        _cpu_child(json.loads(args.cpu_child))
        return 0
    if args.impl == "reference":
        rank = int(os.environ.get("RANK", "0"))
        if rank != 0:
            return 0        # other ranks exit without work
        dist = type("D", (), {"rank": 0, "world": 1, "local_rank": 0})()
        run_reference(args, dist)
        return 0
    dist = Dist(args.gpus)
    try:
        run_ours(args, dist)
    finally:
        dist.finish()
    return 0


if __name__ == "__main__":
    sys.exit(main())
