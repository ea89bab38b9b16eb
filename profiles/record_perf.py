"""Record-body dispatch kernels on one GPU (dispatch_record_kernel against dispatch_thread_kernel).

Times the dispatch kernel alone: the C ABI (bench.RawEngine), FBR_POOL_TIMING events around each launch, arguments
and output resident on the device (FBR_ARGS_DEVICE | FBR_OUT_DEVICE: one direct wave, no copy), warm-up excluded.
About 1e8 tasks per map (2e7 for the 256 B records), so every working set is far beyond the 126 MB L2.  Twins that
compute the same function through the two kernels are alternated in the same process.  The denominator of the
"copy fraction" is a device-to-device copy moving the same algorithmic bytes, timed in the same run.

    python profiles/record_perf.py [--out profiles/record_perf_b200.json] [--reps 7]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# (body, tasks); twins are listed next to each other and timed alternately
CASES = [
    [("poly_f64_thread", 10 ** 8), ("poly_f64", 10 ** 8), ("poly_f64_staged", 10 ** 8)],   # 1. f64 -> f64
    [("dot_w64_thread", 10 ** 8), ("dot_w64", 10 ** 8), ("stats_w64", 10 ** 8)],   # 2. 64 B -> f64 / 16 B
    [("affine_f3", 10 ** 8)],                                              # 3. float3 -> float3
    [("mix_256", 2 * 10 ** 7)],                                            # 4. 256 B -> 256 B
]


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # noqa: BLE001 -- recorded, not fatal
        return {"name": "unknown", "error": str(e)}


def copy_rate(torch, nbytes, reps):
    """GB/s of algorithmic bytes (read + written) of a device-to-device copy moving `nbytes` of them in all."""
    half = nbytes // 2
    src = torch.empty(half, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)
    src.fill_(7)
    dst.copy_(src)
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        dst.copy_(src)
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    ms = ts[len(ts) // 2]
    del src, dst
    return 2 * half / (ms * 1e-3) / 1e9, ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "record_perf_b200.json"))
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()

    import torch
    import bench
    from fiber_b200 import registry
    from tests import record_bodies  # noqa: F401 -- registers the bodies

    eng = bench.RawEngine(0, 0)
    rows = []
    for group in CASES:
        bufs = {}
        for body, n in group:
            s = registry.spec(body)
            base = s._leaves[0][1]                         # the records' scalar type: real values of it
            if base.kind == "f":
                tdt = torch.float32 if base.itemsize == 4 else torch.float64
                a = torch.empty(n * s.arg_bytes // base.itemsize, dtype=tdt, device="cuda").normal_()
            else:
                a = torch.empty(n * s.arg_bytes // 4, dtype=torch.int32, device="cuda").random_(-2 ** 31, 2 ** 31 - 1)
            bufs[body] = (a, torch.empty(n * s.result_bytes, dtype=torch.uint8, device="cuda"), s, n)
        times = {b: [] for b in bufs}
        for rep in range(args.reps + 1):                  # rep 0 is the warm-up
            for body, (a, out, s, n) in bufs.items():
                eng.stats(reset=True)
                seq = eng.submit(body, n, out.data_ptr(), args_dev=a.data_ptr(), arg_stride=s.arg_bytes, want_sum=False)
                eng.wait(seq)
                st = eng.stats(reset=True)
                assert st["dispatch_launches"] == 1 and st["gather_launches"] == 0, st
                if rep:
                    times[body].append(st["dispatch_ms"])
        for body, (a, out, s, n) in bufs.items():
            ts = sorted(times[body])
            ms = ts[len(ts) // 2]
            nbytes = (s.arg_bytes + s.result_bytes) * n
            cgbs, cms = copy_rate(torch, nbytes, args.reps)
            gbs = nbytes / (ms * 1e-3) / 1e9
            # FBR_EXPORT_RECORD_BODY runs 8 B -> 8 B records one thread per record; poly_f64_staged forces the staged kernel
            kernel = "thread" if body.endswith("_thread") or (s.flags & 0x10 and s.arg_bytes == s.result_bytes == 8
                                                              and not body.endswith("_staged")) else "record (staged)"
            rows.append({"body": body, "export": "record" if s.flags & 0x10 else "thread", "kernel": kernel,
                         "arg_bytes": s.arg_bytes,
                         "result_bytes": s.result_bytes, "tasks": n, "kernel_ms_median": round(ms, 4),
                         "kernel_ms_min": round(ts[0], 4), "kernel_ms_max": round(ts[-1], 4), "bytes": nbytes,
                         "GBps": round(gbs, 1), "copy_GBps": round(cgbs, 1), "copy_fraction": round(gbs / cgbs, 3)})
            print(json.dumps(rows[-1]), flush=True)
        del bufs
        torch.cuda.empty_cache()
    res = {"gpu": gpu_info(), "method": "C ABI, FBR_POOL_TIMING events, FBR_ARGS_DEVICE | FBR_OUT_DEVICE (one direct wave), "
           "median of %d maps after one warm-up; copy = torch device-to-device copy of the same algorithmic bytes" % args.reps,
           "rows": rows}
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res["gpu"]))


if __name__ == "__main__":
    main()
