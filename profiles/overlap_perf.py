"""Pipelined pi steps with FBR_POOL_OVERLAP (gather(k) on a second stream while dispatch(k+1) runs)."""
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from fiber_b200 import _abi  # noqa: E402

steps = int(sys.argv[1]) if len(sys.argv) > 1 else 30
e2 = bench.RawEngine(0, 320 << 20, _abi.FBR_POOL_OVERLAP)
o2 = e2.dalloc(bench.PI_TASKS)
for _ in range(3):
    e2.wait(e2.submit("pi_inside_det", bench.PI_TASKS, o2))
t0 = time.perf_counter()
seqs = [e2.submit("pi_inside_det", bench.PI_TASKS, o2) for _ in range(steps)]
cnt = [e2.wait(q)[0] for q in seqs]
dt = (time.perf_counter() - t0) / steps
print("overlap  %.4f ms/step  count %d" % (dt * 1e3, cnt[-1]), flush=True)
e2.dfree(o2)
e2.close()
