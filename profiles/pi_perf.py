"""Event-timed pi dispatch / gather kernels only.

    python profiles/pi_perf.py [steps] [pi_inside_det|pi_inside_bits8]
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

steps = int(sys.argv[1]) if len(sys.argv) > 1 else 20
body = sys.argv[2] if len(sys.argv) > 2 else "pi_inside_det"
n = bench.PI_TASKS if body == "pi_inside_det" else bench.PI_TASKS // 8     # bits8: one task = 8 indices = 1 byte
eng = bench.RawEngine(0, 160 << 20)
out = eng.dalloc(n)
cnt = None
for i in range(steps + 3):
    if i == 3:
        eng.stats(reset=True)
    cnt = eng.wait(eng.submit(body, n, out))[0]
st = eng.stats()
print("%s  dispatch %.4f ms  gather %.4f ms  count %d" % (
    body, st["dispatch_ms"] / st["dispatch_launches"], st["gather_ms"] / max(1, st["gather_launches"]), cnt), flush=True)   # direct placement: no gather
eng.dfree(out)
eng.close()
