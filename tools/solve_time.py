"""Time the S1 solve (resolve, CUDA-synchronised wall clock) and print the per-kernel-class device time."""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
from egdst_b200 import examples

kw = {}
for a in sys.argv[1:]:
    k, v = a.split("="); kw[k] = float(v) if "." in v else int(v)
m = examples.retirement2_scaled(**kw); m.compile()
lib = m._capi()
stream = torch.cuda.Stream(); torch.cuda.set_stream(stream); lib.set_stream(stream.cuda_stream)
sol = lib.solve(m, strict=True)
for _ in range(3):
    lib.resolve(sol, m)
torch.cuda.synchronize()
t = time.perf_counter()
for _ in range(10):
    lib.resolve(sol, m)
torch.cuda.synchronize()
ms = (time.perf_counter() - t) / 10 * 1e3
print("solve %.3f ms  status %s  units %d" % (ms, sol.status(), sol.units()))
lib.profile_enable(True)
for _ in range(3):
    lib.resolve(sol, m)
torch.cuda.synchronize()
prof = lib.profile_read(); lib.profile_enable(False)
for k, (t_ms, n) in prof.items():
    if n:
        print("  %-10s %8.3f ms/solve  %6.1f us/launch  (%d launches/solve)" % (k, t_ms / 3, t_ms / n * 1e3, n // 3))
ph = sol.phase_ms()
for k, v in ph.items():
    print("  phase %-10s %8.3f ms/solve  %6.1f us/period" % (k, v / 3, v / 3 / max(m.nt - 1, 1) * 1e3))
print("  resends handled:", sol.resends())
