"""Time the simulation of retirement2_smooth with modal choices against choice draws (egdst_solution_set_choice_draws):
sims+moments and moments only, the same solution, agents and Philox seed, the two modes alternating (CUDA events).

    python tools/sim_choice_time.py [nsim (default 4000000)] [rounds (default 3)]
"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from egdst_b200 import capi, examples  # noqa: E402

nsim = int(sys.argv[1]) if len(sys.argv) > 1 else 4_000_000
rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 3
reps = 5
m = examples.retirement2_smooth()
m.compile()
lib = m._capi()
sol = lib.solve(m, strict=True)
dev = torch.device("cuda", 0)
try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True).stdout.strip()
except OSError:
    q = "%s, power limit not readable" % torch.cuda.get_device_name(dev)
print("card: %s" % q)
nt, nso = m.nt, m.nsimout()
print("retirement2_smooth: sigma_eps %g, nt %d, nd %d, nsimout %d, %d agents, %d launches per timing" % (m.sigma_eps, nt, m.nd, nso, nsim, reps))
d_init = torch.empty(2 * nsim, dtype=torch.float64, device=dev)
d_init[:nsim] = 1.0
d_init[nsim:] = m.a0 + 0.5 * (m.mmax - m.a0) * torch.rand(nsim, dtype=torch.float64, device=dev, generator=torch.Generator(device=dev).manual_seed(1))
d_sims = torch.empty(nso * nt * nsim, dtype=torch.float64, device=dev)
d_mom = torch.zeros(3 * nso * nt, dtype=torch.float64, device=dev)
desc = capi.Desc(m)


def run(ps, pm):
    lib.simulate_device(m, sol, d_init.data_ptr(), nsim, 0, 12345, ps, pm, desc=desc)


times = {}
for label, ps, pm in (("sims+moments", d_sims.data_ptr(), d_mom.data_ptr()), ("moments only", 0, d_mom.data_ptr())):
    for draws in (False, True):  # warm-up of both instantiations
        sol.set_choice_draws(draws)
        run(ps, pm)
    torch.cuda.synchronize()
    for _ in range(rounds):
        for draws in (False, True):
            sol.set_choice_draws(draws)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                run(ps, pm)
            e1.record()
            torch.cuda.synchronize()
            times.setdefault((label, draws), []).append(e0.elapsed_time(e1) / reps)
sol.set_choice_draws(False)
for label in ("sims+moments", "moments only"):
    mo, dr = times[(label, False)], times[(label, True)]
    print("%-13s modal %s ms   draws %s ms   draws/modal %.2f (medians)" % (
        label, " ".join("%7.2f" % t for t in mo), " ".join("%7.2f" % t for t in dr), sorted(dr)[len(dr) // 2] / sorted(mo)[len(mo) // 2]))
