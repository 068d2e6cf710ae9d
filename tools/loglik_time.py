"""Time the choice log-likelihood (egdst_choice_loglik_device) of retirement2_smooth at its defaults: a panel from a
Philox draw simulation, evaluated for nvec = 1 and 64 parameter vectors, once in agent-major row order and once sorted
by (age, state), with warm-up (CUDA events).

    python tools/loglik_time.py [agents (default 200000)] [reps (default 20)]
"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from egdst_b200 import capi, examples  # noqa: E402

nsim = int(sys.argv[1]) if len(sys.argv) > 1 else 200_000
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 20
m = examples.retirement2_smooth()
m.compile()
lib = m._capi()
dev = torch.device("cuda", 0)
try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True).stdout.strip()
except OSError:
    q = "%s, power limit not readable" % torch.cuda.get_device_name(dev)
print("card: %s" % q)
names = [p["ref"] for p in m.param]
pv = np.array([list(m.param_vector())] * 64)
pv[:, names.index("duw")] *= 1.0 + 0.01 * (np.arange(64) - 32)
sol = lib.solve_batch(m, pv)
rng = np.random.default_rng(1)
init = np.column_stack([np.ones(nsim), m.a0 + 0.6 * (m.mmax - m.a0) * rng.random(nsim)])
sol.set_choice_draws(True)
sims, _ = lib.simulate_philox(m, sol, init, seed=12345, ivec=32)
sol.set_choice_draws(False)
obs = capi.observations_from_sims(m, sims)
nobs, k = obs.shape
print("retirement2_smooth: sigma_eps %g, nt %d, nd %d, %d agents, %d observations (k = %d), %d launches per timing" % (
    m.sigma_eps, m.nt, m.nd, nsim, nobs, k, reps))
orders = {"agent-major": obs, "sorted by (age, state)": obs[np.lexsort((obs[:, 1], obs[:, 0]))]}
desc = capi.Desc(m)
d_tot = torch.zeros(64, dtype=torch.float64, device=dev)
for label, o in orders.items():
    d_obs = torch.from_numpy(np.ascontiguousarray(o.ravel(order="F"))).to(dev)
    for nvec in (1, 64):
        def run():
            lib.choice_loglik_device(m, sol, d_obs.data_ptr(), nobs, k, d_tot.data_ptr(), sigma_c=0.1, ivec0=0, nvec=nvec, desc=desc)
        for _ in range(3):
            run()
        torch.cuda.synchronize()
        ts = []
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                run()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) / reps)
        med = sorted(ts)[1]
        print("%-24s nvec %2d: %s ms per call (median %.3f ms), %.3g rows x vectors per second" % (
            label, nvec, " ".join("%.3f" % t for t in ts), med, nobs * nvec / (med * 1e-3)))
