"""Time the choice log-likelihood (egdst_choice_loglik_device) of retirement2_smooth at its defaults: a panel from a
Philox draw simulation, evaluated for nvec = 1 and 64 parameter vectors, once in agent-major row order and once sorted
by (age, state), with warm-up (CUDA events).  Then the mixture log-likelihood (egdst_mixture_loglik_device) on the
agent-major panel, one individual per agent, at the same 64 vectors: 32 mixtures of K = 2 types and 64 one-type
mixtures with the per-individual values written out, timed in alternation with the plain choice log-likelihood.

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
obs, start = capi.observations_from_sims(m, sims, start=True)
nobs, k = obs.shape
print("retirement2_smooth: sigma_eps %g, nt %d, nd %d, %d agents, %d observations (k = %d), %d launches per timing" % (
    m.sigma_eps, m.nt, m.nd, nsim, nobs, k, reps))
orders = {"agent-major": obs, "sorted by (age, state)": obs[np.lexsort((obs[:, 1], obs[:, 0]))]}
desc = capi.Desc(m)
d_tot = torch.zeros(64, dtype=torch.float64, device=dev)


def timed(run):
    """ms per call of ``run`` over ``reps`` calls."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        run()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


for label, o in orders.items():
    d_obs = torch.from_numpy(np.ascontiguousarray(o.ravel(order="F"))).to(dev)
    for nvec in (1, 64):
        def run():
            lib.choice_loglik_device(m, sol, d_obs.data_ptr(), nobs, k, d_tot.data_ptr(), sigma_c=0.1, ivec0=0, nvec=nvec, desc=desc)
        for _ in range(3):
            run()
        torch.cuda.synchronize()
        ts = [timed(run) for _ in range(3)]
        med = sorted(ts)[1]
        print("%-24s nvec %2d: %s ms per call (median %.3f ms), %.3g rows x vectors per second" % (
            label, nvec, " ".join("%.3f" % t for t in ts), med, nobs * nvec / (med * 1e-3)))

# mixture leg: agent-major rows, one individual per agent, 64 vectors
nind = start.size - 1
d_obs = torch.from_numpy(np.ascontiguousarray(obs.ravel(order="F"))).to(dev)
d_start = torch.from_numpy(start).to(dev)
d_indll = torch.empty(64 * nind, dtype=torch.float64, device=dev)
legs = {}
for K, nmix in ((2, 32), (1, 64)):
    tv = torch.arange(64, dtype=torch.int32, device=dev).reshape(nmix, K).contiguous()
    w = torch.full((nmix, K), 1.0 / K, dtype=torch.float64, device=dev)
    legs["mixture K = %d x %d" % (K, nmix)] = (K, nmix, tv, w)


def run_choice():
    lib.choice_loglik_device(m, sol, d_obs.data_ptr(), nobs, k, d_tot.data_ptr(), sigma_c=0.1, ivec0=0, nvec=64, desc=desc)


runs = {"choice loglik nvec 64": run_choice}
for label, (K, nmix, tv, w) in legs.items():
    def run(K=K, nmix=nmix, tv=tv, w=w):
        lib.mixture_loglik_device(m, sol, d_obs.data_ptr(), nobs, k, d_start.data_ptr(), nind, tv.data_ptr(), w.data_ptr(),
                                  K, nmix, d_tot.data_ptr(), sigma_c=0.1, d_indll=d_indll.data_ptr() if K == 1 else 0,
                                  ivec0=0, nvec=64, desc=desc)
    runs[label] = run
for run in runs.values():
    for _ in range(3):
        run()
torch.cuda.synchronize()
ts = {label: [] for label in runs}
for _ in range(3):  # alternating rounds
    for label, run in runs.items():
        ts[label].append(timed(run))
print("mixture leg (agent-major, %d individuals, 64 vectors, medians of 3 alternating rounds of %d calls):" % (nind, reps))
base = sorted(ts["choice loglik nvec 64"])[1]
for label, t in ts.items():
    med = sorted(t)[1]
    print("  %-24s %s ms per call (median %.3f ms, %+.3f ms against the choice log-likelihood)" % (
        label, " ".join("%.3f" % x for x in t), med, med - base))
