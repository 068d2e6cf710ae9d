"""Time the choice log-likelihood (egdst_choice_loglik_device) of retirement2_smooth at its defaults: a panel from a
Philox draw simulation, evaluated for nvec = 1 and 64 parameter vectors, once in agent-major row order and once sorted
by (age, state), with warm-up (CUDA events).  Then the mixture log-likelihood (egdst_mixture_loglik_device) on the
agent-major panel, one individual per agent, at the same 64 vectors: 32 mixtures of K = 2 types and 64 one-type
mixtures with the per-individual values written out, timed in alternation with the plain choice log-likelihood.
Then the central-difference scores (egdst_mixture_scores_device) of (duw, wage, interest) over their 7-vector
stencil, in alternation with the mixture log-likelihood of the same 7 vectors, and one BHHH iteration of
EgdstModel.fit end to end (host clock).

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

# scores leg: the central-difference stencil of (duw, wage, interest) at the defaults (7 vectors, centre first), the
# same agent-major panel; the scores (egdst_mixture_scores_device, P = 3) against the mixture log-likelihood of the
# same 7 one-type mixtures, in alternation: the difference is the cost of the score pass
free = ["duw", "wage", "interest"]
idx = [names.index(f) for f in free]
npar, nv = len(idx), 2 * len(idx) + 1
pv7 = np.tile(m.param_vector(), (nv, 1))
for p, j in enumerate(idx):
    h = 1e-4 * max(abs(pv7[0, j]), 1.0)
    pv7[1 + 2 * p, j] += h
    pv7[2 + 2 * p, j] -= h
mplus, mminus = 1 + 2 * np.arange(npar), 2 + 2 * np.arange(npar)
sol7 = lib.solve_batch(m, pv7)
tv7 = torch.arange(nv, dtype=torch.int32, device=dev)
w7 = torch.ones(nv, dtype=torch.float64, device=dev)
d_mp = torch.from_numpy(mplus.astype(np.int32)).to(dev)
d_mm = torch.from_numpy(mminus.astype(np.int32)).to(dev)
d_h = torch.from_numpy(1.0 / (pv7[mplus, idx] - pv7[mminus, idx])).to(dev)
d_grad = torch.zeros(npar, dtype=torch.float64, device=dev)
d_opg = torch.zeros(npar * npar, dtype=torch.float64, device=dev)


def run_mix7():
    lib.mixture_loglik_device(m, sol7, d_obs.data_ptr(), nobs, k, d_start.data_ptr(), nind, tv7.data_ptr(), w7.data_ptr(),
                              1, nv, d_tot.data_ptr(), sigma_c=0.1, ivec0=0, nvec=nv, desc=desc)


def run_scores():
    lib.mixture_scores_device(m, sol7, d_obs.data_ptr(), nobs, k, d_start.data_ptr(), nind, tv7.data_ptr(), w7.data_ptr(),
                              1, nv, npar, d_mp.data_ptr(), d_mm.data_ptr(), d_h.data_ptr(), d_tot.data_ptr(),
                              d_grad.data_ptr(), d_opg.data_ptr(), sigma_c=0.1, ivec0=0, nvec=nv, desc=desc)


runs = {"mixture loglik 7 x 1": run_mix7, "scores P = 3": run_scores}
for run in runs.values():
    for _ in range(3):
        run()
torch.cuda.synchronize()
ts = {label: [] for label in runs}
for _ in range(3):
    for label, run in runs.items():
        ts[label].append(timed(run))
print("scores leg (agent-major, %d individuals, 7 vectors, medians of 3 alternating rounds of %d calls):" % (nind, reps))
base = sorted(ts["mixture loglik 7 x 1"])[1]
for label, t in ts.items():
    med = sorted(t)[1]
    print("  %-24s %s ms per call (median %.3f ms, %+.3f ms against the mixture log-likelihood)" % (
        label, " ".join("%.3f" % x for x in t), med, med - base))

# one BHHH iteration of EgdstModel.fit end to end (host clock, synchronous calls, host row checks and uploads
# included): the scores (a 7-vector batched solve and one egdst_mixture_scores call) and the line search (a 4-vector
# batched solve and one egdst_mixture_loglik call)
import time  # noqa: E402
lam = np.array([1.0, 0.5, 0.25, 0.125])


def scores_step():
    return m.scores(obs, start, free, sigma_c=0.1)


def line_search():
    p4 = np.tile(m.param_vector(), (lam.size, 1))
    p4[:, idx] += lam[:, None] * 1e-3
    s4 = lib.solve_batch(m, p4)
    return lib.mixture_loglik(m, s4, obs, start, np.arange(lam.size).reshape(-1, 1), np.ones((lam.size, 1)), sigma_c=0.1)


def wall(fn):
    t = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return 1e3 * (time.perf_counter() - t)


for fn in (scores_step, line_search):
    fn()
tw = {"scores": [], "line search": []}
for _ in range(3):
    tw["scores"].append(wall(scores_step))
    tw["line search"].append(wall(line_search))
med = {label: sorted(t)[1] for label, t in tw.items()}
print("one BHHH iteration (P = 3, %d rows, medians of 3): scores %.1f ms (%s), line search %.1f ms (%s), total %.1f ms" % (
    nobs, med["scores"], " ".join("%.1f" % x for x in tw["scores"]), med["line search"],
    " ".join("%.1f" % x for x in tw["line search"]), med["scores"] + med["line search"]))
