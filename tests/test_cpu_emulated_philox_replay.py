"""The Philox-driven simulator on the host emulator, replayed agent by agent through the reference simulator's C
restatement (tests/philox_replay_checks.py): PB = 1 and PB = 2 (the emulator's launch takes PB = 2 from 1024 agents
on), sims only, moments only and both, agent ids and seeds with high words, the randstream entry points fed the same
uniforms, a batched sweep and an imported solution with more thresholds in some cells than the per-cell headers carry.
Each launch asserts the instantiation of egdst_k_simulate it took (egdst_test_sim_variant) against the one it names."""
import os
import shutil
import sys

import numpy as np
import pytest

from egdst_b200 import capi, examples
from tests import philox_replay_checks as R

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "tools", "hostemu"))

pytestmark = pytest.mark.skipif(shutil.which("g++") is None, reason="g++ not available")

AGENT0, SEED = 2**32 - 700, 2**40 + 5  # the launch crosses the high word of the agent id; the seed has a high word
NSIM = 2053                            # 65 tiles, the last one a tail: PB = 2 for launches that write the paths
NSIM_PB1 = 700                         # 22 tiles: below the PB = 2 threshold


def _launch(lib, m, sol, init, agent0, expect, sims=True, moments=True):
    """simulate_device on host buffers (the emulator's device pointers), which must take the instantiation `expect`:
    paths [nsim, nt, nsimout] and moments [nt, nsimout, 3], None where not requested."""
    n = init.shape[0]
    flat = np.ascontiguousarray(np.concatenate([init[:, 0], init[:, 1]]))
    s = np.full(n * m.nt * m.nsimout(), 7.0) if sims else None
    mo = np.zeros(3 * m.nsimout() * m.nt) if moments else None
    n0 = lib.sim_variant()[1]
    lib.simulate_device(m, sol, flat.ctypes.data, n, agent0, SEED, s.ctypes.data if sims else 0, mo.ctypes.data if moments else 0)
    R.check_variant(lib, n0, expect, label=m.label)
    return (s.reshape(n, m.nt, m.nsimout()) if sims else None), (mo.reshape(m.nt, m.nsimout(), 3) if moments else None)


def _init(m, n, seed=3):
    rng = np.random.default_rng(seed)
    m0 = m.a0 + 0.5 * (m.mmax - m.a0) * rng.random(n)
    m0[::37] = m.a0 - 1.0  # about 3 % skipped agents: NaN from period 0
    return R.init_matrix(np.ones(n), m0)  # state 1: the first grid point of a continuous state


def _bits_equal(a, b):
    nan = np.isnan(a)
    return np.array_equal(nan, np.isnan(b)) and np.array_equal(a[~nan].view(np.int64), b[~nan].view(np.int64))


MODELS = {
    "retirement2": lambda: examples.retirement2(T=6, ngridm=40, ngridmax=200, ny=4),
    "retirement_mortal": lambda: examples.retirement_mortal(T=6, ngridm=40, ngridmax=200, ny=4),
    # nt * nst = 130 > 128: no per-cell headers (HDR = false); PB = 2 on the plain period order (continuous state)
    "humancapital": lambda: examples.humancapital(T=26, ngridm=30, ngridmax=150, ny=3),
}


@pytest.fixture(scope="module", params=sorted(MODELS))
def solved(request):
    from build import build  # tools/hostemu/build.py
    m = MODELS[request.param]()
    m.prepare()
    lib = capi.ModelLibrary(build(m))
    sol = lib.solve(m)
    assert sol.status()[0] == 0, sol.status()
    init = _init(m, NSIM)
    rs = R.philox_randstream(NSIM, m.nt, SEED, AGENT0)
    rp = R.Replay(m, sol, 0, init, rs)
    return request.param, m, lib, sol, init, rs, rp


def test_emulated_philox_launches_match_the_replay(solved):
    name, m, lib, sol, init, rs, rp = solved
    hdr = m.nt * m.nst <= 128
    assert hdr == (name != "humancapital")
    port = rp.paths
    live = ~np.isnan(port[:, :, 0])
    assert not live[::37].any() and live[:, 0].sum() == NSIM - len(range(0, NSIM, 37))
    if name == "retirement_mortal":
        assert (live[:, 0] & ~live[:, -1]).any()  # deaths on the way
    ref = R.moment_reference(port)
    # PB = 2: sims and moments, then sims alone
    full, mom = _launch(lib, m, sol, init, AGENT0, (True, 3, hdr, 2, True))
    tol = R.compare_paths(full, port, rp.cells, replay=rp, label="%s <true, 3, %s, 2>" % (name, hdr))["max"]
    R.check_moments(mom, ref, tol, label="%s <true, 3, %s, 2>" % (name, hdr))
    only, _ = _launch(lib, m, sol, init, AGENT0, (True, 1, hdr, 2), moments=False)
    assert _bits_equal(only, full)
    # moments only: PB = 1, no path array to check them against
    _, mom2 = _launch(lib, m, sol, init, AGENT0, (True, 2, hdr, 1, True), sims=False)
    R.check_moments(mom2, ref, tol, label="%s <true, 2, %s, 1>" % (name, hdr))
    # PB = 1: the first agents of the same launch, with their own ids
    n1 = NSIM_PB1
    part, mom1 = _launch(lib, m, sol, init[:n1], AGENT0, (True, 3, hdr, 1, True))
    tol1 = R.compare_paths(part, port[:n1], rp.cells, replay=rp, label="%s <true, 3, %s, 1>" % (name, hdr))["max"]
    R.check_moments(mom1, R.moment_reference(port[:n1]), tol1, label="%s <true, 3, %s, 1>" % (name, hdr))
    assert _bits_equal(part, full[:n1])  # PB = 2 against PB = 1 (DESIGN section 5)
    # the randstream entry point fed the Philox uniforms: the same records to the bit
    n0 = lib.sim_variant()[1]
    assert _bits_equal(lib.simulate(m, sol, init, rs), full)
    R.check_variant(lib, n0, (False, 1, hdr, 1), label=m.label)
    # rndtype 1: every agent on one block, against the port's rndtype 1 replay
    r1 = R.replay(m, sol, 0, init[:n1], SEED, AGENT0, rndtype=1)
    R.compare_paths(lib.simulate(m, sol, init[:n1], r1.rs.ravel(), rndtype=1), r1.paths, r1.cells, label="%s rndtype 1" % name)


def test_emulated_sweep_moments_match_the_replays():
    """Moments of a batched sweep (one launch, blockIdx.y over the vectors) against the replay of each vector under
    its own parameter values."""
    from build import build
    kw = dict(T=6, ngridm=40, ngridmax=200, ny=4)
    m = examples.retirement2(**kw)
    m.prepare()
    lib = capi.ModelLibrary(build(m))
    rng = np.random.default_rng(11)
    nvec = 5
    params = np.column_stack([rng.uniform(0.3, 0.7, nvec), rng.uniform(0.02, 0.06, nvec), rng.uniform(0.9, 1.2, nvec)])  # duw, interest, wage
    sol = lib.solve_batch(m, params)
    assert sol.warning is None, sol.warning
    n = 600
    init = _init(m, n, seed=5)
    n0 = lib.sim_variant()[1]
    mom = lib.sim_moments(m, sol, init, SEED, agent0=AGENT0)  # [nvec, 3, nsimout, nt]
    R.check_variant(lib, n0, (True, 2, False, 1), label="sweep")
    rs = R.philox_randstream(n, m.nt, SEED, AGENT0)
    for i in (0, 2, nvec - 1):
        mi = examples.retirement2(duw=params[i, 0], interest=params[i, 1], wage=params[i, 2], **kw)
        rp = R.Replay(mi, sol, i, init, rs)
        # the vector's own paths (a single-vector launch) bound what its records may differ from the port's
        paths, _ = lib.simulate_philox(m, sol, init, SEED, agent0=AGENT0, ivec=i)
        tol = R.compare_paths(paths, rp.paths, rp.cells, replay=rp, label="sweep vector %d" % i)["max"]
        R.check_moments(mom[i].transpose(2, 1, 0), R.moment_reference(rp.paths), tol, label="sweep vector %d" % i)
    # a vector replayed with the base model's parameters differs: the check sees the parameter values
    rp0 = R.Replay(m, sol, nvec - 1, init, rs)
    with pytest.raises(AssertionError):
        R.check_moments(mom[nvec - 1].transpose(2, 1, 0), R.moment_reference(rp0.paths), tol)


def test_emulated_thresholds_beyond_the_headers_match_the_replay():
    """Per-cell headers carry EGDST_SIM_TH8 = 4 thresholds; a cell with more takes the policy decision from the threshold
    table in global memory.  No shipped example has such a cell, so an imported solution gets 6 thresholds in the
    even periods and keeps the solver's (at most 2) in the odd ones: PB = 2 (pipelined) and PB = 1, both with headers."""
    from build import build
    m = MODELS["retirement2"]()
    m.prepare()
    lib = capi.ModelLibrary(build(m))
    # six thresholds over the cash the agents hold (initial cash up to the middle of the grid)
    M, D = R.with_thresholds(*lib.solve(m).cells(0), periods=range(0, m.nt, 2), k=6, lo=m.a0, hi=m.a0 + 0.5 * (m.mmax - m.a0))
    sol = lib.import_solution(m, M, D)
    nth = [sol.cells(0)[1][0][it].shape[0] for it in range(m.nt)]
    assert max(nth) > 4 and min(nth) <= 4, nth
    init = _init(m, NSIM)
    rp = R.replay(m, sol, 0, init, SEED, AGENT0)
    ref = R.moment_reference(rp.paths)
    full, mom = _launch(lib, m, sol, init, AGENT0, (True, 3, True, 2, True))
    tol = R.compare_paths(full, rp.paths, rp.cells, replay=rp, label="imported thresholds <true, 3, true, 2>")["max"]
    R.check_moments(mom, ref, tol, label="imported thresholds <true, 3, true, 2>")
    assert len(np.unique(full[:, 0::2, 4][~np.isnan(full[:, 0::2, 4])])) == 2  # both decisions taken in the 6-threshold cells
    part, _ = _launch(lib, m, sol, init[:NSIM_PB1], AGENT0, (True, 1, True, 1), moments=False)
    assert _bits_equal(part, full[:NSIM_PB1])
