"""Choice log-likelihood of the smoothing mode (egdst_choice_loglik) on the host emulator of the kernels: the row values
against numpy (tests/choice_loglik_checks.py) for both sources of choice draws, the edge rules above and below the
grid, an unavailable decision, the consumption term, deterministic totals, batched solutions, refusals and the
row checks of the host entry point."""
import math
import shutil
import sys
import os

import numpy as np
import pytest

from egdst_b200 import capi, examples
from tests import choice_draw_checks as cd
from tests import choice_loglik_checks as cl

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "tools", "hostemu"))

pytestmark = pytest.mark.skipif(shutil.which("g++") is None, reason="g++ not available")

_CACHE = {}


def _solved():
    """retirement2_smooth (T=6), sigma_eps = 0.2, solved on the emulator."""
    if "sol" not in _CACHE:
        from build import build  # tools/hostemu/build.py
        m = examples.retirement2_smooth(sigma_eps=0.2, T=6, ngridm=300, ny=5)
        m.prepare()
        lib = capi.ModelLibrary(build(m))
        sol = lib.solve(m)
        assert sol.status()[0] == 0, sol.status()
        _CACHE["sol"] = (m, lib, sol)
    return _CACHE["sol"]


def _init(m, n, seed=1):
    rng = np.random.default_rng(seed)
    return np.column_stack([np.ones(n), m.a0 + 0.6 * (m.mmax - m.a0) * rng.random(n)])


def _drawn_sims(source, n=2000):
    m, lib, sol = _solved()
    sol.set_choice_draws(True)
    try:
        if source == "randstream":
            rs = np.random.default_rng(7).random(4 * m.nt * n)
            return lib.simulate(m, sol, _init(m, n), rs)
        return lib.simulate_philox(m, sol, _init(m, n, seed=2), seed=12345, agent0=5)[0]
    finally:
        sol.set_choice_draws(False)


@pytest.mark.parametrize("source", ["randstream", "philox"])
def test_rows_are_the_log_choice_probabilities(source):
    m, lib, sol = _solved()
    cl.check_mechanism(cd.ChoiceCells(sol, m), lib, _drawn_sims(source))


def test_held_above_the_grid_and_constrained_below_it():
    m, lib, sol = _solved()
    cc = cd.ChoiceCells(sol, m)
    it, ist = 2, 0
    cells = [c for c in cc.cells(it, ist) if c is not None and c.shape[0] >= 3]
    top = max(c[-1, 0] for c in cells)
    low = min(c[1, 0] for c in cells)
    age = m.t0 + it
    # two cash values above every decision's grid, both decisions: the probabilities are held at the bound
    obs = np.array([[age, 1, top + 0.5, d] for d in (1, 2)] + [[age, 1, top + 3.0, d] for d in (1, 2)], dtype=float)
    _, r = lib.choice_loglik(m, sol, obs, rows=True)
    assert np.all(np.isfinite(r))
    assert np.array_equal(r[0, :2].view(np.int64), r[0, 2:].view(np.int64))
    # below every decision's M[1]: the credit-constrained branch
    M = m.a0 + (low - m.a0) * np.array([0.05, 0.3, 0.7, 0.95])
    assert np.all(M < low)
    obs = np.array([[age, 1, x, d] for d in (1, 2) for x in M], dtype=float)
    _, r = lib.choice_loglik(m, sol, obs, rows=True)
    want = np.concatenate(list(cl.constrained_logp(cc, lib, it, ist, M)))
    # retiring in debt (a0 < 0) has no finite value (evf_d(a0) = -inf): probability 0; working rows are finite
    assert np.all(want[:4] == -np.inf) and np.all(np.isfinite(want[4:]))
    assert np.array_equal(np.isfinite(r[0]), np.isfinite(want))
    np.testing.assert_allclose(r[0], want, rtol=0, atol=1e-10)


def test_unavailable_decision_is_minus_infinity():
    from build import build  # tools/hostemu/build.py
    m = examples.model2()
    m.sigma_eps = 0.2
    m.prepare()
    lib = capi.ModelLibrary(build(m))
    sol = lib.solve(m)
    assert sol.status()[0] == 0, sol.status()
    # state 1 (retired) is absorbing: decision 2 (work) is not available there
    obs = np.array([[m.t0, 1, 5.0, 2], [m.t0, 1, 5.0, 1], [m.t0 + 1, 1, 20.0, 2], [m.t0 + 1, 1, 20.0, 1]], dtype=float)
    tot, r = lib.choice_loglik(m, sol, obs, rows=True)
    assert np.array_equal(r[0], [-np.inf, 0.0, -np.inf, 0.0])
    assert tot[0] == -np.inf
    # the working state has both decisions, with probabilities that sum to one
    obs = np.array([[m.t0, 2, 5.0, 1], [m.t0, 2, 5.0, 2]], dtype=float)
    _, r = lib.choice_loglik(m, sol, obs, rows=True)
    assert np.all(np.isfinite(r)) and abs(np.exp(r[0]).sum() - 1.0) < 1e-12


def test_consumption_term():
    m, lib, sol = _solved()
    cc = cd.ChoiceCells(sol, m)
    obs, _, _ = cl.interior_obs(cc, _drawn_sims("philox"), consumption=True)
    obs[::5, 4] = np.nan  # consumption not observed
    diff, k4, s0 = cl.consumption_terms(lib, m, sol, obs, 0.1)
    seen = ~np.isnan(obs[:, 4])
    np.testing.assert_allclose(diff[seen], -math.log(0.1) - cl.LOG_SQRT_2PI, rtol=0, atol=1e-9)
    assert np.all(diff[~seen] == 0.0)
    assert np.array_equal(k4.view(np.int64), s0.view(np.int64))
    # consumption off the model's by delta: -delta^2 / (2 sigma_c^2) on top of the constant
    delta = np.where(np.arange(obs.shape[0]) % 2 == 0, 0.03, -0.07)
    off = obs.copy()
    off[:, 4] += delta
    diff_off, _, _ = cl.consumption_terms(lib, m, sol, off, 0.1)
    want = -math.log(0.1) - cl.LOG_SQRT_2PI - 0.5 * (delta / 0.1) ** 2
    np.testing.assert_allclose(diff_off[seen], want[seen], rtol=0, atol=1e-9)
    assert np.all(diff_off[~seen] == 0.0)


def test_totals_are_deterministic_and_shards_sum_to_them():
    m, lib, sol = _solved()
    obs = capi.observations_from_sims(m, _drawn_sims("philox"))
    t1, r = lib.choice_loglik(m, sol, obs, sigma_c=0.2, rows=True)
    t2 = lib.choice_loglik(m, sol, obs, sigma_c=0.2)
    assert np.array_equal(t1.view(np.int64), t2.view(np.int64))
    cl.check_total(t1[0], r[0])
    parts = [lib.choice_loglik(m, sol, obs[lo:hi], sigma_c=0.2)[0] for lo, hi in ((0, 700), (700, 701), (701, obs.shape[0]))]
    assert abs(math.fsum(parts) - t1[0]) <= 1e-12 * abs(t1[0])
    # EgdstModel.loglik evaluates the model's current solution
    m.__dict__["_solution"] = sol
    m.__dict__["_lib"] = lib
    m.__dict__["needtocompile"] = False
    assert m.loglik(obs, sigma_c=0.2) == t1[0]


@pytest.mark.parametrize("scope", ["cta", "warp"])
def test_batched_vectors_match_single_vector_calls(monkeypatch, scope):
    from build import build  # tools/hostemu/build.py
    m = examples.retirement2_smooth(sigma_eps=0.2, T=6, ngridm=100, ngridmax=300, ny=5)
    m.prepare()
    lib = capi.ModelLibrary(build(m))
    names = [p["ref"] for p in m.param]
    pv = np.array([list(m.param_vector())] * 12)
    pv[:, names.index("duw")] *= 1.0 + 0.03 * np.arange(12)
    monkeypatch.setenv("EGDST_SOLVE_SCOPE", scope)
    monkeypatch.setenv("EGDST_WARP_G", "5")
    sol = lib.solve_batch(m, pv)
    for v in range(12):
        assert sol.status(v)[0] == 0, (v, sol.status(v))
    sol.set_choice_draws(True)
    sims, _ = lib.simulate_philox(m, sol, _init(m, 300, seed=6), seed=555)
    sol.set_choice_draws(False)
    obs = capi.observations_from_sims(m, sims)
    tot, r = lib.choice_loglik(m, sol, obs, sigma_c=0.1, rows=True)
    assert tot.shape == (12,) and r.shape == (12, obs.shape[0])
    assert np.unique(tot).size == 12
    for v in range(12):
        t1, r1 = lib.choice_loglik(m, sol, obs, sigma_c=0.1, ivec0=v, nvec=1, rows=True)
        assert np.array_equal(r1[0].view(np.int64), r[v].view(np.int64)), v
        assert np.array_equal(t1.view(np.int64), tot[v:v + 1].view(np.int64)), v


def test_refusals_and_row_checks():
    from build import build  # tools/hostemu/build.py
    m, lib, sol = _solved()
    good = np.array([[m.t0 + 1, 1, 2.0, 1, 1.0]] * 3)

    def refused(fn, *words):
        with pytest.raises(capi.EgdstError) as e:
            fn()
        assert e.value.code == 2 and all(w in str(e.value) for w in words), str(e.value)

    imported = lib.import_solution(m, sol.M, sol.D)
    refused(lambda: lib.choice_loglik(m, imported, good), "imported")
    refused(lambda: lib.choice_loglik(m, sol, good[:, :3]), "4 or 5")
    refused(lambda: lib.choice_loglik(m, sol, good, sigma_c=-1.0), "sigma_c")
    refused(lambda: lib.choice_loglik(m, sol, good, ivec0=1, nvec=1), "out of range")
    for col, val, word in ((0, m.T + 1, "age"), (3, 0, "decision"), (2, np.nan, "cash"), (1, 1.5, "state"), (2, m.a0 - 1, "cash")):
        bad = good.copy()
        bad[2, col] = val
        refused(lambda: lib.choice_loglik(m, sol, bad), "row 2", word)
    # the _device entry point checks no rows: NaN rows and a NaN total
    bad = np.array([[m.t0 + 1, 1, 2.0, 1], [m.T + 1, 1, 2.0, 1], [m.t0 + 1, 1, 2.0, 0], [m.t0 + 1, 1, np.nan, 1]], dtype=float)
    obsf = np.ascontiguousarray(bad.ravel(order="F"))
    tot = np.zeros(1)
    rowll = np.full(4, 7.0)
    lib.choice_loglik_device(m, sol, obsf.ctypes.data, 4, 4, tot.ctypes.data, d_rowll=rowll.ctypes.data)
    assert np.isfinite(rowll[0]) and np.all(np.isnan(rowll[1:])) and np.isnan(tot[0])
    # an image without taste shocks
    m2 = examples.retirement2(T=6, ngridm=40, ngridmax=200, ny=4)
    m2.prepare()
    lib2 = capi.ModelLibrary(build(m2))
    sol2 = lib2.solve(m2)
    refused(lambda: lib2.choice_loglik(m2, sol2, good[:, :4]), "sigma_eps")
