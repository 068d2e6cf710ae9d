"""Choice draws, choice log-likelihoods, mixtures and scores of smoothing images with continuous states
(egdst_choice_values_cont) on the host emulator of the kernels: humancapital_smooth (one continuous state, two corner
cells) and humancapital2_smooth (two, four corners) against the numpy restatement of tests/continuous_choice_checks.py;
determinism, sharding, the observation layout and the refusals; and the solver of these images: the sigma_eps -> 0
limit against the reference's humancapital solution and the Euler and Bellman equations."""
import os
import shutil
import sys

import numpy as np
import pytest

from egdst_b200 import capi, examples
from tests import choice_draw_checks as cd
from tests import continuous_choice_checks as ccc
from tests.goldens import load
from tests.mixture_loglik_checks import bits
from tests.parity import solution_errors

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "tools", "hostemu"))

pytestmark = pytest.mark.skipif(shutil.which("g++") is None, reason="g++ not available")

_CACHE = {}
MODELS = {"K1": examples.humancapital_smooth, "K2": examples.humancapital2_smooth}


def _lib(m):
    from build import build  # tools/hostemu/build.py
    m.prepare()
    return capi.ModelLibrary(build(m))


def _solved(name):
    if name not in _CACHE:
        m = MODELS[name](sigma_eps=0.2, T=6, ngridm=60, ngridmax=400, ny=4, nz=4)
        lib = _lib(m)
        sol = lib.solve(m)
        assert sol.status()[0] == 0, sol.status()
        _CACHE[name] = (m, lib, sol)
    return _CACHE[name]


def _panel(name, n=3000, seed=11):
    key = (name, "panel")
    if key not in _CACHE:
        m, lib, sol = _solved(name)
        _CACHE[key] = ccc.draw_panel(lib, m, sol, n, seed)
    return _CACHE[key]


@pytest.mark.parametrize("name", sorted(MODELS))
def test_philox_draws_follow_the_corner_rule(name):
    m, lib, sol = _solved(name)
    init, sims = _panel(name)
    checked, counts, below = ccc.check_draws(cd.ChoiceCells(sol, m), sims, cd.philox_uniforms(init.shape[0], m.nt, 11))
    assert checked >= 5000 and (counts > 500).all(), (checked, counts)
    assert below >= 500, below  # z leaves its grid below once an agent at the lowest grid point retires


@pytest.mark.parametrize("name", sorted(MODELS))
def test_randstream_draws_follow_the_corner_rule(name):
    m, lib, sol = _solved(name)
    n = 1000
    rng = np.random.default_rng(3)
    init = np.column_stack([np.ones(n), m.a0 + 0.6 * (m.mmax - m.a0) * rng.random(n)])
    rs = rng.random(4 * m.nt * n)
    sol.set_choice_draws(True)
    try:
        sims = lib.simulate(m, sol, init, rs)
    finally:
        sol.set_choice_draws(False)
    checked, counts, below = ccc.check_draws(cd.ChoiceCells(sol, m), sims, cd.randstream_uniforms(rs, n, m.nt))
    assert checked >= 1500 and (counts > 100).all() and below > 100, (checked, counts, below)


@pytest.mark.parametrize("name", sorted(MODELS))
def test_rows_follow_the_corner_rule(name):
    m, lib, sol = _solved(name)
    _, sims = _panel(name)
    obs = ccc.observations(m, sims)
    cc = cd.ChoiceCells(sol, m)
    for o, sig in ((obs, 0.05), (obs[:, :-1], 0.0), (obs, 0.0)):
        rows, below = ccc.check_rows(cc, lib, o, sigma_c=sig)
        assert rows >= 5000 and below >= 500, (rows, below)
    # the consumption term is centred on the recorded consumption: a row at its own record's consumption adds log phi(0)
    _, r5 = lib.choice_loglik(m, sol, obs, sigma_c=0.05, rows=True)
    _, r4 = lib.choice_loglik(m, sol, obs[:, :-1], rows=True)
    np.testing.assert_allclose(r5[0] - r4[0], -ccc.LOG_SQRT_2PI - np.log(0.05), rtol=0, atol=1e-9)


def test_observation_columns():
    m, lib, sol = _solved("K2")
    _, sims = _panel("K2", n=200)
    obs, start = capi.observations_from_sims(m, sims, start=True)
    live = ~np.isnan(sims[:, :, 0])
    ai, ti = np.nonzero(live)
    assert obs.shape == (ai.size, 7) and start[-1] == ai.size
    np.testing.assert_array_equal(obs[:, 4], sims[ai, ti, 11])
    np.testing.assert_array_equal(obs[:, 5], sims[ai, ti, 12])
    np.testing.assert_array_equal(obs[:, 6], sims[ai, ti, 1])
    assert capi.observations_from_sims(m, sims, consumption=False).shape == (ai.size, 6)


def test_totals_mixtures_and_scores():
    """Totals independent of nvec and ivec0; a one-type mixture equals indll bit for bit; scores equal the numpy
    difference of mixll."""
    m, lib, _ = _solved("K1")
    names = [p["ref"] for p in m.param]
    pv = np.tile(m.param_vector(), (5, 1))
    j, k = names.index("duw"), names.index("gain")
    pv[1, j] += 1e-4; pv[2, j] -= 1e-4; pv[3, k] += 1e-4; pv[4, k] -= 1e-4
    sol = lib.solve_batch(m, pv)
    for v in range(5):
        assert sol.status(v)[0] == 0, (v, sol.status(v))
    _, sims = _panel("K1", n=600, seed=4)
    obs, start = capi.observations_from_sims(m, sims, start=True)
    tot, rows = lib.choice_loglik(m, sol, obs, sigma_c=0.05, rows=True)
    assert np.all(np.isfinite(rows))
    for v in range(5):
        t1, r1 = lib.choice_loglik(m, sol, obs, sigma_c=0.05, ivec0=v, nvec=1, rows=True)
        assert np.array_equal(bits(t1), bits(tot[v:v + 1])) and np.array_equal(bits(r1[0]), bits(rows[v])), v
    tvec = np.arange(5).reshape(5, 1)
    mt, indll, mixll, _ = lib.mixture_loglik(m, sol, obs, start, tvec, np.ones((5, 1)), sigma_c=0.05, individuals=True,
                                             posterior=True)
    assert np.array_equal(bits(mixll), bits(indll))
    hinv = 1.0 / np.array([pv[1, j] - pv[2, j], pv[3, k] - pv[4, k]])
    stot, grad, opg, scores = lib.mixture_scores(m, sol, obs, start, tvec, np.ones((5, 1)), [1, 3], [2, 4], hinv,
                                                 sigma_c=0.05, scores=True)
    want = np.stack([(mixll[1] - mixll[2]) * hinv[0], (mixll[3] - mixll[4]) * hinv[1]])
    np.testing.assert_allclose(scores, want, rtol=1e-13, atol=0)
    np.testing.assert_allclose(grad, want.sum(axis=1), rtol=1e-10)
    np.testing.assert_allclose(opg, want @ want.T, rtol=1e-10)
    assert np.array_equal(bits(stot), bits(mt))
    assert np.any(np.abs(grad) > 0)


def test_draws_do_not_depend_on_sharding():
    m, lib, sol = _solved("K2")
    n = 1024
    rng = np.random.default_rng(9)
    init = np.column_stack([np.ones(n), m.a0 + 0.6 * (m.mmax - m.a0) * rng.random(n)])
    sol.set_choice_draws(True)
    try:
        full, _ = lib.simulate_philox(m, sol, init, seed=77)
        for lo in range(0, n, 256):
            part, _ = lib.simulate_philox(m, sol, init[lo:lo + 256], seed=77, agent0=lo)
            assert np.array_equal(bits(part), bits(full[lo:lo + 256])), lo
    finally:
        sol.set_choice_draws(False)
    assert not np.isnan(full[:, :, 0]).any()


def test_refusals_and_row_checks():
    m, lib, sol = _solved("K1")

    def refused(fn, *words):
        with pytest.raises(capi.EgdstError) as e:
            fn()
        assert e.value.code == 2 and all(w in str(e.value) for w in words), str(e.value)

    # z = 0.2 lies below the grid [0.4, 1.6]: legal, held at the edge
    good = np.array([[m.t0 + 1, 1, 2.0, 1, 0.2, 1.0]] * 3)
    tot, rows = lib.choice_loglik(m, sol, good, sigma_c=0.1, rows=True)
    assert np.all(np.isfinite(rows))
    at_edge = good.copy()
    at_edge[:, 4] = m.s[0]["grid"][0]
    assert np.array_equal(bits(lib.choice_loglik(m, sol, at_edge, rows=True)[1]),
                          bits(lib.choice_loglik(m, sol, good, rows=True)[1]))
    # the state column's grid part is ignored
    other = good.copy()
    other[:, 1] = 3
    assert np.array_equal(bits(lib.choice_loglik(m, sol, other, rows=True)[1]), bits(lib.choice_loglik(m, sol, good, rows=True)[1]))
    refused(lambda: lib.choice_loglik(m, sol, good[:, :4]), "5 or 6")
    refused(lambda: lib.choice_loglik(m, sol, np.column_stack([good, good[:, :1]])), "5 or 6")
    for val in (np.nan, np.inf):
        bad = good.copy()
        bad[2, 4] = val
        refused(lambda: lib.choice_loglik(m, sol, bad), "row 2", "continuous state 1")
        start = np.array([0, 3], dtype=np.int32)
        refused(lambda: lib.mixture_loglik(m, sol, bad, start, [[0]], [[1.0]]), "row 2", "continuous state 1")
    imported = lib.import_solution(m, sol.M, sol.D)
    refused(lambda: imported.set_choice_draws(True), "imported")
    refused(lambda: lib.choice_loglik(m, imported, good), "imported")
    # the _device entry point checks no rows: NaN rows (never a read outside the grid) and a NaN total
    bad = np.vstack([good[:1], good[:1], good[:1], good[:1]])
    bad[1, 4] = np.nan
    bad[2, 4] = -np.inf
    bad[3, 4] = 1e300  # finite, far above the grid: held at the edge
    obsf = np.ascontiguousarray(bad.ravel(order="F"))
    tot = np.zeros(1)
    rowll = np.full(4, 7.0)
    lib.choice_loglik_device(m, sol, obsf.ctypes.data, 4, 6, tot.ctypes.data, d_rowll=rowll.ctypes.data)
    assert np.isfinite(rowll[0]) and np.all(np.isnan(rowll[1:3])) and np.isfinite(rowll[3]) and np.isnan(tot[0])


def test_vanishing_taste_shocks_reproduce_the_reference():
    """humancapital_smooth at sigma_eps = 1e-8 against the reference's humancapital solution (tests/golden), in the
    metric and tolerance of the retirement2 limit test."""
    m = examples.humancapital_smooth(sigma_eps=1e-8)
    lib = _lib(m)
    sol = lib.solve(m)
    assert sol.status(0)[0] == 0, sol.status(0)
    g = load("humancapital")
    e = solution_errors(sol.M, sol.D, g["M"], g["D"])
    assert e["C"] < 1e-6 and e["V"] < 1e-6 and e["TH"] < 1e-6 and e["Dseq"], e


def test_euler_and_bellman_equations_hold_with_a_continuous_state():
    m = examples.humancapital_smooth(sigma_eps=0.2, T=5, ngridm=300, ngridmax=900, ny=5, nz=5)
    lib = _lib(m)
    sol = lib.solve(m)
    assert sol.status(0)[0] == 0, sol.status(0)
    for it in (3, 2, 0):
        w = ccc.euler_bellman_residuals_humancapital(sol, m, it)
        assert w["euler"] < 1e-8 and w["bellman"] < 1e-7 and w["points"] > 1000, (it, w)
