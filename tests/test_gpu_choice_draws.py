"""Choice draws of the smoothing mode (egdst_solution_set_choice_draws) on the GPU: the drawn decision and its record
against a numpy restatement at full size, the distribution of the draws, the limit sigma_eps -> 0, large launches and
batched sweeps (tests/choice_draw_checks.py)."""
import numpy as np
import pytest
import torch

from egdst_b200 import capi, examples
from tests import choice_draw_checks as cd

pytestmark = pytest.mark.gpu


def _solved(sigma_eps, **kw):
    m = examples.retirement2_smooth(sigma_eps=sigma_eps, **kw)
    m.compile()
    lib = m._capi()
    sol = lib.solve(m, strict=True)
    return m, lib, sol


def _init(m, n, seed=1):
    rng = np.random.default_rng(seed)
    return np.column_stack([np.ones(n), m.a0 + 0.6 * (m.mmax - m.a0) * rng.random(n)])


@pytest.mark.parametrize("sigma_eps", [0.2, 0.05])
def test_randstream_draws_follow_the_choice_probabilities(sigma_eps):
    m, lib, sol = _solved(sigma_eps)
    n = 20000
    init = _init(m, n)
    rs = np.random.default_rng(7).random(4 * m.nt * n)
    sol.set_choice_draws(True)
    sims = lib.simulate(m, sol, init, rs)
    checked, counts = cd.check_mechanism(cd.ChoiceCells(sol, m), sims, cd.randstream_uniforms(rs, n, m.nt))
    assert checked >= 10000 and (counts > 100).all(), (checked, counts)


def test_draw_frequencies_match_the_choice_probabilities():
    m, lib, sol = _solved(0.2)
    cc = cd.ChoiceCells(sol, m)
    lo, hi = cc.grid(0, 0)
    m0 = lo + 0.37 * (hi - lo)
    n = 1_000_000
    init = np.column_stack([np.ones(n), np.full(n, m0)])
    sol.set_choice_draws(True)
    _, mom = lib.simulate_philox(m, sol, init, seed=2024, want_sims=False, want_moments=True)
    # decisions are 0/1: the sum of the decision column of period 0 counts the draws of decision 1
    assert mom[2, cd.DEC, 0] == n
    p1 = cc.probabilities(0, 0, [m0])[1, 0]
    assert 0.05 < p1 < 0.95, p1
    assert abs(mom[0, cd.DEC, 0] - n * p1) <= 5 * np.sqrt(n * p1 * (1 - p1)), (mom[0, cd.DEC, 0] / n, p1)
    # every interior record of a sample of agents with spread initial cash
    sims, _ = lib.simulate_philox(m, sol, _init(m, 4096, seed=5), seed=77)
    ai, ti = cd.interior_records(cc, sims)
    assert ai.size > 10000
    dev, var = np.zeros(m.nd), np.zeros(m.nd)
    for it in np.unique(ti):
        a = ai[ti == it]
        P = cc.probabilities(int(it), 0, sims[a, it, cd.CASH])
        for d in range(m.nd):
            dev[d] += np.sum((sims[a, it, cd.DEC] == d) - P[d])
            var[d] += np.sum(P[d] * (1 - P[d]))
    assert np.all(np.abs(dev) <= 5 * np.sqrt(var)), (dev, var)


def test_vanishing_taste_shocks_draw_the_modal_choice():
    m, lib, sol = _solved(1e-8)
    n = 20000
    init = _init(m, n, seed=3)
    rs = np.random.default_rng(9).random(4 * m.nt * n)
    modal = lib.simulate(m, sol, init, rs)
    sol.set_choice_draws(True)
    drawn = lib.simulate(m, sol, init, rs)
    discrete = [cd.DEC, cd.IST] + list(range(11 + m.nnst, 11 + m.nnst + m.nnd))
    same = np.all((modal[:, :, discrete] == drawn[:, :, discrete]) | (np.isnan(modal[:, :, discrete]) & np.isnan(drawn[:, :, discrete])), axis=(1, 2))
    assert same.mean() >= 0.999, same.mean()
    a, b = modal[same], drawn[same]
    assert np.array_equal(np.isnan(a), np.isnan(b))
    fin = ~np.isnan(a)
    assert np.all((a[fin] == b[fin]) | (np.abs(a[fin] - b[fin]) <= 1e-9))  # == covers equal infinities


def test_large_draw_launches_hold_the_records_of_small_ones():
    m, lib, sol = _solved(0.2, T=24)  # nt even: modal mode would take the two-periods-per-write kernel at this size
    sol.set_choice_draws(True)
    nt, nso = m.nt, m.nsimout()
    dev = torch.device("cuda", 0)
    big, small = 300_000, 1024
    init = _init(m, big, seed=4)
    init[::101, 1] = m.a0 - 1.0  # skipped agents
    desc = capi.Desc(m)
    out = []
    for n in (big, small):
        d_init = torch.from_numpy(np.ascontiguousarray(np.concatenate([init[:n, 0], init[:n, 1]]))).to(dev)
        d_sims = torch.full((n * nt * nso,), 7.0, dtype=torch.float64, device=dev)
        lib.simulate_device(m, sol, d_init.data_ptr(), n, 0, 31337, d_sims.data_ptr(), 0, desc=desc)
        torch.cuda.synchronize()
        out.append(d_sims[:small * nt * nso].cpu().numpy())
    a, b = out
    assert np.array_equal(np.isnan(a), np.isnan(b)) and np.isnan(a).any()
    assert np.array_equal(a[~np.isnan(a)].view(np.int64), b[~np.isnan(b)].view(np.int64))


@pytest.mark.parametrize("scope", ["cta", "warp"])
def test_sweep_moments_with_draws(monkeypatch, scope):
    m = examples.retirement2_smooth(sigma_eps=0.1, ngridm=200, ngridmax=600)
    m.compile()
    lib = m._capi()
    names = [p["ref"] for p in m.param]
    pv = np.array([list(m.param_vector())] * 12)
    pv[:, names.index("duw")] *= 1.0 + 0.03 * np.arange(12)
    monkeypatch.setenv("EGDST_SOLVE_SCOPE", scope)
    monkeypatch.setenv("EGDST_WARP_G", "5")
    sol = lib.solve_batch(m, pv)
    for v in range(12):
        assert sol.status(v)[0] == 0, (v, sol.status(v))
    sol.set_choice_draws(True)
    init = _init(m, 50_000, seed=6)
    sweep = lib.sim_moments(m, sol, init, seed=555)
    drawn0 = None
    for v in range(12):
        _, mom = lib.simulate_philox(m, sol, init, seed=555, ivec=v, want_sims=False, want_moments=True)
        np.testing.assert_allclose(sweep[v], mom, rtol=1e-12, atol=0)
        if v == 0:
            drawn0 = mom
    sol.set_choice_draws(False)
    _, m0 = lib.simulate_philox(m, sol, init, seed=555, ivec=0, want_sims=False, want_moments=True)
    assert not np.array_equal(m0[0, cd.DEC], drawn0[0, cd.DEC])
