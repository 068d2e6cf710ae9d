"""Choice draws and choice log-likelihoods of smoothing images with continuous states (egdst_choice_values_cont) on the
GPU: humancapital_smooth (K = 1) and humancapital2_smooth (K = 2) at full size against the numpy restatement of
tests/continuous_choice_checks.py, the distribution of the draws, the limit sigma_eps -> 0 against the modal records,
a large likelihood launch, the solver's limit, and BHHH recovery of (duw, gain) from a draw panel."""
import numpy as np
import pytest
import torch

from egdst_b200 import capi, examples
from tests import choice_draw_checks as cd
from tests import continuous_choice_checks as ccc
from tests.goldens import load
from tests.parity import solution_errors

pytestmark = pytest.mark.gpu

MODELS = {"K1": examples.humancapital_smooth, "K2": examples.humancapital2_smooth}
SIGMA_C = 0.05
# BHHH stopping rule of the recovery panel (as for the retirement2_smooth panel of the same size): the numerical noise
# of the totals bounds the criterion that can be reached
FIT_TOL = 1e-6


def _solved(name, sigma_eps=0.2, **kw):
    m = MODELS[name](sigma_eps=sigma_eps, **kw)
    m.compile()
    lib = m._capi()
    sol = lib.solve(m, strict=True)
    return m, lib, sol


@pytest.mark.parametrize("name", sorted(MODELS))
def test_draws_and_rows_follow_the_corner_rule(name):
    m, lib, sol = _solved(name)
    n = 100_000
    init, sims = ccc.draw_panel(lib, m, sol, n, seed=21)
    cc = cd.ChoiceCells(sol, m)
    checked, counts, below = ccc.check_draws(cc, sims, cd.philox_uniforms(n, m.nt, 21))
    assert checked >= 300_000 and (counts > 10_000).all() and below >= 5_000, (checked, counts, below)
    obs = ccc.observations(m, sims)
    rows, below = ccc.check_rows(cc, lib, obs, sigma_c=SIGMA_C)
    assert rows >= 300_000 and below >= 5_000, (rows, below)
    rs = np.random.default_rng(5).random(4 * m.nt * 20_000)
    sol.set_choice_draws(True)
    sims = lib.simulate(m, sol, init[:20_000], rs)
    sol.set_choice_draws(False)
    checked, counts, _ = ccc.check_draws(cc, sims, cd.randstream_uniforms(rs, 20_000, m.nt))
    assert checked >= 100_000 and (counts > 1000).all(), (checked, counts)


@pytest.mark.parametrize("name", sorted(MODELS))
def test_draw_frequencies_match_the_choice_probabilities(name):
    m, lib, sol = _solved(name)
    _, sims = ccc.draw_panel(lib, m, sol, 50_000, seed=8)
    ai, ti, ist, M, X = ccc.record_points(m, sims)
    R = ccc.Restated(cd.ChoiceCells(sol, m), ti, ist, M, X)
    dec = sims[ai, ti, cd.DEC]
    keep = R.inside
    for d in range(m.nd):
        dev = np.sum((dec[keep] == d) - R.P[d, keep])
        var = np.sum(R.P[d, keep] * (1.0 - R.P[d, keep]))
        assert var > 1000 and abs(dev) <= 5.0 * np.sqrt(var), (d, dev, var)


@pytest.mark.parametrize("name", sorted(MODELS))
def test_vanishing_taste_shocks_draw_the_modal_choice(name):
    """At sigma_eps = 1e-8, records whose x lies inside the grid and whose kept corners all share the modal decision
    are the modal records, in the tolerances of the all-discrete limit test."""
    m, lib, sol = _solved(name, sigma_eps=1e-8)
    n = 20_000
    rng = np.random.default_rng(3)
    init = np.column_stack([np.ones(n), m.a0 + 0.6 * (m.mmax - m.a0) * rng.random(n)])
    rs = rng.random(4 * m.nt * n)
    modal = lib.simulate(m, sol, init, rs)
    sol.set_choice_draws(True)
    drawn = lib.simulate(m, sol, init, rs)
    sol.set_choice_draws(False)
    cc = cd.ChoiceCells(sol, m)
    ai, ti, ist, M, X = ccc.record_points(m, modal)
    cist, w = ccc.corners(m, ist, X)
    inside = ~ccc.below_grid(m, X) & np.all(np.stack([X[:, k] <= m.s[j]["grid"][-1] for k, j in enumerate(ccc.cont_vars(m))]), axis=0)
    # the modal decision of every kept corner (the thresholds of its merged cell)
    agree = inside.copy()
    for ii in range(cist.shape[0]):
        kept = w[ii] > 0
        for t in np.unique(ti[kept]):
            for s in np.unique(cist[ii][kept & (ti == t)]):
                sel = np.nonzero(kept & (ti == t) & (cist[ii] == s))[0]
                v, _ = cc.policy(int(t), int(s), M[sel])
                g = cc.grid(int(t), int(s))
                agree[sel] &= (v.argmax(axis=0) == modal[ai[sel], ti[sel], cd.DEC]) & (M[sel] >= g[0]) & (M[sel] <= g[1])
    # a record is compared while its agent's path up to it is one the two modes share
    first = np.zeros(n, dtype=bool)
    checked = 0
    for t in range(m.nt):
        sel = np.nonzero(ti == t)[0]
        a = ai[sel]
        ok = agree[sel] & ~first[a]
        first[a[~agree[sel]]] = True
        A, B = modal[a[ok], t], drawn[a[ok], t]
        assert np.array_equal(A[:, [cd.DEC, cd.IST]], B[:, [cd.DEC, cd.IST]])
        np.testing.assert_allclose(B[:, :4], A[:, :4], rtol=0, atol=1e-9)
        checked += int(ok.sum())
    assert checked >= 0.3 * ai.size, (checked, ai.size)


def test_large_likelihood_launch_holds_the_rows_of_a_small_one():
    m, lib, sol = _solved("K2")
    _, sims = ccc.draw_panel(lib, m, sol, 200_000, seed=13)
    obs = ccc.observations(m, sims)
    reps = -(-2_000_000 // obs.shape[0])
    big = np.tile(obs, (reps, 1))[:2_000_000]
    dev = torch.device("cuda", 0)
    out = []
    for o in (big, big[:1024]):
        d_obs = torch.from_numpy(np.ascontiguousarray(o.ravel(order="F"))).to(dev)
        d_tot = torch.zeros(1, dtype=torch.float64, device=dev)
        d_rows = torch.full((o.shape[0],), 7.0, dtype=torch.float64, device=dev)
        lib.choice_loglik_device(m, sol, d_obs.data_ptr(), o.shape[0], o.shape[1], d_tot.data_ptr(), sigma_c=SIGMA_C,
                                 d_rowll=d_rows.data_ptr())
        torch.cuda.synchronize()
        out.append(d_rows[:1024].cpu().numpy())
    assert np.all(np.isfinite(out[0]))
    assert np.array_equal(out[0].view(np.int64), out[1].view(np.int64))


def test_solver_limit_and_equations_with_a_continuous_state():
    m, lib, sol = _solved("K1", sigma_eps=1e-8)
    g = load("humancapital")
    e = solution_errors(sol.M, sol.D, g["M"], g["D"])
    assert e["C"] < 1e-6 and e["V"] < 1e-6 and e["TH"] < 1e-6 and e["Dseq"], e
    m, lib, sol = _solved("K1", sigma_eps=0.2, T=5, ngridm=300, ngridmax=900, ny=5, nz=5)
    for it in (3, 2, 0):
        w = ccc.euler_bellman_residuals_humancapital(sol, m, it)
        assert w["euler"] < 1e-8 and w["bellman"] < 1e-7 and w["points"] > 1000, (it, w)


def test_a_cached_solution_object_solves_after_a_smaller_plan():
    """A released solution object is taken from the cache by the next solve of its shape; the solve kernel's shared
    memory limit set by a smaller model's plan in between must not refuse its launch."""
    m1 = examples.humancapital_smooth(sigma_eps=0.2)
    m1.compile()
    lib = m1._capi()
    s1 = lib.solve(m1, strict=True)
    want = s1.M
    del s1  # released into the cache
    m2 = examples.humancapital_smooth(sigma_eps=0.2, T=5, ngridm=300, ngridmax=900, ny=5)
    m2.prepare()
    lib.solve(m2, strict=True)
    got = lib.solve(m1, strict=True).M
    for a, b in zip(want, got):
        for x, y in zip(a, b):
            assert (x is None and y is None) or np.array_equal(x, y)


def test_bhhh_recovers_duw_and_gain():
    m = examples.humancapital_smooth(sigma_eps=0.2)
    m.compile()
    m.solve()
    lib = m._capi()
    _, sims = ccc.draw_panel(lib, m, m._solution, 200_000, seed=606)
    obs, start = capi.observations_from_sims(m, sims, start=True)
    obs[:, -1] += np.random.default_rng(607).normal(0.0, SIGMA_C, obs.shape[0])
    names = [p["ref"] for p in m.param]
    idx = [names.index("duw"), names.index("gain")]
    truth = m.param_vector()[idx]
    before = m.param_vector()
    m.setparam("duw", 0.46, "gain", 0.17)
    try:
        est, se, total, grad, opg, it = m.fit(obs, start, ["duw", "gain"], sigma_c=SIGMA_C, tol=FIT_TOL)
    finally:
        m.setparam(before)
    z = (est - truth) / se
    print("BHHH (duw, gain) from (0.46, 0.17): %d iterations, total %.6f, estimates %s, truth %s, OPG SE %s, z %s"
          % (it, total, np.array2string(est, precision=6), np.array2string(truth, precision=6),
             np.array2string(se, precision=6), np.array2string(z, precision=3)))
    assert np.all(np.abs(z) < 3.0), (est, se, z)
