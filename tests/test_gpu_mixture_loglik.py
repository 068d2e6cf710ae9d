"""Finite-mixture log-likelihood over unobserved types (egdst_mixture_loglik) on the GPU at full size
(retirement2_smooth, sigma_eps = 0.2): the numpy oracle of tests/mixture_loglik_checks.py on a two-type draw panel,
large launches against small ones, and the recovery of a type share by grid search and by EM on the posteriors."""
import numpy as np
import pytest

from egdst_b200 import capi, examples
from tests import choice_loglik_checks as cl
from tests import mixture_loglik_checks as mc

pytestmark = pytest.mark.gpu

DUW = (0.35, 0.65)
# Type-share recovery: 30 % of REC_AGENTS agents of type 0, with the consumption term (REC_SIGMA_C).  The panel size
# and the tolerances (|pi - 0.3| < 4 SE, SE < 0.02) were set from the first run on a B200 and are not to be loosened.
# That run used the choices alone and found pi = 0.2888 at SE 0.0031 (-3.6 SE): the choice probabilities condition on
# the observed cash, whose path depends on the type through consumption, so a choices-only mixture leaves out a
# type-dependent factor and its share estimate is biased.  The consumption term carries that information; with it the
# same panel gives pi = 0.2995 at SE 0.0023 (-0.2 SE).
REC_AGENTS = 40_000
REC_SHARE = 0.3
REC_SIGMA_C = 0.05


def _two_types():
    m = examples.retirement2_smooth(sigma_eps=0.2)
    m.compile()
    lib = m._capi()
    names = [p["ref"] for p in m.param]
    pv = np.array([list(m.param_vector())] * len(DUW))
    pv[:, names.index("duw")] = DUW
    sol = lib.solve_batch(m, pv)
    for v in range(len(DUW)):
        assert sol.status(v)[0] == 0, (v, sol.status(v))
    return m, lib, sol


def _mixed_panel(lib, m, sol, n, share, seed):
    """Philox draw panel: the first round(share * n) agents simulated under vector 0, the others under vector 1, with
    disjoint agent0 ranges.  Returns (obs, start, n0)."""
    n0 = int(round(share * n))
    rng = np.random.default_rng(seed)
    init = np.column_stack([np.ones(n), m.a0 + 0.6 * (m.mmax - m.a0) * rng.random(n)])
    sol.set_choice_draws(True)
    try:
        s0, _ = lib.simulate_philox(m, sol, init[:n0], seed=seed, agent0=0, ivec=0)
        s1, _ = lib.simulate_philox(m, sol, init[n0:], seed=seed, agent0=n0, ivec=1)
    finally:
        sol.set_choice_draws(False)
    obs, start = capi.observations_from_sims(m, np.concatenate([s0, s1]), start=True)
    return obs, start, n0


def test_oracle_on_a_two_type_panel():
    m, lib, sol = _two_types()
    obs, start, _ = _mixed_panel(lib, m, sol, 20_000, 0.5, seed=31)
    tvec = [[0, 1], [1, 0], [0, 0]]
    w = [[0.3, 0.7], [2.0, 5.0], [0.0, 1.0]]
    tot, indll, mixll, post = mc.check_against_oracle(lib, m, sol, obs, start, tvec, w, sigma_c=0.05)
    assert np.all(np.isfinite(tot))
    np.testing.assert_allclose(post.sum(axis=1), 1.0, rtol=0, atol=1e-12)


def test_large_launches_hold_the_individuals_of_small_ones():
    m, lib, sol = _two_types()
    obs, sims = cl.recovery_panel(lib, m, sol, 100_000, seed=11)
    _, start = capi.observations_from_sims(m, sims, start=True)
    assert obs.shape[0] >= 2_000_000, obs.shape
    tvec, w = [[0, 1], [1, 1]], [[0.4, 0.6], [1.0, 1.0]]
    big = lib.mixture_loglik(m, sol, obs, start, tvec, w, sigma_c=0.05, individuals=True, posterior=True)
    small = 1024
    sm = lib.mixture_loglik(m, sol, obs[:start[small]], start[:small + 1], tvec, w, sigma_c=0.05, individuals=True,
                            posterior=True)
    assert np.array_equal(mc.bits(big[1][:, :small]), mc.bits(sm[1]))
    assert np.array_equal(mc.bits(big[2][:, :small]), mc.bits(sm[2]))
    assert np.array_equal(mc.bits(big[3][:, :, :small]), mc.bits(sm[3]))
    assert np.all(np.isfinite(big[2]))
    np.testing.assert_allclose(big[0], big[2].sum(axis=1), rtol=1e-12, atol=0)


def test_type_share_recovery():
    m, lib, sol = _two_types()
    obs, start, n0 = _mixed_panel(lib, m, sol, REC_AGENTS, REC_SHARE, seed=2024)
    nind = start.size - 1
    assert n0 == int(REC_SHARE * REC_AGENTS) and np.all(np.diff(start) > 0)
    # grid search over the share of type 0
    grid = np.round(np.arange(1, 10) * 0.1, 10)
    tot = lib.mixture_loglik(m, sol, obs, start, [[0, 1]] * grid.size, np.column_stack([grid, 1.0 - grid]),
                             sigma_c=REC_SIGMA_C)
    assert np.all(np.isfinite(tot)), tot
    assert abs(grid[int(np.argmax(tot))] - REC_SHARE) < 1e-9, tot
    # EM on the share from 0.5: pi <- mean posterior of type 0
    pi = 0.5
    for it in range(500):
        _, post = lib.mixture_loglik(m, sol, obs, start, [0, 1], [pi, 1.0 - pi], sigma_c=REC_SIGMA_C, posterior=True)
        new = float(post[0, 0].mean())
        if abs(new - pi) < 1e-10:
            pi = new
            break
        pi = new
    else:
        pytest.fail("EM did not converge: pi = %r" % pi)
    # standard error from the curvature of the total at the estimate, the three mixtures in one launch
    d = 5e-3
    t = lib.mixture_loglik(m, sol, obs, start, [[0, 1]] * 3, [[pi - d, 1 - pi + d], [pi, 1 - pi], [pi + d, 1 - pi - d]],
                           sigma_c=REC_SIGMA_C)
    curv = (t[0] - 2.0 * t[1] + t[2]) / d ** 2
    assert curv < 0, t
    se = 1.0 / np.sqrt(-curv)
    print("type-share recovery: %d individuals, %d EM iterations, pi = %.5f, SE = %.5f, (pi - %.1f) / SE = %.2f" % (
        nind, it + 1, pi, se, REC_SHARE, (pi - REC_SHARE) / se))
    assert se < 0.02, se
    assert abs(pi - REC_SHARE) < 4.0 * se, (pi, se)
    assert t[1] >= max(t[0], t[2]), t
