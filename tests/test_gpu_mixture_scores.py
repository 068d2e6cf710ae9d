"""Central-difference mixture scores (egdst_mixture_scores) on the GPU at full size (retirement2_smooth,
sigma_eps = 0.2, Philox draw panels): the oracle of tests/score_checks.py, large launches against small ones, the
score and the information-matrix equality at the truth, BHHH recovery (EgdstModel.fit), and the type-share score
against the posterior identity."""
import numpy as np
import pytest

from egdst_b200 import capi, examples
from tests import choice_loglik_checks as cl
from tests import score_checks as sc
from tests.test_gpu_mixture_loglik import _mixed_panel, _two_types

pytestmark = pytest.mark.gpu

FREE = ["duw", "wage", "interest"]
SIGMA_C = 0.05
TRUTH_AGENTS = 200_000
# Tolerances of the truth panel, set from the first run on a B200 and not to be loosened: the largest
# |opg_pq + H_pq| / sqrt(opg_pp opg_qq) over the three parameters (the information-matrix equality; 0.0016 observed,
# OPG / -H between 0.9984 and 1.0015), and the largest relative difference of the OPG and the curvature standard errors
# at the BHHH estimate (0.0019 observed, for wage; 0.0001 for duw).
IME_TOL = 0.01
SE_TOL = 0.02
# BHHH stopping rule for the truth panel.  With the default 1e-8 the first run reached (0.49971, 1.04995) at
# g' OPG^-1 g = 1.45e-7 and then found no improving step length: that criterion is a distance of 4e-4 standard errors
# from the optimum, where the numerical noise of the totals (about 6.3e6 here) outweighs the remaining gain.
FIT_TOL = 1e-6

_CACHE = {}


def _truth():
    """The model at its defaults (compiled, solved) and a TRUTH_AGENTS draw panel whose consumption column carries
    N(0, SIGMA_C^2) measurement error, so that sigma_c = SIGMA_C is correctly specified."""
    if "truth" not in _CACHE:
        m = examples.retirement2_smooth(sigma_eps=0.2)
        m.compile()
        m.solve()
        lib = m._capi()
        _, sims = cl.recovery_panel(lib, m, m._solution, TRUTH_AGENTS, seed=606)
        obs, start = capi.observations_from_sims(m, sims, start=True)
        obs[:, 4] += np.random.default_rng(607).normal(0.0, SIGMA_C, obs.shape[0])
        _CACHE["truth"] = (m, lib, obs, start)
    return _CACHE["truth"]


def _index(m, free):
    names = [p["ref"] for p in m.param]
    return [names.index(f) for f in free]


def _hessian(m, lib, obs, start, theta, idx, rel=1e-3):
    """H of the total at theta from second differences over 1 + 2P + 4 P(P-1)/2 vectors in one batch (19 for P = 3),
    with h_p = rel * max(|theta_p|, 1)."""
    npar = len(idx)
    h = np.array([rel * max(abs(theta[j]), 1.0) for j in idx])
    rows, pairs = [np.zeros(npar)], []
    for p in range(npar):
        e = np.zeros(npar)
        e[p] = h[p]
        rows += [e, -e]
    for p in range(npar):
        for q in range(p + 1, npar):
            for a, b in ((1, 1), (1, -1), (-1, 1), (-1, -1)):
                e = np.zeros(npar)
                e[p], e[q] = a * h[p], b * h[q]
                rows.append(e)
            pairs.append((p, q))
    pv = np.tile(theta, (len(rows), 1))
    pv[:, idx] += np.array(rows)
    sol = lib.solve_batch(m, pv)
    tv, w = sc.one_type(len(rows))
    f = lib.mixture_loglik(m, sol, obs, start, tv, w, sigma_c=SIGMA_C)
    assert np.all(np.isfinite(f)), f
    H = np.empty((npar, npar))
    for p in range(npar):
        H[p, p] = (f[1 + 2 * p] - 2.0 * f[0] + f[2 + 2 * p]) / h[p] ** 2
    for k, (p, q) in enumerate(pairs):
        c = f[1 + 2 * npar + 4 * k:5 + 2 * npar + 4 * k]
        H[p, q] = H[q, p] = (c[0] - c[1] - c[2] + c[3]) / (4.0 * h[p] * h[q])
    return H


def test_oracle_and_large_launches_against_small_ones():
    m, lib = _truth()[:2]
    idx = _index(m, FREE)
    pv, mplus, mminus, hinv = sc.stencil(m.param_vector(), idx)
    sol = lib.solve_batch(m, pv)
    tv, w = sc.one_type(pv.shape[0])
    obs, sims = cl.recovery_panel(lib, m, m._solution, 20_000, seed=41)
    _, start = capi.observations_from_sims(m, sims, start=True)
    _, grad, opg, s, _ = sc.check_against_oracle(lib, m, sol, obs, start, tv, w, mplus, mminus, hinv, sigma_c=SIGMA_C)
    assert np.all(np.isfinite(s)) and np.all(np.linalg.eigvalsh(opg) > 0)
    obs, sims = cl.recovery_panel(lib, m, m._solution, 100_000, seed=42)
    _, start = capi.observations_from_sims(m, sims, start=True)
    big = lib.mixture_scores(m, sol, obs, start, tv, w, mplus, mminus, hinv, sigma_c=SIGMA_C, scores=True)
    small = 1024
    sm = lib.mixture_scores(m, sol, obs[:start[small]], start[:small + 1], tv, w, mplus, mminus, hinv, sigma_c=SIGMA_C,
                            scores=True)
    assert sc.same(big[3][:, :small], sm[3])
    np.testing.assert_allclose(big[1], big[3].sum(axis=1), rtol=1e-10)


def test_score_and_information_at_the_truth():
    m, lib, obs, start = _truth()
    total, grad, opg = m.scores(obs, start, FREE, sigma_c=SIGMA_C)
    z = grad / np.sqrt(np.diag(opg))
    H = _hessian(m, lib, obs, start, m.param_vector(), _index(m, FREE))
    d = 1.0 / np.sqrt(np.diag(opg))
    ime = (opg + H) * d[:, None] * d[None, :]
    print("truth panel: %d individuals, %d rows, total %.6f" % (start.size - 1, obs.shape[0], total))
    print("score z (duw, wage, interest): %s" % np.array2string(z, precision=3))
    print("OPG / -H (elementwise):\n%s" % np.array2string(opg / -H, precision=4))
    print("max |opg + H| / sqrt(opg_pp opg_qq) = %.4f" % np.abs(ime).max())
    assert np.all(np.abs(z) < 4.0), z
    assert np.abs(ime).max() < IME_TOL, ime


def test_bhhh_recovers_duw_and_wage():
    m, lib, obs, start = _truth()
    truth = m.param_vector()
    idx = _index(m, ["duw", "wage"])
    before = m.param_vector()
    m.setparam("duw", 0.6, "wage", 1.155)
    try:
        est, se, total, grad, opg, it = m.fit(obs, start, ["duw", "wage"], sigma_c=SIGMA_C, tol=FIT_TOL)
        assert np.array_equal(m.param_vector()[idx], [0.6, 1.155])
    finally:
        m.setparam(before)
    theta = truth.copy()
    theta[idx] = est
    H = _hessian(m, lib, obs, start, theta, idx)
    se_curv = np.sqrt(np.diag(np.linalg.inv(-H)))
    print("BHHH (duw, wage) from (0.6, 1.155): %d iterations, total %.6f" % (it, total))
    print("  estimates %s, truth %s" % (np.array2string(est, precision=6), np.array2string(truth[idx], precision=6)))
    print("  OPG SE %s, curvature SE %s, (est - truth) / SE %s" % (
        np.array2string(se, precision=6), np.array2string(se_curv, precision=6),
        np.array2string((est - truth[idx]) / se, precision=3)))
    print("  OPG SE / curvature SE - 1: %s" % np.array2string(se / se_curv - 1.0, precision=4))
    assert it <= 100
    assert np.all(np.abs(est - truth[idx]) < 4.0 * se), (est, se)
    assert np.all(np.abs(se / se_curv - 1.0) < SE_TOL), (se, se_curv)


def test_type_share_score_is_the_posterior_identity():
    m, lib, sol = _two_types()
    obs, start, _ = _mixed_panel(lib, m, sol, 20_000, 0.3, seed=77)
    pi, h = 0.3, 1e-4
    tv = [[0, 1]] * 3
    w = [[pi, 1 - pi], [pi + h, 1 - pi - h], [pi - h, 1 - pi + h]]
    _, _, _, s, _ = sc.check_against_oracle(lib, m, sol, obs, start, tv, w, [1], [2], [1.0 / ((pi + h) - (pi - h))],
                                            sigma_c=SIGMA_C)
    _, post = lib.mixture_loglik(m, sol, obs, start, [0, 1], [pi, 1 - pi], sigma_c=SIGMA_C, posterior=True)
    want = post[0, 0] / pi - post[0, 1] / (1 - pi)
    err = np.abs(s[0] - want) / np.maximum(np.abs(want), 1.0)
    print("type-share score against post_0/pi - post_1/(1-pi): max relative error %.3g" % err.max())
    assert err.max() < 1e-6, err.max()
