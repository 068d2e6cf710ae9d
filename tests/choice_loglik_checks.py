"""Checks of the choice log-likelihood of the smoothing mode (egdst_choice_loglik), shared by the emulated (CPU) and
the GPU tests.  The probabilities are those of choice_draw_checks.ChoiceCells (numpy interpolants of the exported
choice cells, valid inside every decision's grid); below the first grid point numpy restates the credit-constrained
branch, v_d(M) = u(M - a0, d) + discount * evf_d with evf_d = row 0 of the choice cell."""
import math

import numpy as np

from egdst_b200 import capi
from tests import choice_draw_checks as cd

LOG_SQRT_2PI = 0.5 * math.log(2.0 * math.pi)


def interior_obs(cc, sims, consumption=False):
    """Observations of the records that choice_draw_checks.interior_records keeps, and their (agent, it)."""
    ai, ti = cd.interior_records(cc, sims)
    rec = sims[ai, ti]
    cols = [cc.m.t0 + ti.astype(float), rec[:, cd.IST] + 1, rec[:, cd.CASH], rec[:, cd.DEC] + 1]
    if consumption:
        cols.append(rec[:, cd.CONS])
    return np.column_stack(cols), ai, ti


def numpy_logp(cc, obs):
    """log P_d(M) of every row by ChoiceCells.probabilities (rows inside the grid only)."""
    out = np.full(obs.shape[0], np.nan)
    it_all = (obs[:, 0] - cc.m.t0).astype(int)
    ist_all = obs[:, 1].astype(int) - 1
    for it in np.unique(it_all):
        for ist in np.unique(ist_all[it_all == it]):
            sel = np.nonzero((it_all == it) & (ist_all == ist))[0]
            P = cc.probabilities(int(it), int(ist), obs[sel, 2])
            with np.errstate(divide="ignore"):
                out[sel] = np.log(P[obs[sel, 3].astype(int) - 1, np.arange(sel.size)])
    return out


def constrained_logp(cc, lib, it, ist, M):
    """[nd, n] log P_d(M) for cash M below every available decision's M[1] (the credit-constrained branch)."""
    m, sol = cc.m, cc.sol
    M = np.asarray(M, dtype=np.float64)
    age = m.t0 + it
    v = np.full((m.nd, M.size), -np.inf)
    df = lib.call(m, sol, 3, np.column_stack([np.full(M.size, age), np.full(M.size, ist + 1)]))
    for d, cell in enumerate(cc.cells(it, ist)):
        if cell is None or cell.shape[0] < 3:
            continue
        assert np.all(M < cell[1, 0])
        u = lib.call(m, sol, 1, np.column_stack([np.full(M.size, age), np.full(M.size, ist + 1), np.full(M.size, d + 1), M - m.a0]))
        v[d] = u + df * cell[0, 3]
    z = v / m.sigma_eps
    z = z - z.max(axis=0)
    return z - np.log(np.exp(z).sum(axis=0))


def check_mechanism(cc, lib, sims, ivec=0, atol=1e-10, min_rows=300):
    """rowll of the interior records equals log of the numpy probability at the observed decision.  Returns rows."""
    obs, _, _ = interior_obs(cc, sims)
    assert obs.shape[0] >= min_rows, obs.shape
    tot, rowll = lib.choice_loglik(cc.m, cc.sol, obs, ivec0=ivec, nvec=1, rows=True)
    want = numpy_logp(cc, obs)
    assert np.all(np.isfinite(rowll[0])), np.count_nonzero(~np.isfinite(rowll[0]))
    np.testing.assert_allclose(rowll[0], want, rtol=0, atol=atol)
    check_total(tot[0], rowll[0])
    return obs.shape[0]


def check_total(total, rowll, rtol=1e-12):
    want = math.fsum(rowll)
    assert abs(total - want) <= rtol * abs(want), (total, want)


def consumption_terms(lib, m, sol, obs, sigma_c):
    """rowll with the consumption term minus rowll without it, and the per-row rowll of k = 4 and of (k = 5, sigma_c = 0)."""
    _, with_c = lib.choice_loglik(m, sol, obs, sigma_c=sigma_c, rows=True)
    _, k4 = lib.choice_loglik(m, sol, obs[:, :4], sigma_c=sigma_c, rows=True)
    _, s0 = lib.choice_loglik(m, sol, obs, sigma_c=0.0, rows=True)
    return with_c[0] - k4[0], k4[0], s0[0]


def recovery_panel(lib, m, sol, n, seed):
    """Observations (with consumption) of a Philox draw simulation of n agents."""
    rng = np.random.default_rng(seed)
    init = np.column_stack([np.ones(n), m.a0 + 0.6 * (m.mmax - m.a0) * rng.random(n)])
    sol.set_choice_draws(True)
    try:
        sims, _ = lib.simulate_philox(m, sol, init, seed=seed)
    finally:
        sol.set_choice_draws(False)
    return capi.observations_from_sims(m, sims), sims
