"""Checks of the choice draws and the choice log-likelihood of smoothing images with continuous states, shared by the
emulated (CPU) and the GPU tests.

numpy restates the corner rule of egdst_choice_values_cont.  At a record's exact continuous state x (record columns
11 + j of the continuous state variables j): the 2^K grid cells around x (egdst_gridcell, linear weights, end
intervals extended outwards), corners with weight <= 0 dropped and the kept weights renormalised to sum 1.  The mixed
values v_d = sum w v_d^corner and c_d = sum w c_d^corner come from np.interp on each corner's exported choice cells
(choice_draw_checks.ChoiceCells), so only records whose cash lies inside every kept corner's grid are restated.  Then
P_d = softmax(v_d / sigma_eps), the drawn decision is the first whose cumulative probability reaches the record's
uniform, and the record holds c = min(c_d, M - a0), v_d and the corner at which the cumulated weight passes 1/2.
"""
import math

import numpy as np

from egdst_b200 import capi
from tests import choice_draw_checks as cd

LOG_SQRT_2PI = 0.5 * math.log(2.0 * math.pi)


def cont_vars(m):
    """Positions in st[] of the continuous state variables (egdst_contvar)."""
    return [j for j, v in enumerate(m.s) if v["continuous"]]


def corners(m, ist, X):
    """For states ist [n] (0-based; their grid part is ignored) and exact values X [n, K]: the corner states [2^K, n]
    and the normalised weights [2^K, n] (0 for dropped corners), in the kernel's corner order."""
    cv = cont_vars(m)
    K = len(cv)
    nnst = len(m.s)
    ist = np.asarray(ist, dtype=np.int64)
    X = np.asarray(X, dtype=np.float64).reshape(ist.size, K)
    base = ist.copy()
    j1, wlo, whi, stride = [], [], [], []
    for k, j0 in enumerate(cv):
        g = np.asarray(m.s[j0]["grid"])
        n, st = int(m.stm[j0]), int(m.stm[nnst + j0])
        base -= ((ist // st) % n) * st
        x = X[:, k]
        j = np.minimum(np.sum(x[:, None] >= g[None, 1:n - 1], axis=1), n - 2)
        j1.append(j)
        wlo.append((g[j + 1] - x) / (g[j + 1] - g[j]))
        whi.append((x - g[j]) / (g[j + 1] - g[j]))
        stride.append(st)
    nc = 1 << K
    cist = np.zeros((nc, ist.size), dtype=np.int64)
    wt = np.ones((nc, ist.size))
    for ii in range(nc):
        cist[ii] = base
        for k in range(K):
            up = (ii >> k) & 1
            wt[ii] *= whi[k] if up else wlo[k]
            cist[ii] += stride[k] * (j1[k] + up)
    wt = np.where(wt > 0, wt, 0.0)
    return cist, wt / wt.sum(axis=0)


class Restated:
    """Mixed choice values, probabilities and recorded corner of a set of points (it [n], ist [n], M [n], X [n, K])."""

    def __init__(self, cc, it, ist, M, X):
        m = cc.m
        it = np.asarray(it, dtype=np.int64)
        M = np.asarray(M, dtype=np.float64)
        self.cist, self.w = corners(m, ist, X)
        n, nd = M.size, m.nd
        self.v, self.c = np.zeros((nd, n)), np.zeros((nd, n))
        self.inside = np.ones(n, dtype=bool)
        for ii in range(self.cist.shape[0]):
            kept = self.w[ii] > 0
            for t in np.unique(it[kept]):
                for s in np.unique(self.cist[ii][kept & (it == t)]):
                    sel = np.nonzero(kept & (it == t) & (self.cist[ii] == s))[0]
                    g = cc.grid(int(t), int(s))
                    if g is None:
                        self.inside[sel] = False
                        continue
                    self.inside[sel] &= (M[sel] >= g[0]) & (M[sel] <= g[1])
                    v, c = cc.policy(int(t), int(s), M[sel])
                    w = self.w[ii, sel]
                    self.v[:, sel] += w * v
                    self.c[:, sel] += w * np.where(np.isfinite(v), c, 0.0)
        z = self.v / m.sigma_eps
        with np.errstate(invalid="ignore"):
            e = np.exp(z - z.max(axis=0))
            self.P = e / e.sum(axis=0)
        # the corner at which the cumulated normalised weight passes 1/2 (else the last kept corner)
        rr = 0.5 - np.cumsum(self.w, axis=0)
        passed = (rr < 0) & (self.w > 0)
        last = self.cist.shape[0] - 1 - np.argmax((self.w > 0)[::-1], axis=0)
        pick = np.where(passed.any(axis=0), np.argmax(passed, axis=0), last)
        self.istrec = self.cist[pick, np.arange(n)]
        self.a0, self.M = m.a0, M

    def consumption(self, d):
        """The recorded consumption min(c_d, M - a0) of decisions d [n]."""
        cols = np.arange(self.M.size)
        return np.minimum(self.c[d, cols], self.M - self.a0)


def record_points(m, sims):
    """(agent, it) of the live records and their (ist, M, X)."""
    alive = ~np.isnan(sims[:, :, cd.CASH])
    ai, ti = np.nonzero(alive)
    rec = sims[ai, ti]
    X = rec[:, [11 + j for j in cont_vars(m)]]
    return ai, ti, rec[:, cd.IST].astype(np.int64), rec[:, cd.CASH], X


def below_grid(m, X):
    """Rows of X [n, K] with some value below its grid."""
    return np.any(np.stack([X[:, k] < m.s[j]["grid"][0] for k, j in enumerate(cont_vars(m))], axis=1), axis=1)


def check_draws(cc, sims, U, margin=1e-9, tol=1e-12):
    """Every restated record (cash inside every kept corner's grid) whose uniform is more than `margin` from a
    cumulative boundary holds the numpy draw, its consumption, savings, value and recorded corner.  Returns (records
    checked, count per decision, records checked with x below the grid)."""
    m = cc.m
    ai, ti, ist, M, X = record_points(m, sims)
    R = Restated(cc, ti, ist, M, X)
    u = U[ai, ti]
    cum = np.cumsum(R.P, axis=0)
    clear = R.inside & np.all(np.abs(cum - u[None, :]) > margin, axis=0)
    d = np.argmax(cum >= u[None, :], axis=0)
    rec = sims[ai, ti]
    sel = np.nonzero(clear)[0]
    assert np.array_equal(rec[sel, cd.DEC], d[sel].astype(float)), np.count_nonzero(rec[sel, cd.DEC] != d[sel])
    np.testing.assert_allclose(rec[sel, cd.CONS], R.consumption(d)[sel], rtol=0, atol=tol)
    np.testing.assert_allclose(rec[sel, cd.VAL], R.v[d[sel], sel], rtol=0, atol=tol)
    np.testing.assert_allclose(rec[sel, cd.SAV], rec[sel, cd.CASH] - rec[sel, cd.CONS], rtol=0, atol=tol)
    assert np.array_equal(rec[sel, cd.IST], R.istrec[sel].astype(float))
    return sel.size, np.bincount(d[sel], minlength=m.nd), int(np.count_nonzero(below_grid(m, X[sel])))


def check_rows(cc, lib, obs, sigma_c=0.0, atol=1e-10):
    """rowll of the restated rows of obs [nobs, 4 + K (+1)] equals log P_d at the observed decision (+ the consumption
    term centred on the recorded consumption).  Returns (rows checked, rows with x below the grid)."""
    m = cc.m
    K = len(cont_vars(m))
    it = (obs[:, 0] - m.t0).astype(np.int64)
    d = obs[:, 3].astype(np.int64) - 1
    X = obs[:, 4:4 + K]
    R = Restated(cc, it, obs[:, 1].astype(np.int64) - 1, obs[:, 2], X)
    tot, rowll = lib.choice_loglik(m, cc.sol, obs, sigma_c=sigma_c, rows=True)
    cols = np.arange(obs.shape[0])
    with np.errstate(divide="ignore"):
        want = np.log(R.P[d, cols])
    if obs.shape[1] == 5 + K and sigma_c > 0:
        z = (obs[:, 4 + K] - R.consumption(d)) / sigma_c
        want = want + np.where(np.isnan(obs[:, 4 + K]), 0.0, -0.5 * z * z - LOG_SQRT_2PI - math.log(sigma_c))
    sel = R.inside
    assert np.all(np.isfinite(rowll[0])), np.count_nonzero(~np.isfinite(rowll[0]))
    np.testing.assert_allclose(rowll[0, sel], want[sel], rtol=0, atol=atol)
    want_tot = math.fsum(rowll[0])
    assert abs(tot[0] - want_tot) <= 1e-12 * abs(want_tot), (tot[0], want_tot)
    return int(sel.sum()), int(np.count_nonzero(below_grid(m, X[sel])))


def draw_panel(lib, m, sol, n, seed, agent0=0, init_seed=None):
    """Philox draw simulation of n agents starting at the first state (z at its lowest grid point) with random cash;
    returns (init, sims)."""
    rng = np.random.default_rng(seed if init_seed is None else init_seed)
    init = np.column_stack([np.ones(n), m.a0 + 0.6 * (m.mmax - m.a0) * rng.random(n)])
    sol.set_choice_draws(True)
    try:
        sims, _ = lib.simulate_philox(m, sol, init, seed=seed, agent0=agent0)
    finally:
        sol.set_choice_draws(False)
    return init, sims


def observations(m, sims, consumption=True, start=False):
    return capi.observations_from_sims(m, sims, consumption=consumption, start=start)


def euler_bellman_residuals_humancapital(sol, m, it):
    """smoothing_checks.euler_bellman_residuals for humancapital_smooth (one continuous state z): next period's z' =
    depr z + gain d is spread over its two grid cells with the linear weights of trpr (compile.m:527-537), and
         rhs = beta (1+r) sum_iy w_iy sum_j' p_j' sum_d' P_d'(M') u'(c_d'(M')),
         ev  = sum_iy w_iy sum_j' p_j' sigma log sum_d' exp(v_d'(M')/sigma),   M' = A (1+r) + wage z shock d,
    at every point of every choice cell of period `it` whose z' and M' (for every node) lie inside the grids."""
    from scipy.stats import norm
    from egdst_b200.quadrature import model_quadrature
    sig = m.sigma_eps
    p = {q["ref"]: q["value"] for q in m.param}
    r, duw, wage, depr, gain = p["interest"], p["duw"], p["wage"], p["depr"], p["gain"]
    beta = 1.0 / (1.0 + r)
    sg = float(m.shock["sigma"])
    q = model_quadrature(m.ny)
    w, shocks = q[:m.ny], np.exp(-0.5 * sg * sg + norm.ppf(q[m.ny:]) * sg)
    g = np.asarray(m.s[0]["grid"])
    cc = cd.ChoiceCells(sol, m)
    worst = {"euler": 0.0, "bellman": 0.0, "points": 0}
    for ist in range(m.nst):
        z = g[ist]
        for d in range(m.nd):
            cell = sol.choice_cell(it, ist, d)
            if cell is None or cell.shape[0] < 3:
                continue
            z1 = depr * z + gain * d
            if not (g[0] <= z1 <= g[-1]):
                continue
            j = min(int(np.sum(z1 >= g[1:-1])), g.size - 2)
            pz = ((j, (g[j + 1] - z1) / (g[j + 1] - g[j])), (j + 1, (z1 - g[j]) / (g[j + 1] - g[j])))
            M, C, A, V = cell[1:, 0], cell[1:, 1], cell[1:, 2], cell[1:, 3]
            rhs, ev = np.zeros_like(M), np.zeros_like(M)
            inside = np.ones_like(M, dtype=bool)
            inside[-1] = False  # the last point of a list cut at the unified grid's bound is interpolated
            for wi, sh in zip(w, shocks):
                M1 = A * (1.0 + r) + wage * z * sh * d
                for j1, pj in pz:
                    if pj == 0.0:
                        continue
                    lo, hi = cc.grid(it + 1, j1)
                    inside &= (M1 >= lo) & (M1 <= hi)
                    v, c = cc.policy(it + 1, j1, M1)
                    vmax = v.max(axis=0)
                    e = np.exp((v - vmax) / sig)
                    P = e / e.sum(axis=0)
                    rhs += wi * pj * np.nansum(np.where(P > 0, P / c, 0.0), axis=0)
                    ev += wi * pj * (vmax + sig * np.log(e.sum(axis=0)))
            rhs *= beta * (1.0 + r)
            euler = np.abs(C - 1.0 / rhs) / np.maximum(1.0, np.abs(C))
            keep = inside & (euler < 1e-4)  # kink points of the secondary envelope satisfy no Euler equation
            assert keep.sum() >= inside.sum() - 6, (it, ist, d, int(keep.sum()), int(inside.sum()))
            if not keep.any():
                continue
            worst["euler"] = max(worst["euler"], float(np.max(euler[keep])))
            bell = np.abs(V[keep] - (np.log(C[keep]) + duw * (d == 0) + beta * ev[keep]))
            worst["bellman"] = max(worst["bellman"], float(np.max(bell)))
            worst["points"] += int(keep.sum())
    return worst
