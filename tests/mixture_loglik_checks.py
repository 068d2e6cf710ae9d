"""Checks of the finite-mixture log-likelihood (egdst_mixture_loglik), shared by the emulated (CPU) and the GPU tests.
The numpy oracle starts from the row values of ``choice_loglik(rows=True)`` (pinned by tests/choice_loglik_checks.py):
math.fsum per individual, then a log-sum-exp over the types with positive weight."""
import math

import numpy as np


def oracle(rowll, start, tvec, w):
    """(indll [nvec, nind], mixll [nmix, nind], post [nmix, ntypes, nind], totals [nmix]) from rowll [nvec, nobs]."""
    start = np.asarray(start)
    tvec = np.atleast_2d(np.asarray(tvec))
    w = np.atleast_2d(np.asarray(w, dtype=np.float64))
    nvec, nind = rowll.shape[0], start.size - 1
    indll = np.array([[math.fsum(rowll[v, start[i]:start[i + 1]]) for i in range(nind)] for v in range(nvec)]).reshape(nvec, nind)
    nmix, ntypes = tvec.shape
    mixll = np.empty((nmix, nind))
    post = np.zeros((nmix, ntypes, nind))
    for x in range(nmix):
        pos = w[x] > 0
        a = np.log(w[x, pos] / w[x].sum())[:, None] + indll[tvec[x, pos]]
        m = a.max(axis=0)
        with np.errstate(invalid="ignore", divide="ignore"):
            e = np.exp(a - m)
            s = e.sum(axis=0)
            mixll[x] = np.where(m == -np.inf, -np.inf, m + np.log(s))
            post[x, pos] = np.where(m == -np.inf, np.nan, e / s)
    tot = np.array([math.fsum(r) if np.all(np.isfinite(r)) else np.sum(r) for r in mixll])
    return indll, mixll, post, tot


def check_against_oracle(lib, m, sol, obs, start, tvec, w, sigma_c=0.0, ivec0=0, nvec=None, tol=1e-12):
    """mixture_loglik against the oracle built from choice_loglik rows of the same window.  Returns the outputs."""
    tot, indll, mixll, post = lib.mixture_loglik(m, sol, obs, start, tvec, w, sigma_c=sigma_c, ivec0=ivec0, nvec=nvec,
                                                 individuals=True, posterior=True)
    _, rowll = lib.choice_loglik(m, sol, obs, sigma_c=sigma_c, ivec0=ivec0, nvec=nvec, rows=True)
    want = oracle(rowll, start, tvec, w)
    for got, exp, name in zip((indll, mixll, post), want[:3], ("indll", "mixll", "post")):
        assert got.shape == exp.shape, (name, got.shape, exp.shape)
        np.testing.assert_allclose(got, exp, rtol=tol, atol=tol, equal_nan=True, err_msg=name)
    for t, r, e in zip(tot, mixll, want[3]):
        if np.isfinite(e):
            assert abs(t - math.fsum(r)) <= tol * abs(e) + tol and abs(t - e) <= tol * abs(e) + tol, (t, e)
        else:
            assert np.array_equal([t], [e], equal_nan=True), (t, e)
    return tot, indll, mixll, post


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)
