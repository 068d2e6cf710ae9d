"""Checks of the central-difference mixture scores (egdst_mixture_scores), shared by the emulated (CPU) and the GPU
tests.  The oracle starts from the per-individual mixture values of ``mixture_loglik(individuals=True)`` (pinned by
tests/mixture_loglik_checks.py): the scores are the same IEEE operations in numpy, and the gradient and the OPG are
math.fsum over the numpy products."""
import math

import numpy as np

from tests.mixture_loglik_checks import bits


def stencil(theta, idx, step=1e-4):
    """Central-difference stencil of ``EgdstModel.scores``: (param matrix [2P+1, nparam], mplus, mminus, hinv)."""
    npar = len(idx)
    pv = np.tile(np.asarray(theta, dtype=np.float64), (2 * npar + 1, 1))
    for p, j in enumerate(idx):
        h = step * max(abs(theta[j]), 1.0)
        pv[1 + 2 * p, j] += h
        pv[2 + 2 * p, j] -= h
    mplus, mminus = 1 + 2 * np.arange(npar), 2 + 2 * np.arange(npar)
    return pv, mplus, mminus, 1.0 / (pv[mplus, idx] - pv[mminus, idx])


def one_type(nvec):
    """One-type mixtures of weight 1, one per vector: (tvec, weights)."""
    return np.arange(nvec).reshape(nvec, 1), np.ones((nvec, 1))


def same(a, b):
    """Equal bits, except that any NaN matches any NaN (the payload of inf - inf differs between CPU and GPU)."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    if a.shape != b.shape or not np.array_equal(np.isnan(a), np.isnan(b)):
        return False
    ok = ~np.isnan(a)
    return np.array_equal(bits(a[ok]), bits(b[ok]))


def oracle_sums(sc):
    """(grad [P], opg [P, P]) by math.fsum from scores [P, nind]."""
    npar = sc.shape[0]
    grad = np.array([math.fsum(r) if np.all(np.isfinite(r)) else np.sum(r) for r in sc])
    opg = np.empty((npar, npar))
    for p in range(npar):
        for q in range(npar):
            t = sc[p] * sc[q]
            opg[p, q] = math.fsum(t) if np.all(np.isfinite(t)) else np.sum(t)
    return grad, opg


def close(got, want, tol):
    got, want = np.asarray(got), np.asarray(want)
    fin = np.isfinite(want)
    assert np.array_equal(np.isnan(got), np.isnan(want)), (got, want)
    assert np.all(np.abs(got[fin] - want[fin]) <= tol * np.abs(want[fin]) + 1e-300), (got, want)


def check_against_oracle(lib, m, sol, obs, start, tvec, w, mplus, mminus, hinv, sigma_c=0.0, ivec0=0, nvec=None,
                         tol=1e-12):
    """mixture_scores against the oracle built from the mixll of mixture_loglik over the same mixtures.  Returns
    (totals, grad, opg, scores, mixll)."""
    tot, grad, opg, sc = lib.mixture_scores(m, sol, obs, start, tvec, w, mplus, mminus, hinv, sigma_c=sigma_c, ivec0=ivec0,
                                            nvec=nvec, scores=True)
    t2, _, mixll = lib.mixture_loglik(m, sol, obs, start, tvec, w, sigma_c=sigma_c, ivec0=ivec0, nvec=nvec, individuals=True)
    assert same(tot, t2)
    mplus, mminus = np.asarray(mplus), np.asarray(mminus)
    with np.errstate(invalid="ignore"):
        want = (mixll[mplus] - mixll[mminus]) * np.asarray(hinv, dtype=np.float64)[:, None]
    assert same(sc, want)
    g, o = oracle_sums(want)
    close(grad, g, tol)
    close(opg, o, tol)
    assert same(opg, opg.T)
    return tot, grad, opg, sc, mixll
