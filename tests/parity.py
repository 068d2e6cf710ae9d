"""Function-space parity metrics between two solutions (SURVEY 8(c) protocol).

Row counts may differ by a row or two where a discrete branch (fold test, stop rule, tie) flips on
the last ulp (SURVEY 7, hard part 3), so policies and values are compared as *functions*: both
solutions' C(M), V(M) are interpolated on a common probe grid over the overlap of their M ranges,
excluding +-excl = 1e-9 neighbourhoods of thresholds and double points (where C jumps; SURVEY 8c); error = |d| / max(1, |f|).
Thresholds, evf(a0) (row 0 of V) and the decision sequence are compared directly.
"""
import numpy as np

from tests.stored import NOT_SAMPLED, SampledCell


def _interp(M, F, x):
    # rows 1.. (row 0 is the a0 row: V there is evf(a0), not a value)
    return np.interp(x, M[1:, 0], F)


def _gap(a, b):
    """max |a-b| / max(1,|b|) over the probes.  Probes where both sides are the SAME infinity or both NaN agree (the
    reference writes C = -inf rows in places, e.g. the second half of a double point on an analytic segment); a probe
    where only one side is non-finite, or the infinities differ, is a mismatch (inf) -- never silently skipped."""
    if a.size == 0:
        return 0.0
    fa, fb = np.isfinite(a), np.isfinite(b)
    same_nonfinite = (~fa & ~fb) & ((a == b) | (np.isnan(a) & np.isnan(b)))
    if np.any((~fa | ~fb) & ~same_nonfinite):
        return float("inf")
    both = fa & fb
    return float(np.max(np.abs(a[both] - b[both]) / np.maximum(1.0, np.abs(b[both])))) if both.any() else 0.0


def cell_errors(Ma, Da, Mb, Db, nprobe=50001, excl=1e-9):
    """``Mb`` may be a stored SampledCell (tests/stored.py): its sampled rows are the probes then."""
    sampled = isinstance(Mb, SampledCell)
    if sampled:
        out = {"range_lo": 0.0, "range_hi": 0.0}
        x = Mb.x
        mask = (x >= Ma[1, 0]) & (x <= Ma[-1, 0])
    else:
        lo = max(Ma[1, 0], Mb[1, 0])
        hi = min(Ma[-1, 0], Mb[-1, 0])
        out = {"range_lo": abs(Ma[1, 0] - Mb[1, 0]), "range_hi": abs(Ma[-1, 0] - Mb[-1, 0])}
        x = np.linspace(lo, hi, nprobe)
        mask = np.ones_like(x, dtype=bool)
    for th in np.concatenate([Da[:, 1], Db[:, 1]]):
        mask &= np.abs(x - th) > excl
    # also stay away from each solution's own double points (secondary-envelope kinks insert them too)
    for M in ((Ma,) if sampled else (Ma, Mb)):
        dm = np.diff(M[1:, 0])
        for xd in M[1:-1, 0][dm < 1e-9]:
            mask &= np.abs(x - xd) > excl
    x = x[mask]
    ca, va = _interp(Ma, Ma[1:, 1], x), _interp(Ma, Ma[1:, 3], x)
    if sampled:
        cb, vb = Mb.c[mask], Mb.v[mask]
    else:
        cb, vb = _interp(Mb, Mb[1:, 1], x), _interp(Mb, Mb[1:, 3], x)
    out["C"] = _gap(ca, cb)
    out["V"] = _gap(va, vb)
    ea, eb = Ma[0, 3], (Mb.evf if sampled else Mb[0, 3])
    out["evf"] = 0.0 if (ea == eb or (np.isinf(ea) and np.isinf(eb) and ea == eb)) else float(abs(ea - eb) / max(1.0, abs(eb)))
    out["nth"] = (Da.shape[0], Db.shape[0])
    if Da.shape[0] == Db.shape[0]:
        out["TH"] = float(np.max(np.abs(Da[:, 1] - Db[:, 1])))
        out["Dseq"] = bool(np.all(Da[:, 0] == Db[:, 0]))
    else:
        out["TH"] = float("inf")
        out["Dseq"] = False
    out["rows"] = (Ma.shape[0], Mb.nrows if sampled else Mb.shape[0])
    return out


def solution_errors(Ma, Da, Mb, Db, **kw):
    """Worst case over all (ist, it) cells; Ma/Da = candidate, Mb/Db = oracle."""
    worst = {"C": 0.0, "V": 0.0, "evf": 0.0, "TH": 0.0, "Dseq": True, "rowdiff": 0, "cells": 0, "where": {}}
    for ist in range(len(Mb)):
        for it in range(len(Mb[ist])):
            a, b = Ma[ist][it], Mb[ist][it]
            if b is NOT_SAMPLED:
                assert a is not None and a.size, "candidate lacks cell (ist=%d,it=%d)" % (ist, it)
                continue
            if b is None or b.size == 0:
                assert a is None or a.size == 0, "candidate has a solution where the oracle has none"
                continue
            assert a is not None, "candidate lacks cell (ist=%d,it=%d)" % (ist, it)
            e = cell_errors(a, Da[ist][it], b, Db[ist][it], **kw)
            worst["cells"] += 1
            for k in ("C", "V", "evf", "TH"):
                if e[k] > worst[k]:
                    worst[k] = e[k]
                    worst["where"][k] = (ist, it)
            worst["Dseq"] = worst["Dseq"] and e["Dseq"]
            worst["rowdiff"] = max(worst["rowdiff"], abs(e["rows"][0] - e["rows"][1]))
    return worst
