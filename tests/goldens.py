"""Load the golden vectors of tests/golden/ (outputs of the unmodified reference C on its own example
models, written by tests/golden/make_golden.py in the development container)."""
import os

import numpy as np

from egdst_b200 import examples
from tests.stored import SampledSims

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")

# name -> keyword overrides used when the vectors were generated (must match make_golden.CASES)
CASES = {
    "cake1": {}, "cake2": {}, "deaton1": {}, "deaton2": {}, "retirement1": {}, "retirement2": {}, "occ3": {},
    "model2": dict(T=8, sigma=0.25, duw=float(np.log(5.0)), ngridm=60, nquad=8),
    "humancapital": {},  # continuous state (not a shipped example: the reference ships none with one)
}
MODELS = dict(examples.ALL, **examples.EXTRA)


def model_for(name):
    return MODELS[name](**CASES[name])


def load(name):
    """Returns dict(M, D nested [ist][it]; init; randstream; sims [nsim, nt, nsimout])."""
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    nst, nt = int(z["nst"]), int(z["nt"])
    M = [[None] * nt for _ in range(nst)]
    D = [[None] * nt for _ in range(nst)]
    for ist in range(nst):
        for it in range(nt):
            k = "M_%d_%d" % (ist, it)
            if k in z.files:
                M[ist][it] = z[k]
                D[ist][it] = z["D_%d_%d" % (ist, it)]
    # columns of the simulation record the reference leaves unassigned for this model (the value column when a state is
    # continuous, egdst_simulator.c:343 with policy(...,0)): NaN in the fixture, ignored by sims_errors
    skip = [int(c) for c in z["skipcols"]] if "skipcols" in z.files else []
    return {"M": M, "D": D, "init": z["init"], "randstream": z["randstream"], "sims": z["sims"], "nst": nst, "nt": nt,
            "skipcols": skip}


def paired(sa, sb):
    """(sa, sb, period): the two simulations on the records ``sb`` holds, as [n, k, nsimout] arrays, and the period of
    each record.  A stored ``SampledSims`` holds k = 1 record per row."""
    if isinstance(sb, SampledSims):
        return sb.pick(sa)[:, None, :], sb.records[:, None, :], sb.periods[:, None]
    return sa, sb, np.broadcast_to(np.arange(sb.shape[1]), sb.shape[:2])


def sims_errors(sa, sb, skipcols=()):
    """Compare two [nsim, nt, nsimout] simulation arrays: NaN pattern, discrete columns (id=4, ist=5)
    exactly, everything else |d|/max(1,|f|).  ``skipcols`` are left out of the comparison.  ``sb`` may be the stored
    records of a simulation (tests/stored.py): the same records of ``sa`` are compared then."""
    sa, sb, _ = paired(sa, sb)
    if len(skipcols):
        sa, sb = sa.copy(), sb.copy()
        sa[:, :, list(skipcols)] = 0.0
        sb[:, :, list(skipcols)] = 0.0
    nan_a, nan_b = np.isnan(sa), np.isnan(sb)
    out = {"nan_mismatch": int((nan_a ^ nan_b).sum())}
    both = ~(nan_a | nan_b)
    d = np.zeros_like(sa)
    with np.errstate(invalid="ignore"):
        fin = both & np.isfinite(sa) & np.isfinite(sb)
        d[fin] = np.abs(sa[fin] - sb[fin]) / np.maximum(1.0, np.abs(sb[fin]))
        inf_mismatch = both & ~fin & (sa != sb)
    out["inf_mismatch"] = int(inf_mismatch.sum())
    out["discrete_mismatch"] = int(((sa[:, :, 4] != sb[:, :, 4]) & both[:, :, 4]).sum() + ((sa[:, :, 5] != sb[:, :, 5]) & both[:, :, 5]).sum())
    out["max"] = float(d.max()) if d.size else 0.0
    return out
