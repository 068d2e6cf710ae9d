"""Checks of the Philox-driven simulator against the reference simulator's C restatement (oracle/port), shared by the
emulated (CPU) and the GPU tests.

The Philox source of egdst_k_simulate is restated as a reference-layout randstream: slot 3*(it-1)+k of agent i's 4*nt
block is (w_k + 0.5) / 2^32, w_k word k of the Philox4x32-10 block of counter (gid, gid >> 32, it, 0) and key
(seed, seed >> 32), k = 0, 1, 2 and it >= 1 (the transition into period it: state, shock, survival); slot 3*(nt-1)+it
is word 3 of block (gid, it), the choice uniform of period it.  (w + 0.5) / 2^32 is exact in double, so the port
replays the agents on exactly the kernel's uniforms, from the solution's own exported cells: the paths must agree to
the parity bar, and the discrete columns and the NaN pattern exactly.  The moments of every launch are held to exact
sums over the replayed paths, not over the kernel's own paths, which moments-only launches do not have.
"""
import math

import numpy as np

from oracle.port import Port
from tests.choice_draw_checks import philox4x32
from tests.goldens import sims_errors

TOL = 1e-9          # the project's parity bar (|d| / max(1, |f|))
TH_EXCL = 1e-9      # cash this close to a threshold of its cell may pick either decision (the S2 rule, test_gpu_scale)
EDGE_EXCL = 1e-12   # a transition uniform this close to a cumulative trpr boundary may pick either next state
MAX_EXCUSED = 1e-4  # largest share of the live records left out under the two rules above
CASH, DEC, IST = 0, 4, 5


def philox_randstream(nsim, nt, seed, agent0=0):
    """[nsim, 4*nt] randstream (rndtype 0 layout) holding the uniforms the Philox source of egdst_k_simulate draws for
    agents agent0 .. agent0 + nsim - 1 under `seed`."""
    gid = np.arange(nsim, dtype=np.uint64)[:, None] + np.uint64(agent0) + np.zeros((1, nt), dtype=np.uint64)
    it = np.broadcast_to(np.arange(nt, dtype=np.uint64)[None, :], gid.shape)
    seed = int(seed)
    w = philox4x32(gid, gid >> np.uint64(32), it, 0, seed & 0xFFFFFFFF, seed >> 32)
    u = [(x.astype(np.float64) + 0.5) * (1.0 / 4294967296.0) for x in w]
    rs = np.full((nsim, 4 * nt), 0.5)
    if nt > 1:
        rs[:, :3 * (nt - 1)] = np.stack(u[:3], axis=2)[:, 1:, :].reshape(nsim, 3 * (nt - 1))
    rs[:, 3 * (nt - 1):3 * (nt - 1) + nt] = u[3]
    return rs


def init_matrix(ist, m0):
    """[nsim, 2] init matrix of the reference (1-based state, initial cash)."""
    return np.column_stack([np.asarray(ist, dtype=np.float64), np.asarray(m0, dtype=np.float64)])


def check_variant(lib, launches_before, expect, launches=1, label=""):
    """The <PHILOX, OUT, HDR, PB> (and, if given as a fifth entry, mom_smem) that the library reports for this thread's
    last simulation launch (egdst_test_sim_variant) must be `expect`, after `launches` launches since the count
    `launches_before`: a case whose configuration no longer selects the variant it names fails.  Returns mom_smem."""
    v, n = lib.sim_variant()
    assert v[:len(expect)] == tuple(expect), ("launch took %s, the case names %s" % (v, expect))
    assert n - launches_before == launches, (n - launches_before, launches)
    print("%s: <%s, %d, %s, %d> mom_smem=%d" % ((label,) + v))
    return v[4]


def with_thresholds(M, D, periods, k, lo, hi):
    """Solution cells (M, D) of a one-state model whose threshold tables in `periods` are replaced by k thresholds
    spread over [lo, hi) (the first at lo, which the reference's tables start at a0) with alternating decisions: a
    solution for egdst_solution_import with more thresholds in some cells than the per-cell headers carry
    (EGDST_SIM_TH8) and fewer in the others."""
    D = [list(row) for row in D]
    for it in periods:
        d0 = int(D[0][it][0, 0])
        D[0][it] = np.column_stack([(d0 + np.arange(k)) % 2, lo + (hi - lo) * np.arange(k) / k]).astype(np.float64)
    return M, D


class Replay:
    """The port's paths of `nsim` agents on a solution's exported cells of vector `ivec`.  `model` must carry the
    parameter values of that vector (Port reads them from Desc(model))."""

    def __init__(self, model, sol, ivec, init, rs, rndtype=0):
        self.model, self.init, self.rndtype = model, np.asarray(init, dtype=np.float64), rndtype
        self.rs = np.asarray(rs, dtype=np.float64)
        self.cells = sol.cells(ivec)
        self.port = Port(model)
        self.paths = self.port.simulate(*self.cells, self.init, self.rs, rndtype)

    def near_edge(self, i, it):
        """Whether agent i's transition uniform into period it lies within EDGE_EXCL of a cumulative trpr boundary:
        moved by +-EDGE_EXCL it gives the port another next state."""
        if it < 1 or self.rndtype != 0:
            return False
        nt = self.model.nt
        for s in (-EDGE_EXCL, EDGE_EXCL):
            rs = self.rs.reshape(-1, 4 * nt)[i].copy()
            rs[3 * (it - 1)] += s
            p = self.port.simulate(*self.cells, self.init[i:i + 1], rs, 0)
            if not (p[0, it, IST] == self.paths[i, it, IST] or (np.isnan(p[0, it, IST]) and np.isnan(self.paths[i, it, IST]))):
                return True
        return False


def replay(model_for_vector, sol, ivec, init, seed, agent0, rndtype=0):
    """The port's replay (a Replay) of the agents of a Philox launch of vector ivec; rndtype 1: every agent on the
    block of agent0."""
    n = 1 if rndtype == 1 else np.asarray(init).shape[0]
    return Replay(model_for_vector, sol, ivec, init, philox_randstream(n, model_for_vector.nt, seed, agent0), rndtype)


def _near_threshold(cells, port, i, it):
    _, D = cells
    ist, cash = port[i, it, IST], port[i, it, CASH]
    if np.isnan(ist) or np.isnan(cash):
        return False
    d = D[int(ist)][it]
    return d is not None and d.size > 0 and np.min(np.abs(d[:, 1] - cash)) < TH_EXCL


def compare_paths(kernel, port, cells, skipcols=(), replay=None, label="", chunk=1 << 15):
    """Kernel paths against the port's [nsim, nt, nsimout]: NaN pattern and discrete columns (4, 5) exactly, the rest
    to TOL.  A record may differ in them where the port's cash is within TH_EXCL of a threshold of its cell, or (with a
    Replay) where the transition uniform into it is within EDGE_EXCL of a cumulative trpr boundary; that agent's later
    records are then left out.  Returns dict(records, excused, max); fails on anything else."""
    kernel = np.asarray(kernel)
    assert kernel.shape == port.shape, (kernel.shape, port.shape)
    live = int((~np.isnan(port[:, :, CASH])).sum())
    excused, unexplained, worst = 0, [], 0.0
    for lo in range(0, port.shape[0], chunk):  # agent blocks: bounded host memory at a few hundred thousand agents
        k, p = kernel[lo:lo + chunk].copy(), port[lo:lo + chunk].copy()
        if len(skipcols):
            k[:, :, list(skipcols)] = 0.0
            p[:, :, list(skipcols)] = 0.0
        nan_k, nan_p = np.isnan(k), np.isnan(p)
        bad = (nan_k != nan_p).any(axis=2)
        both = ~(nan_k | nan_p)
        bad |= ((k[:, :, DEC] != p[:, :, DEC]) & both[:, :, DEC]) | ((k[:, :, IST] != p[:, :, IST]) & both[:, :, IST])
        for i in np.unique(np.nonzero(bad)[0]):
            it = int(np.argmax(bad[i]))
            if _near_threshold(cells, p, i, it) or (replay is not None and replay.near_edge(lo + i, it)):
                excused += int((~np.isnan(p[i, it:, CASH])).sum())
                k[i, it:], p[i, it:] = np.nan, np.nan
            else:
                unexplained.append((lo + int(i), it))
        e = sims_errors(k, p)
        assert e["nan_mismatch"] == 0 and e["inf_mismatch"] == 0 and e["discrete_mismatch"] == 0 or unexplained, e
        worst = max(worst, e["max"])
    print("%s: %d records compared, %d left out (threshold/boundary rule), largest relative difference %.3g"
          % (label, live - excused, excused, worst))
    assert not unexplained, ("discrete or NaN mismatches (agent, period)", unexplained[:10], len(unexplained))
    assert worst < TOL, worst
    assert excused <= MAX_EXCUSED * max(live, 1), (excused, live)
    return {"records": live - excused, "excused": excused, "max": worst}


def moment_reference(port_paths):
    """(ref, mag): ref [nt, nsimout, 3] the exact moments of paths [nsim, nt, nsimout], math.fsum of x and of x*x and
    the count of non-NaN x per (period, column); mag [nt, nsimout, 5] the sums fsum |x|, x*x, w, w|x|, w*w with
    w = max(1, |x|), which bound the moments' error in check_moments (numpy sums: a bound needs no exact sum).  A
    (period, column) holding +-inf gets the non-finite sums numpy gives."""
    x = np.asarray(port_paths, dtype=np.float64)
    nsim, nt, nso = x.shape
    ref = np.zeros((nt, nso, 3))
    mag = np.zeros((nt, nso, 5))
    for it in range(nt):
        xt = np.ascontiguousarray(x[:, it, :].T)  # [nso, nsim]
        for j in range(nso):
            v = xt[j][~np.isnan(xt[j])]
            ref[it, j, 2] = v.size
            if not np.all(np.isfinite(v)):
                ref[it, j, 0], ref[it, j, 1] = v.sum(), (v * v).sum()
                mag[it, j] = np.inf
                continue
            a = np.abs(v)
            w = np.maximum(1.0, a)
            ref[it, j, 0], ref[it, j, 1] = math.fsum(v), math.fsum(v * v)
            mag[it, j] = [a.sum(), ref[it, j, 1], w.sum(), (w * a).sum(), (w * w).sum()]
    return ref, mag


def check_moments(mom, ref, path_tol=0.0, label=""):
    """Kernel moments [nt, nsimout, 3] against moment_reference of the replayed paths.  The counts must be equal
    exactly.  A sum may differ by the rounding of a sum in any order, 8 * n * 2^-53 * fsum(|x|) (x*x alike: the
    kernel's atomics add in no fixed order), plus what the kernel's records differ from the port's.  That second term is
    needed because the summands are not the same numbers: the kernel's records agree with the port's to the last bits,
    not to the bit (one division for both interpolation weights instead of four, contracted products), and a column
    that is nearly cancelled -- savings in the last period, utility at consumption near zero (u about -10; the deaton2
    sweep vectors differ by up to 1e-10) -- has fsum(|x|) far below those differences.  path_tol is the largest
    |d| / max(1, |x|) that compare_paths measured on the records of this launch (or, for a moments-only launch, of the
    same agents' launch with paths, whose records the kernel writes identically), so the sum of x moves by at most
    path_tol * fsum(w) and that of x*x by path_tol * (2 fsum(w|x|) + path_tol * fsum(w*w)).  Columns holding +-inf or
    NaN must have the same non-finite sums."""
    r, mag = ref
    mom = np.asarray(mom)
    assert np.array_equal(mom[..., 2], r[..., 2]), ("counts", np.argwhere(mom[..., 2] != r[..., 2])[:10])
    n = r[..., 2]
    t = float(path_tol)
    slack = (t * mag[..., 2], t * (2.0 * mag[..., 3] + t * mag[..., 4]))
    for q in (0, 1):
        a, b, s = mom[..., q], r[..., q], mag[..., q]
        fin = np.isfinite(b) & np.isfinite(s)
        assert np.array_equal(np.isnan(a[~fin]), np.isnan(b[~fin])) and np.array_equal(a[~fin & ~np.isnan(b)], b[~fin & ~np.isnan(b)]), \
            ("non-finite pattern", q)
        bound = 8.0 * n[fin] * 2.0 ** -53 * s[fin] + slack[q][fin]
        err = np.abs(a[fin] - b[fin])
        assert np.all(err <= bound), ("sum %d" % q, np.argwhere(fin)[np.argmax(err - bound)], float(np.max(err - bound)))
    print("%s: moments of %d (period, column) cells match the exact sums over the replayed paths" % (label, n.size))
