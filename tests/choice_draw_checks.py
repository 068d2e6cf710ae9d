"""Checks of the choice draws of the taste-shock smoothing mode (egdst_solution_set_choice_draws), shared by the
emulated (CPU) and the GPU tests.

For a record at cash M inside every choice cell's grid [max_d M_d[1], min_d M_d[last]] of its (it, ist), numpy restates
the draw from the exported choice cells: v_d(M) and c_d(M) by np.interp, P_d = softmax(v_d / sigma_eps), and the drawn
decision is the first whose cumulative probability reaches the record's uniform.  The uniforms are restated too: slot
3*(nt-1)+it of the agent's randstream block, or word 3 of the Philox4x32-10 block of counter (agent, it).
"""
import numpy as np

# columns of a record (include/egdst_b200.h, egdst_simulator.c:122-143)
CASH, CONS, SAV, VAL, DEC, IST = 0, 1, 2, 3, 4, 5


def philox4x32(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 on uint64 arrays holding 32-bit words (egdst_philox4x32)."""
    m32 = np.uint64(0xFFFFFFFF)
    c0, c1, c2, c3 = (np.asarray(x, dtype=np.uint64) & m32 for x in (c0, c1, c2, c3))
    k0, k1 = np.uint64(k0) & m32, np.uint64(k1) & m32
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0
        p1 = np.uint64(0xCD9E8D57) * c2
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & m32, p1 >> np.uint64(32), p1 & m32
        c0, c1, c2, c3 = hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0
        k0 = (k0 + np.uint64(0x9E3779B9)) & m32
        k1 = (k1 + np.uint64(0xBB67AE85)) & m32
    return c0, c1, c2, c3


def philox_uniforms(nsim, nt, seed, agent0=0):
    """[nsim, nt] choice uniforms of the Philox source: word 3 of the block of counter (agent0 + i, it)."""
    gid = np.arange(agent0, agent0 + nsim, dtype=np.uint64)[:, None] * np.ones((1, nt), dtype=np.uint64)
    it = np.arange(nt, dtype=np.uint64)[None, :] * np.ones((nsim, 1), dtype=np.uint64)
    _, _, _, w3 = philox4x32(gid, gid >> np.uint64(32), it, 0, seed, seed >> 32)
    return (w3.astype(np.float64) + 0.5) * (1.0 / 4294967296.0)


def randstream_uniforms(rs, nsim, nt):
    """[nsim, nt] choice uniforms of a randstream (rndtype 0): slot 3*(nt-1)+it of each agent's 4*nt block."""
    return np.asarray(rs).reshape(nsim, 4 * nt)[:, 3 * (nt - 1):3 * (nt - 1) + nt]


class ChoiceCells:
    """The exported choice cells of a solution, per (it, ist), with the interpolants of the draw."""

    def __init__(self, sol, m, ivec=0):
        self.sol, self.m, self.ivec, self._c = sol, m, ivec, {}

    def cells(self, it, ist):
        key = (it, ist)
        if key not in self._c:
            self._c[key] = [self.sol.choice_cell(it, ist, d, ivec=self.ivec) for d in range(self.m.nd)]
        return self._c[key]

    def grid(self, it, ist):
        """[max_d M_d[1], min_d M_d[last]] over the available decisions, or None."""
        cs = [c for c in self.cells(it, ist) if c is not None and c.shape[0] >= 3]
        if not cs:
            return None
        return max(c[1, 0] for c in cs), min(c[-1, 0] for c in cs)

    def policy(self, it, ist, M):
        """v [nd, n], c [nd, n] at cash M (inside the grid); -inf / nan for unavailable decisions."""
        M = np.asarray(M, dtype=np.float64)
        v = np.full((self.m.nd, M.size), -np.inf)
        c = np.full((self.m.nd, M.size), np.nan)
        for d, cell in enumerate(self.cells(it, ist)):
            if cell is None or cell.shape[0] < 3:
                continue
            v[d] = np.interp(M, cell[1:, 0], cell[1:, 3])
            c[d] = np.interp(M, cell[1:, 0], cell[1:, 1])
        return v, c

    def probabilities(self, it, ist, M):
        v, _ = self.policy(it, ist, M)
        z = v / self.m.sigma_eps
        e = np.exp(z - z.max(axis=0))
        return e / e.sum(axis=0)


def interior_records(cc, sims):
    """(agent, it) index arrays of the live records whose cash lies inside every choice cell's grid."""
    alive = ~np.isnan(sims[:, :, CASH])
    ai, ti = np.nonzero(alive)
    keep = np.zeros(ai.size, dtype=bool)
    for it in np.unique(ti):
        for ist in np.unique(sims[ai[ti == it], it, IST]).astype(int):
            g = cc.grid(int(it), ist)
            if g is None:
                continue
            sel = (ti == it) & (sims[ai, ti, IST] == ist)
            M = sims[ai[sel], it, CASH]
            keep[np.nonzero(sel)[0]] = (M >= g[0]) & (M <= g[1])
    return ai[keep], ti[keep]


def check_mechanism(cc, sims, U, margin=1e-9, tol=1e-12):
    """Every interior record whose uniform is more than `margin` from a cumulative boundary holds the numpy draw, and
    the drawn decision's consumption, value and savings.  Returns (records checked, count per decision)."""
    ai, ti = interior_records(cc, sims)
    checked, counts = 0, np.zeros(cc.m.nd, dtype=int)
    for it in np.unique(ti):
        for ist in np.unique(sims[ai[ti == it], it, IST]).astype(int):
            sel = (ti == it) & (sims[ai, ti, IST] == ist)
            a = ai[sel]
            rec = sims[a, it]
            M, u = rec[:, CASH], U[a, it]
            v, c = cc.policy(int(it), ist, M)
            P = cc.probabilities(int(it), ist, M)
            cum = np.cumsum(P, axis=0)
            clear = np.all(np.abs(cum - u[None, :]) > margin, axis=0)
            d = np.argmax(cum >= u[None, :], axis=0)
            d = d[clear]
            rec = rec[clear]
            cols = np.arange(d.size)
            assert np.array_equal(rec[:, DEC], d.astype(float)), (it, ist, rec[:, DEC], d)
            np.testing.assert_allclose(rec[:, CONS], c[d, np.nonzero(clear)[0]], rtol=0, atol=tol)
            np.testing.assert_allclose(rec[:, VAL], v[d, np.nonzero(clear)[0]], rtol=0, atol=tol)
            np.testing.assert_allclose(rec[:, SAV], rec[:, CASH] - rec[:, CONS], rtol=0, atol=tol)
            checked += cols.size
            counts += np.bincount(d, minlength=cc.m.nd)
    return checked, counts
