"""Stored checker: sampled outputs of the configurations the GPU tests compare, for machines without the compiled
reference (oracle/_ref).

tests/golden/stored.npz holds, per model configuration (keyed by a hash of ``model.to_dict()``), the solver's status,
every threshold row of D, and a seeded sample of the rows of M (cash, consumption, value), with the row count and
evf(a0) of each cell; and, per simulation input (model, init, randstream, rndtype), a seeded sample of the
simulation records.  The solutions were recorded on a B200 by this project's own solver, and the simulations by the C
restatement of the reference's simulator (oracle/port) on those solutions, when this file was added: they are not
outputs of the reference C.  They pin this project's results for every later change; wherever oracle/_ref is present
the tests compare with the reference instead.

Recording: run the suite with EGDST_STORE_RECORD=<dir> on a GPU machine; every configuration without a stored entry
is solved and written to <dir>/<key>.npz.  ``python tests/stored.py merge <dir>`` folds them into stored.npz.  Entries
already in stored.npz are never recorded again, so a later build is always compared with the same vectors.
"""
from __future__ import annotations

import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
STORE = os.path.join(HERE, "golden", "stored.npz")
RECORD = os.environ.get("EGDST_STORE_RECORD")

ROWS = 24        # sampled rows of M per configuration, spread over its cells (at least one per cell); or every row
                 # (oracle_for(..., whole=True)) where a test inspects the rows themselves
MAXCELLS = 64    # cells sampled per configuration
RECORDS = 6      # sampled (agent, period) records per simulation
EXCL = 1e-9      # sampled rows keep this distance from thresholds and double points (parity.cell_errors excludes them too)

_cache = {}


class StoreMissing(LookupError):
    """A configuration without a stored entry: a test error, never a skip (a changed example or model property changes
    the key, and the comparison must not silently disappear)."""


class SampledCell:
    """Sampled rows of one solution cell: ``x``, ``c``, ``v`` (cash, consumption, value), ``nrows`` of the full cell,
    ``evf`` (row 0 of V)."""

    def __init__(self, x, c, v, nrows, evf):
        self.x, self.c, self.v, self.nrows, self.evf = x, c, v, int(nrows), evf
        self.size = self.nrows


class SampledSims:
    """Sampled records of a [nsim, nt, nsimout] simulation: ``agents``, ``periods`` and ``records`` [k, nsimout]."""

    def __init__(self, agents, periods, records):
        self.agents, self.periods, self.records = agents, periods, records

    def pick(self, sims):
        return sims[self.agents, self.periods, :]


NOT_SAMPLED = SampledCell(np.zeros(0), np.zeros(0), np.zeros(0), 0, 0.0)


def model_key(model) -> str:
    d = model.to_dict()
    if d["ngridmax"] <= d["ngridm"]:  # what solve() does before it runs
        d["ngridmax"] = 2 * d["ngridm"]
    return hashlib.sha1(json.dumps(d, sort_keys=True, default=repr).encode()).hexdigest()[:16]


def sim_key(mkey, init, rs, rndtype) -> str:
    h = hashlib.sha1(mkey.encode())
    h.update(np.ascontiguousarray(init, dtype=np.float64).tobytes())
    h.update(np.ascontiguousarray(rs, dtype=np.float64).tobytes())
    h.update(str(int(rndtype)).encode())
    return h.hexdigest()[:16]


def _load(key):
    if key in _cache:
        return _cache[key]
    if RECORD:
        p = os.path.join(RECORD, key + ".npz")
        if os.path.isfile(p):
            with np.load(p) as z:
                _cache[key] = z["a"]
            return _cache[key]
    if "store" not in _cache:
        _cache["store"] = _read_store()
    return _cache["store"].get(key)


def _read_store():
    """stored.npz: ``keys``, ``shapes`` [n, 2] and ``data`` (every entry flattened column by column, concatenated)."""
    if not os.path.isfile(STORE):
        return {}
    with np.load(STORE) as z:
        keys, shapes, data = z["keys"], z["shapes"], z["data"]
    out, off = {}, 0
    for k, (r, c) in zip(keys, shapes):
        out[str(k)] = data[off:off + r * c].reshape((r, c), order="F")
        off += r * c
    return out


def _save(key, a):
    os.makedirs(RECORD, exist_ok=True)
    np.savez(os.path.join(RECORD, key + ".npz"), a=a)
    _cache[key] = a


# solve table: one row per record, (code, x, y, z) with code = tag + 4 * (it + 4096 * ist);
# tag 0: cell header (nrows, evf, -); 1: sampled row (M, C, V); 2: row of D (decision, threshold, -); 3: status (code)
def _sample_solution(key, M, D, status, whole=False):
    out = [[3.0, float(status), 0.0, 0.0]]
    cells = [(ist, it) for ist in range(len(M)) for it in range(len(M[ist])) if M[ist][it] is not None and M[ist][it].size]
    rng = np.random.default_rng(int(key, 16) % (2 ** 32))
    chosen = set(cells) if len(cells) <= MAXCELLS else {cells[i] for i in rng.choice(len(cells), MAXCELLS, replace=False)}
    per = max(1, ROWS // max(len(chosen), 1))
    for ist, it in cells:
        code = 4 * (it + 4096 * ist)
        for r in D[ist][it]:
            out.append([code + 2, r[0], r[1], 0.0])
        m = M[ist][it]
        out.append([code, m.shape[0] if (ist, it) in chosen else -1, m[0, 3], 0.0])
        if (ist, it) not in chosen:
            continue
        if whole:
            out += [[code + 1, r[0], r[1], r[3]] for r in m]
            continue
        x = m[1:, 0]
        ok = np.ones(x.size, dtype=bool)
        for th in D[ist][it][:, 1]:
            ok &= np.abs(x - th) > EXCL
        close = np.flatnonzero(np.diff(x) < EXCL)
        ok[close] = False
        ok[close + 1] = False
        idx = np.flatnonzero(ok)
        for j in (rng.choice(idx, min(per, idx.size), replace=False) if idx.size else []):
            out.append([code + 1, m[j + 1, 0], m[j + 1, 1], m[j + 1, 3]])
    return np.array(out, dtype=np.float64)


def _unpack_solution(a, nst, nt):
    status = int(a[0, 1])
    M = [[None] * nt for _ in range(nst)]
    D = [[None] * nt for _ in range(nst)]
    rows, drows = {}, {}
    for code, x, y, z in a[1:]:
        code = int(code)
        tag, it, ist = code % 4, (code // 4) % 4096, code // (4 * 4096)
        if tag == 0:
            M[ist][it] = (int(x), y) if x >= 0 else NOT_SAMPLED
            drows.setdefault((ist, it), [])
        elif tag == 1:
            rows.setdefault((ist, it), []).append((x, y, z))
        elif tag == 2:
            drows.setdefault((ist, it), []).append((x, y))
    for (ist, it), d in drows.items():
        D[ist][it] = np.array(d, dtype=np.float64).reshape(-1, 2)
    for ist in range(nst):
        for it in range(nt):
            if isinstance(M[ist][it], tuple):
                r = np.array(rows.get((ist, it), []), dtype=np.float64).reshape(-1, 3)
                nrows, evf = M[ist][it]
                if r.shape[0] == nrows:  # a whole cell (a sample never holds row 0)
                    M[ist][it] = np.column_stack([r[:, 0], r[:, 1], r[:, 0] - r[:, 1], r[:, 2]])
                else:
                    M[ist][it] = SampledCell(r[:, 0], r[:, 1], r[:, 2], nrows, evf)
    return status, M, D


class StoredError(RuntimeError):
    pass


class Stored:
    kind = "stored"
    seconds = None

    def __init__(self, model, whole=False):
        self.model = model
        self.whole = whole
        self.key = model_key(model) + ("w" if whole else "")
        self._full = None

    def _missing(self, what):
        return StoreMissing("tests/golden/stored.npz has no %s for this configuration (key %s); record it (module docstring)" % (what, self.key))

    def solve(self):
        m = self.model
        a = _load(self.key)
        if a is None and RECORD:
            a = self._record_solution()
        if a is None:
            raise self._missing("solution")
        status, M, D = _unpack_solution(a, m.nst, m.nt)
        if status:
            raise StoredError("the stored solve of this configuration reported status %d" % status)
        return M, D

    def _record_solution(self):
        from egdst_b200.model import EgdstModel
        mm = EgdstModel.from_dict(self.model.to_dict())
        mm.compile()
        sol = mm._capi().solve(mm)
        self._full = (sol.M, sol.D)
        a = _sample_solution(self.key.rstrip("w"), sol.M, sol.D, sol.status()[0], self.whole)
        _save(self.key, a)
        return a

    def simulate(self, M, D, init, rs, rndtype=0):
        """On a full solution: the C restatement of the reference's simulator (oracle/port) runs on it.  On the
        sampled solution of ``solve()``: the stored records of that simulation (a ``SampledSims``)."""
        from oracle.port import Port
        init = np.atleast_2d(np.asarray(init, dtype=np.float64))
        rs = np.asarray(rs, dtype=np.float64).ravel()
        if not any(isinstance(c, SampledCell) for row in M for c in row):
            p = Port(self.model)
            sims = p.simulate(M, D, init, rs, rndtype)
            self.seconds = p.last_seconds
            return sims
        k = sim_key(self.key, init, rs, rndtype)
        a = _load(k)
        if a is None and RECORD:
            if self._full is None:
                self._record_solution()
            sims = Port(self.model).simulate(*self._full, init, rs, rndtype)
            rng = np.random.default_rng(int(k, 16) % (2 ** 32))
            ag = rng.integers(0, sims.shape[0], RECORDS)
            pe = rng.integers(0, sims.shape[1], RECORDS)
            a = np.column_stack([ag, pe, sims[ag, pe, :]]).astype(np.float64)
            _save(k, a)
        if a is None:
            raise self._missing("simulation")
        return SampledSims(a[:, 0].astype(int), a[:, 1].astype(int), a[:, 2:])


def merge(src):
    store = _read_store()
    for f in sorted(os.listdir(src)):
        if f.endswith(".npz"):
            with np.load(os.path.join(src, f)) as z:
                store[f[:-4]] = z["a"]
    keys = sorted(store)
    # one flat array rather than one member per entry; columns contiguous, so the index columns compress well
    np.savez_compressed(STORE, keys=np.array(keys), shapes=np.array([store[k].shape for k in keys]),
                        data=np.concatenate([store[k].ravel(order="F") for k in keys]))
    print("%d entries, %d bytes" % (len(store), os.path.getsize(STORE)))

if __name__ == "__main__":
    if len(sys.argv) == 3 and sys.argv[1] == "merge":
        merge(sys.argv[2])
