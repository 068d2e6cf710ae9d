"""Every instantiation of egdst_k_simulate that a Philox launch selects (no choice draws), replayed agent by agent
through the reference simulator's C restatement on the same uniforms (tests/philox_replay_checks.py), and the
randstream instantiations fed those uniforms.  Each launch names the <PHILOX, OUT, HDR, PB> (and, where it matters,
mom_smem) it covers and asserts it against what the library reports it launched (egdst_test_sim_variant), and the
host-buffer case asserts its number of chunk launches: a case whose configuration no longer selects its variant fails."""
import numpy as np
import pytest

from egdst_b200 import capi, examples
from tests import philox_replay_checks as R

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

AGENT0, SEED = 2**32 - 1000, 2**40 + 5  # the launches cross the high word of the agent id; the seed has a high word
NPLAIN = 40_017                          # PB = 1 launches: 1251 tiles, the last one a tail


def _wide_nsim():
    # the PB = 2 threshold (4 tiles of 32 agents per warp of a 12-warp CTA and SM) plus a tail tile
    return 4 * torch.cuda.get_device_properties(0).multi_processor_count * 12 * 32 + 77


def _solve(m):
    m.compile()
    lib = m._capi()
    sol = lib.solve(m, strict=True)
    return lib, sol


def _init(m, n, seed=7, ist=1):
    rng = np.random.default_rng(seed)
    m0 = m.a0 + 0.5 * (m.mmax - m.a0) * rng.random(n)
    m0[::33] = m.a0 - 1.0  # about 3 % skipped agents: NaN from period 0
    return R.init_matrix(np.full(n, float(ist)), m0)


class Launcher:
    """simulate_device of one model on device buffers; each launch must take the instantiation it names."""

    def __init__(self, m, lib, sol, init):
        self.m, self.lib, self.sol, self.desc = m, lib, sol, capi.Desc(m)
        self.init, self.n = init, init.shape[0]
        self.dev = torch.device("cuda", 0)
        self.d_init = torch.from_numpy(np.ascontiguousarray(np.concatenate([init[:, 0], init[:, 1]]))).to(self.dev)

    def __call__(self, expect, n=None, sims=True, moments=True, rs=None, rndtype=0, misalign=False):
        m, n = self.m, n or self.n
        nt, nso = m.nt, m.nsimout()
        d_init = self.d_init if n == self.n else torch.from_numpy(
            np.ascontiguousarray(np.concatenate([self.init[:n, 0], self.init[:n, 1]]))).to(self.dev)
        buf = torch.full((n * nt * nso + 2,), 7.0, dtype=torch.float64, device=self.dev) if sims else None
        off = 1 if misalign else 0  # 8 bytes off 16-byte alignment: the scalar store path of the tile (vecok false)
        mom = torch.zeros(3 * nso * nt, dtype=torch.float64, device=self.dev) if moments else None
        d_rs = torch.from_numpy(np.ascontiguousarray(rs).ravel()).to(self.dev) if rs is not None else None
        n0 = self.lib.sim_variant()[1]
        self.lib.simulate_device(m, self.sol, d_init.data_ptr(), n, AGENT0, SEED, buf.data_ptr() + 8 * off if sims else 0,
                                 mom.data_ptr() if moments else 0, d_randstream=d_rs.data_ptr() if rs is not None else 0,
                                 rndtype=rndtype, desc=self.desc)
        smem = R.check_variant(self.lib, n0, expect, label=m.label)
        s = buf[off:off + n * nt * nso].cpu().numpy().reshape(n, nt, nso) if sims else None
        mo = mom.cpu().numpy().reshape(nt, nso, 3) if moments else None
        return s, mo, smem


def _bits_equal(a, b):
    nan = np.isnan(a)
    return np.array_equal(nan, np.isnan(b)) and np.array_equal(a[~nan].view(np.int64), b[~nan].view(np.int64))


def _full_check(m, lib, sol, init, hdr, pb_sims, label):
    """The launches of one configuration against the replay: sims and moments, sims only, moments only, the same
    records through the randstream instantiation fed the replayed uniforms."""
    rs = R.philox_randstream(init.shape[0], m.nt, SEED, AGENT0)
    rp = R.Replay(m, sol, 0, init, rs)
    ref = R.moment_reference(rp.paths)
    run = Launcher(m, lib, sol, init)
    full, mom, _ = run((True, 3, hdr, pb_sims, True))
    tol = R.compare_paths(full, rp.paths, rp.cells, replay=rp, label=label)["max"]
    R.check_moments(mom, ref, tol, label=label)
    only, _, _ = run((True, 1, hdr, pb_sims), moments=False)
    assert _bits_equal(only, full)
    _, mom2, _ = run((True, 2, hdr, 1, True), sims=False)
    R.check_moments(mom2, ref, tol, label=label + " moments only")
    # the randstream instantiation (PB = 1) on the same uniforms: the same records to the bit (PB = 2 == PB = 1)
    rsf, momr, _ = run((False, 3, hdr, 1, True), rs=rs)
    assert _bits_equal(rsf, full)
    R.check_moments(momr, ref, tol, label=label + " randstream")
    return run, rp, full, tol


@pytest.mark.parametrize("make", [examples.retirement2, examples.retirement_mortal])
def test_plain_launches_match_the_replay(make):
    """<true, 1/2/3, true, 1> and <false, 1/3, true, 1>: nt = 25 (odd: PB = 1 at any size), a tail tile, skipped agents,
    and (retirement_mortal) deaths, so tiles that are not clean."""
    m = make(T=25)
    lib, sol = _solve(m)
    init = _init(m, NPLAIN)
    run, rp, full, _ = _full_check(m, lib, sol, init, True, 1, "%s T=25" % m.label)
    live = ~np.isnan(rp.paths[:, :, 0])
    if m.label == "retire_mortal":
        assert (live[:, 0] & ~live[:, -1]).any()
    # the sims array 8 bytes off 16-byte alignment: the scalar store path
    mis, _, _ = run((True, 1, True, 1), moments=False, misalign=True)
    assert _bits_equal(mis, full)
    # rndtype 1: every agent on one block
    n1 = 5000
    r1 = R.replay(m, sol, 0, init[:n1], SEED, AGENT0, rndtype=1)
    s1, _, _ = run((False, 1, True, 1), n=n1, moments=False, rs=r1.rs, rndtype=1)
    R.compare_paths(s1, r1.paths, r1.cells, label="%s rndtype 1" % m.label)


@pytest.mark.parametrize("make,T", [(examples.retirement2, 24), (examples.retirement_mortal, 24), (examples.retirement_jobloss, 66)])
def test_pipelined_wide_launches_match_the_replay(make, T):
    """<true, 1/3, HDR, 2>, the pipelined period order: retirement2 and retirement_mortal with per-cell headers,
    retirement_jobloss (nst = 2, nt * nst = 132 > 128) without, and shock-dependent transition probabilities."""
    m = make(T=T)
    lib, sol = _solve(m)
    hdr = m.nt * m.nst <= 128
    assert hdr == (m.label != "jobloss")
    init = _init(m, _wide_nsim())
    run, rp, full, _ = _full_check(m, lib, sol, init, hdr, 2, "%s T=%d wide" % (m.label, T))
    # the first agents alone: PB = 1, the same records
    n1 = 20_000
    part, mom1, _ = run((True, 3, hdr, 1), n=n1)
    assert _bits_equal(part, full[:n1])
    R.check_moments(mom1, R.moment_reference(rp.paths[:n1]), R.compare_paths(part, rp.paths[:n1], rp.cells, replay=rp, label="%s PB = 1 shard" % m.label)["max"],
                    label="%s PB = 1 shard" % m.label)


def test_continuous_states_match_the_replay():
    """Continuous states: humancapital (nsimout 14) at PB = 2 on the plain period order (PIPE false), and humancapital2
    (nsimout 15, odd rows: the scalar store path, no headers at nt * nst = 180).  Every agent starts at the first grid
    point of the continuous states, where the reference addresses its initial cell correctly.  The value column, which
    the reference leaves unassigned on this branch, is the mix of the corner values in both the kernel and the port."""
    m = examples.humancapital()
    lib, sol = _solve(m)
    assert m.nsimout() % 2 == 0 and m.nt * m.nst <= 128
    _full_check(m, lib, sol, _init(m, _wide_nsim()), True, 2, "humancapital wide")
    m2 = examples.humancapital2()
    lib2, sol2 = _solve(m2)
    assert m2.nsimout() % 2 == 1 and m2.nt * m2.nst > 128
    _full_check(m2, lib2, sol2, _init(m2, NPLAIN), False, 1, "humancapital2")


def test_moments_in_global_memory_and_host_chunks():
    """retirement2 at T = 100: the PB = 1 moment accumulators no longer fit next to the staged rows (mom_smem = 0,
    atomics to global memory), and the host-buffer entry point splits the agents into three chunks, the last partial."""
    m = examples.retirement2(T=100)
    lib, sol = _solve(m)
    nt, nso = m.nt, m.nsimout()
    chunk = (256 << 20) // (8 * nso * nt) // 32 * 32
    assert chunk >= 4096
    n = 2 * chunk + chunk // 2 + 11
    init = _init(m, n)
    rs = R.philox_randstream(n, nt, SEED, AGENT0)
    rp = R.Replay(m, sol, 0, init, rs)
    ref = R.moment_reference(rp.paths)
    run = Launcher(m, lib, sol, init)
    full, mom, _ = run((True, 3, True, 1, False))
    tol = R.compare_paths(full, rp.paths, rp.cells, replay=rp, label="retirement2 T=100")["max"]
    R.check_moments(mom, ref, tol, label="retirement2 T=100 mom_smem=0")
    _, mom2, _ = run((True, 2, True, 1, False), sims=False)
    R.check_moments(mom2, ref, tol, label="retirement2 T=100 moments only, mom_smem=0")
    # host buffers: three launches of chunk, chunk and chunk / 2 + 11 agents
    n0 = lib.sim_variant()[1]
    hs, hm = lib.simulate_philox(m, sol, init, SEED, agent0=AGENT0, want_moments=True)
    R.check_variant(lib, n0, (True, 3, True, 1, False), launches=3, label="host chunks")
    assert _bits_equal(hs, full)
    R.check_moments(hm.transpose(2, 1, 0), ref, tol, label="retirement2 T=100 host chunks")


def test_cells_without_tables(monkeypatch):
    """EGDST_TABCAP (test hook): every cell exceeds the lookup-table capacity; the headers flag it and the simulator
    bisects the plain columns."""
    monkeypatch.setenv("EGDST_TABCAP", "16")
    m = examples.retirement2(T=12, ngridm=700, ngridmax=1500, nthrhmax=700, ny=8, interest=0.02)
    lib, sol = _solve(m)
    M, _ = sol.cells(0)
    assert min(M[0][it].shape[0] for it in range(m.nt)) > 16
    _full_check(m, lib, sol, _init(m, NPLAIN), True, 1, "retirement2 without tables")


def test_sweep_moments_match_the_replays():
    """<true, 2, false, 1> over a batched solve (blockIdx.y walks the vectors): the moments of vectors 0, 11 and 23,
    each against the replay under its own parameter values."""
    m = examples.deaton2()
    m.compile()
    lib = m._capi()
    rng = np.random.default_rng(4096)
    nvec = 24
    params = np.column_stack([rng.uniform(0.0, 0.05, nvec), rng.uniform(0.75, 1.75, nvec)])  # (interest, income)
    sol = lib.solve_batch(m, params)
    assert sol.warning is None, sol.warning
    n = 4096 + 13
    init = _init(m, n)
    n0 = lib.sim_variant()[1]
    mom = lib.sim_moments(m, sol, init, SEED, agent0=AGENT0)
    R.check_variant(lib, n0, (True, 2, False, 1), label="deaton2 sweep")
    rs = R.philox_randstream(n, m.nt, SEED, AGENT0)
    for i in (0, 11, nvec - 1):
        mi = examples.deaton2(interest=params[i, 0], income=params[i, 1])
        rp = R.Replay(mi, sol, i, init, rs)
        n0 = lib.sim_variant()[1]
        paths, _ = lib.simulate_philox(m, sol, init, SEED, agent0=AGENT0, ivec=i)
        R.check_variant(lib, n0, (True, 1, True, 1), label="deaton2 vector %d" % i)
        tol = R.compare_paths(paths, rp.paths, rp.cells, replay=rp, label="deaton2 vector %d" % i)["max"]
        R.check_moments(mom[i].transpose(2, 1, 0), R.moment_reference(rp.paths), tol, label="deaton2 sweep vector %d" % i)


def test_thresholds_beyond_the_headers_match_the_replay():
    """Per-cell headers carry EGDST_SIM_TH8 = 4 thresholds; a cell with more takes the policy decision from the threshold
    table in global memory.  No shipped example has such a cell, so an imported solution of retirement2 gets 6
    thresholds over the agents' cash in the even periods and keeps the solver's (at most 2) in the odd ones: the
    pipelined PB = 2 and the PB = 1 launch, both with headers."""
    m = examples.retirement2(T=24)
    lib, sol0 = _solve(m)
    M, D = R.with_thresholds(*sol0.cells(0), periods=range(0, m.nt, 2), k=6, lo=m.a0, hi=m.a0 + 0.5 * (m.mmax - m.a0))
    sol = lib.import_solution(m, M, D)
    nth = [sol.cells(0)[1][0][it].shape[0] for it in range(m.nt)]
    assert max(nth) > 4 and min(nth) <= 4, nth
    init = _init(m, _wide_nsim())
    run, rp, full, _ = _full_check(m, lib, sol, init, True, 2, "retirement2 imported thresholds wide")
    assert len(np.unique(full[:, 0::2, 4][~np.isnan(full[:, 0::2, 4])])) == 2
    n1 = 20_000
    part, _, _ = run((True, 1, True, 1), n=n1, moments=False)
    assert _bits_equal(part, full[:n1])
