"""The two-periods-per-write simulator launch (PB = 2) against the one-period launch (PB = 1).

Large Philox launches through the device entry point that write the path array take the wide kernel; the host-buffer
API chunks below its threshold, so only these tests reach it.  The same agents simulated as shards below the
threshold (with their global ids as agent0) take the one-period kernel: records must agree to the bit, NaN pattern
included, and the moments must be the sums over the returned paths."""
import numpy as np
import pytest

from egdst_b200 import capi, examples

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

SEED = 20240611


def _solve(factory):
    m = factory(T=24)  # the wide kernel pairs periods: even nt
    m.compile()
    lib = m._capi()
    sol = lib.solve(m, strict=True)
    return m, lib, sol


@pytest.fixture(scope="module", params=["retirement2", "retirement_mortal"])
def solved(request):
    return _solve(getattr(examples, request.param))


def _wide_nsim():
    # above the wide kernel's threshold (4 tiles of 32 agents per warp and SM) for CTAs of up to 16 warps
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    return max(310_000, 4 * sms * 16 * 32 + 4096)


def _init(m, nsim):
    rng = np.random.default_rng(7)
    ist = np.ones(nsim)
    m0 = m.a0 + 0.5 * (m.mmax - m.a0) * rng.random(nsim)
    m0[::997] = m.a0 - 1.0  # outside the grid: skipped agents, NaN from period 0
    return ist, m0


def _simulate_kernels(fn):
    """The PB template argument of every egdst_k_simulate launch made by fn()."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
    names = [e.key for e in prof.key_averages() if "egdst_k_simulate<" in e.key]
    return sorted({int(n.split("egdst_k_simulate<")[1].split(">")[0].split(",")[-1]) for n in names})


def _run(m, lib, sol, desc, ist, m0, agent0, sims=True, moments=True):
    dev = torch.device("cuda", 0)
    n = ist.shape[0]
    nt, nso = m.nt, m.nsimout()
    d_init = torch.from_numpy(np.concatenate([ist, m0])).to(dev)
    d_sims = torch.full((n * nt * nso,), 7.0, dtype=torch.float64, device=dev) if sims else None
    d_mom = torch.zeros(3 * nso * nt, dtype=torch.float64, device=dev) if moments else None
    lib.simulate_device(m, sol, d_init.data_ptr(), n, agent0, SEED, d_sims.data_ptr() if sims else 0,
                        d_mom.data_ptr() if moments else 0, desc=desc)
    torch.cuda.synchronize()
    # sims [nsimout, nt, nsim] column-major -> [nsim, nt, nsimout]; moments [3, nsimout, nt] -> [nt, nsimout, 3]
    s = d_sims.cpu().numpy().reshape(n, nt, nso) if sims else None
    mo = d_mom.cpu().numpy().reshape(nt, nso, 3) if moments else None
    return s, mo


def test_wide_launch_matches_sharded_launches(solved):
    m, lib, sol = solved
    desc = capi.Desc(m)
    nsim = _wide_nsim()
    ist, m0 = _init(m, nsim)
    out = []
    assert _simulate_kernels(lambda: out.append(_run(m, lib, sol, desc, ist, m0, 0))) == [2]  # the wide kernel ran
    full, mom = out[0]
    nan = np.isnan(full)
    alive = ~nan[:, :, 0]
    assert not (~alive[:, :-1] & alive[:, 1:]).any()  # a record that ends stays NaN
    if m.label == "retire_mortal":
        assert (alive[:, 0] & ~alive[:, -1]).any()  # deaths on the way
    nshard = 8  # about 40 k agents each: the one-period kernel
    bounds = np.linspace(0, nsim, nshard + 1).astype(int)
    mom_sh = np.zeros_like(mom)
    for k, (lo, hi) in enumerate(zip(bounds[:-1], bounds[1:])):
        if k == 0:
            out = []
            assert _simulate_kernels(lambda: out.append(_run(m, lib, sol, desc, ist[lo:hi], m0[lo:hi], int(lo)))) == [1]
            part, pm = out[0]
        else:
            part, pm = _run(m, lib, sol, desc, ist[lo:hi], m0[lo:hi], int(lo))
        assert np.array_equal(np.isnan(part), nan[lo:hi])
        assert np.array_equal(part.view(np.int64)[~nan[lo:hi]], full[lo:hi].view(np.int64)[~nan[lo:hi]])
        mom_sh += pm
    assert np.allclose(mom_sh, mom, rtol=1e-12, atol=1e-9)
    # moments against numpy sums over the returned paths
    s1 = np.where(nan, 0.0, full).sum(axis=0)
    s2 = np.where(nan, 0.0, full * full).sum(axis=0)
    fin = np.isfinite(s1) & np.isfinite(s2)
    assert np.allclose(mom[..., 0][fin], s1[fin], rtol=1e-11, atol=1e-9)
    assert np.allclose(mom[..., 1][fin], s2[fin], rtol=1e-11, atol=1e-9)
    assert np.array_equal(mom[..., 2], (~nan).sum(axis=0).astype(float))
    # the moments-only launch of the same agents
    _, mom_only = _run(m, lib, sol, desc, ist, m0, 0, sims=False)
    assert np.allclose(mom_only, mom, rtol=1e-12, atol=1e-9)
    # the path array alone is the same as with moments
    full2, _ = _run(m, lib, sol, desc, ist, m0, 0, moments=False)
    assert np.array_equal(np.isnan(full2), nan) and np.array_equal(full2.view(np.int64)[~nan], full.view(np.int64)[~nan])

