"""The two-periods-per-write simulator kernel (PB = 2, pipelined period loop) on the host emulator, against the
one-period kernel (PB = 1): the emulator's launch takes PB = 2 from 1024 agents on, smaller shards take PB = 1."""
import os
import shutil
import sys

import numpy as np
import pytest

from egdst_b200 import capi, examples

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "tools", "hostemu"))

pytestmark = pytest.mark.skipif(shutil.which("g++") is None, reason="g++ not available")


def _sim(lib, m, sol, ist, m0, agent0):
    n = ist.shape[0]
    init = np.ascontiguousarray(np.concatenate([ist, m0]))
    sims = np.full(n * m.nt * m.nsimout(), 7.0)
    mom = np.zeros(3 * m.nsimout() * m.nt)
    lib.simulate_device(m, sol, init.ctypes.data, n, agent0, 99, sims.ctypes.data, mom.ctypes.data)
    return sims.reshape(n, m.nt, m.nsimout()), mom.reshape(m.nt, m.nsimout(), 3)


@pytest.mark.parametrize("make", [examples.retirement2, examples.retirement_mortal])
def test_emulated_wide_kernel_matches_sharded_runs(make):
    from build import build  # tools/hostemu/build.py
    m = make(T=6, ngridm=40, ngridmax=200, ny=4)  # even nt
    m.prepare()
    lib = capi.ModelLibrary(build(m))
    sol = lib.solve(m)
    assert sol.status()[0] == 0, sol.status()
    n = 2048
    rng = np.random.default_rng(3)
    ist = np.ones(n)
    m0 = m.a0 + 0.5 * (m.mmax - m.a0) * rng.random(n)
    m0[::97] = m.a0 - 1.0  # skipped agents: NaN from period 0
    full, mom = _sim(lib, m, sol, ist, m0, 0)
    nan = np.isnan(full)
    alive = ~nan[:, :, 0]
    assert not (~alive[:, :-1] & alive[:, 1:]).any()
    if m.label == "retire_mortal":
        assert (alive[:, 0] & ~alive[:, -1]).any()
    mom_sh = np.zeros_like(mom)
    for lo in range(0, n, 256):
        part, pm = _sim(lib, m, sol, ist[lo:lo + 256], m0[lo:lo + 256], lo)
        assert np.array_equal(np.isnan(part), nan[lo:lo + 256])
        assert np.array_equal(part[~nan[lo:lo + 256]].view(np.int64), full[lo:lo + 256][~nan[lo:lo + 256]].view(np.int64))
        mom_sh += pm
    assert np.allclose(mom_sh, mom, rtol=1e-12, atol=1e-9)
    s1 = np.where(nan, 0.0, full).sum(axis=0)
    fin = np.isfinite(s1)
    assert np.allclose(mom[..., 0][fin], s1[fin], rtol=1e-11, atol=1e-9)
    assert np.array_equal(mom[..., 2], (~nan).sum(axis=0).astype(float))
