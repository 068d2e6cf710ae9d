"""Choice draws of the smoothing mode (egdst_solution_set_choice_draws) on the host emulator of the kernels: the drawn
decision and its record against a numpy restatement, for both sources of uniforms; sharding; moments; the modal mode
untouched; refusals."""
import os
import shutil
import sys

import numpy as np
import pytest

from egdst_b200 import capi, examples
from tests import choice_draw_checks as cd

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "tools", "hostemu"))

pytestmark = pytest.mark.skipif(shutil.which("g++") is None, reason="g++ not available")

_CACHE = {}


def _solved():
    """retirement2_smooth (T=6: nt even), sigma_eps = 0.2, solved on the emulator."""
    if "sol" not in _CACHE:
        from build import build  # tools/hostemu/build.py
        m = examples.retirement2_smooth(sigma_eps=0.2, T=6, ngridm=300, ny=5)
        m.prepare()
        lib = capi.ModelLibrary(build(m))
        sol = lib.solve(m)
        assert sol.status()[0] == 0, sol.status()
        _CACHE["sol"] = (m, lib, sol)
    return _CACHE["sol"]


def _init(m, n, seed=1):
    rng = np.random.default_rng(seed)
    return np.column_stack([np.ones(n), m.a0 + 0.6 * (m.mmax - m.a0) * rng.random(n)])


def _device(lib, m, sol, init, agent0, seed=99):
    n = init.shape[0]
    initf = np.ascontiguousarray(init.ravel(order="F"))
    sims = np.full(n * m.nt * m.nsimout(), 7.0)
    mom = np.zeros(3 * m.nsimout() * m.nt)
    lib.simulate_device(m, sol, initf.ctypes.data, n, agent0, seed, sims.ctypes.data, mom.ctypes.data)
    return sims.reshape(n, m.nt, m.nsimout()), mom.reshape(m.nt, m.nsimout(), 3)


def test_randstream_draws_follow_the_choice_probabilities():
    m, lib, sol = _solved()
    n = 2000
    init = _init(m, n)
    rs = np.random.default_rng(7).random(4 * m.nt * n)
    sol.set_choice_draws(True)
    try:
        sims = lib.simulate(m, sol, init, rs)
    finally:
        sol.set_choice_draws(False)
    checked, counts = cd.check_mechanism(cd.ChoiceCells(sol, m), sims, cd.randstream_uniforms(rs, n, m.nt))
    assert checked >= 300 and (counts > 0).all(), (checked, counts)


def test_philox_draws_follow_the_choice_probabilities():
    m, lib, sol = _solved()
    n = 2000
    init = _init(m, n, seed=2)
    sol.set_choice_draws(True)
    try:
        sims, _ = lib.simulate_philox(m, sol, init, seed=12345, agent0=5)
    finally:
        sol.set_choice_draws(False)
    checked, counts = cd.check_mechanism(cd.ChoiceCells(sol, m), sims, cd.philox_uniforms(n, m.nt, 12345, agent0=5))
    assert checked >= 300 and (counts > 0).all(), (checked, counts)


def test_draws_do_not_depend_on_sharding_and_moments_sum_the_records():
    m, lib, sol = _solved()
    n = 2048  # modal mode would take the two-periods-per-write kernel at this size
    init = _init(m, n, seed=3)
    init[::97, 1] = m.a0 - 1.0  # skipped agents: NaN from period 0
    sol.set_choice_draws(True)
    try:
        full, mom = _device(lib, m, sol, init, 0)
        nan = np.isnan(full)
        assert nan.any() and not nan.all()
        for lo in range(0, n, 256):
            part, _ = _device(lib, m, sol, init[lo:lo + 256], lo)
            assert np.array_equal(np.isnan(part), nan[lo:lo + 256])
            assert np.array_equal(part[~nan[lo:lo + 256]].view(np.int64), full[lo:lo + 256][~nan[lo:lo + 256]].view(np.int64))
    finally:
        sol.set_choice_draws(False)
    s1 = np.where(nan, 0.0, full).sum(axis=0)
    s2 = np.where(nan, 0.0, full * full).sum(axis=0)
    fin = np.isfinite(s1)
    assert np.allclose(mom[..., 0][fin], s1[fin], rtol=1e-11, atol=1e-9)
    assert np.allclose(mom[..., 1][fin], s2[fin], rtol=1e-11, atol=1e-9)
    assert np.array_equal(mom[..., 2], (~nan).sum(axis=0).astype(float))


def test_modal_simulation_is_unchanged_by_the_setting():
    m, lib, sol = _solved()
    init = _init(m, 300, seed=4)
    rs = np.random.default_rng(8).random(4 * m.nt * 300)
    before = lib.simulate(m, sol, init, rs)
    sol.set_choice_draws(True)
    drawn = lib.simulate(m, sol, init, rs)
    sol.set_choice_draws(False)
    after = lib.simulate(m, sol, init, rs)
    assert np.array_equal(before.view(np.int64), after.view(np.int64))
    assert not np.array_equal(np.nan_to_num(before[:, :, cd.DEC]), np.nan_to_num(drawn[:, :, cd.DEC]))
    # EgdstModel.sim sets the mode on every call
    m.__dict__["_solution"] = sol
    m.__dict__["_lib"] = lib
    m.__dict__["needtocompile"] = False
    assert np.array_equal(m.sim(init, randstream=rs, draw_choices=True).sims.view(np.int64), drawn.view(np.int64))
    assert np.array_equal(m.sim(init, randstream=rs).sims.view(np.int64), before.view(np.int64))


def test_draws_are_refused_without_choice_cells():
    from build import build  # tools/hostemu/build.py
    m, lib, sol = _solved()
    imported = lib.import_solution(m, sol.M, sol.D)
    with pytest.raises(capi.EgdstError) as e:
        imported.set_choice_draws(True)
    assert e.value.code == 2 and "imported" in str(e.value)
    imported.set_choice_draws(False)
    m2 = examples.retirement2(T=6, ngridm=40, ngridmax=200, ny=4)
    m2.prepare()
    lib2 = capi.ModelLibrary(build(m2))
    sol2 = lib2.solve(m2)
    with pytest.raises(capi.EgdstError) as e:
        sol2.set_choice_draws(True)
    assert e.value.code == 2 and "sigma_eps" in str(e.value)
    sol2.set_choice_draws(False)
