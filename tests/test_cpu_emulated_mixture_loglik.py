"""Finite-mixture log-likelihood over unobserved types (egdst_mixture_loglik) on the host emulator of the kernels: the
numpy oracle of tests/mixture_loglik_checks.py on a ragged panel of a batched retirement2_smooth solve, zero and
unnormalised weights, one type as the plain per-individual likelihood, determinism across mixture batches and vector
windows, the device variant's NaN rules, an individual with an unavailable decision, and the refusals."""
import shutil
import sys
import os

import numpy as np
import pytest

from egdst_b200 import capi, examples
from tests import mixture_loglik_checks as mc

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "tools", "hostemu"))

pytestmark = pytest.mark.skipif(shutil.which("g++") is None, reason="g++ not available")

_CACHE = {}
DUW = (0.35, 0.5, 0.65)
# four mixtures of three types: zero weights, unnormalised weights, a vector repeated across types
TVEC = np.array([[0, 1, 2], [1, 1, 0], [2, 0, 1], [0, 2, 1]])
W = np.array([[0.2, 0.3, 0.5], [1.0, 2.0, 3.0], [0.0, 4.0, 1.0], [0.0, 0.0, 7.0]])


def _solved():
    """retirement2_smooth (T=6), sigma_eps = 0.2, solved on the emulator for three values of duw in one batch."""
    if "sol" not in _CACHE:
        from build import build  # tools/hostemu/build.py
        m = examples.retirement2_smooth(sigma_eps=0.2, T=6, ngridm=100, ngridmax=300, ny=5)
        m.prepare()
        lib = capi.ModelLibrary(build(m))
        names = [p["ref"] for p in m.param]
        pv = np.array([list(m.param_vector())] * len(DUW))
        pv[:, names.index("duw")] = DUW
        sol = lib.solve_batch(m, pv)
        for v in range(len(DUW)):
            assert sol.status(v)[0] == 0, (v, sol.status(v))
        _CACHE["sol"] = (m, lib, sol, pv)
    return _CACHE["sol"]


def _panel(n=240):
    """Draw panel of n agents under vector 1, made ragged: every 7th agent has no record (empty individual), every 5th
    keeps only its first record (one-row individual)."""
    if "panel" not in _CACHE:
        m, lib, sol, _ = _solved()
        rng = np.random.default_rng(4)
        init = np.column_stack([np.ones(n), m.a0 + 0.6 * (m.mmax - m.a0) * rng.random(n)])
        sol.set_choice_draws(True)
        try:
            sims, _ = lib.simulate_philox(m, sol, init, seed=77, ivec=1)
        finally:
            sol.set_choice_draws(False)
        sims = sims.copy()
        sims[::7] = np.nan
        sims[3::5, 1:] = np.nan
        obs, start = capi.observations_from_sims(m, sims, start=True)
        sizes = np.diff(start)
        assert np.any(sizes == 0) and np.any(sizes == 1) and sizes.max() > 1
        _CACHE["panel"] = (obs, start)
    return _CACHE["panel"]


def test_oracle_on_a_ragged_panel():
    m, lib, sol, _ = _solved()
    obs, start = _panel()
    tot, indll, mixll, post = mc.check_against_oracle(lib, m, sol, obs, start, TVEC, W, sigma_c=0.1)
    assert np.all(np.isfinite(tot)) and np.all(np.isfinite(mixll))
    empty = np.diff(start) == 0
    assert np.all(indll[:, empty] == 0.0)
    # posteriors sum to one; zero-weight types get exactly 0
    np.testing.assert_allclose(post.sum(axis=1), 1.0, rtol=0, atol=1e-12)
    assert np.all(post[2, 0] == 0.0) and np.all(post[3, :2] == 0.0)
    # a single positive weight: the mixture is that type's likelihood and its posterior is 1
    np.testing.assert_allclose(mixll[3], indll[1], rtol=1e-15, atol=0)
    assert np.all(post[3, 2] == 1.0)


def test_one_type_is_the_per_individual_likelihood():
    m, lib, sol, _ = _solved()
    obs, start = _panel()
    for wt in (1.0, 2.5):
        tot, indll, mixll, post = lib.mixture_loglik(m, sol, obs, start, [[0], [1], [2]], [[wt]] * 3, individuals=True,
                                                     posterior=True)
        assert np.array_equal(mc.bits(mixll), mc.bits(indll)), wt
        assert np.all(post == 1.0)
        t1 = lib.choice_loglik(m, sol, obs)
        np.testing.assert_allclose(tot, t1, rtol=1e-12, atol=0)


def test_mixtures_alone_equal_mixtures_in_a_batch_and_across_windows():
    m, lib, sol, _ = _solved()
    obs, start = _panel()
    tot, indll, mixll, post = lib.mixture_loglik(m, sol, obs, start, TVEC, W, sigma_c=0.1, individuals=True, posterior=True)
    for x in range(TVEC.shape[0]):
        t1, i1, m1, p1 = lib.mixture_loglik(m, sol, obs, start, TVEC[x], W[x], sigma_c=0.1, individuals=True, posterior=True)
        assert np.array_equal(mc.bits(t1), mc.bits(tot[x:x + 1])), x
        assert np.array_equal(mc.bits(m1), mc.bits(mixll[x:x + 1])), x
        assert np.array_equal(mc.bits(p1), mc.bits(post[x:x + 1])), x
        assert np.array_equal(mc.bits(i1), mc.bits(indll)), x
    # vectors 1 and 2 through the window 0..2 and through the window 1..2
    a = lib.mixture_loglik(m, sol, obs, start, [1, 2], [0.4, 0.6], sigma_c=0.1, individuals=True, posterior=True)
    b = lib.mixture_loglik(m, sol, obs, start, [0, 1], [0.4, 0.6], sigma_c=0.1, ivec0=1, nvec=2, individuals=True,
                           posterior=True)
    assert np.array_equal(mc.bits(a[0]), mc.bits(b[0]))
    assert np.array_equal(mc.bits(a[1][1:]), mc.bits(b[1]))
    assert np.array_equal(mc.bits(a[2]), mc.bits(b[2])) and np.array_equal(mc.bits(a[3]), mc.bits(b[3]))


def test_type_model_entry_point():
    m, lib, sol, pv = _solved()
    obs, start = _panel()
    m.__dict__["_lib"] = lib
    m.__dict__["needtocompile"] = False
    tot, post = m.mixture_loglik(obs, start, pv[[0, 2]], [3.0, 7.0], sigma_c=0.1, posterior=True)
    want = lib.mixture_loglik(m, sol, obs, start, [0, 2], [0.3, 0.7], sigma_c=0.1, posterior=True)
    assert abs(tot - want[0][0]) <= 1e-12 * abs(tot)
    np.testing.assert_allclose(post, want[1][0], rtol=0, atol=1e-12)
    # one type: the descriptor carries the type's parameter values
    t1 = m.mixture_loglik(obs, start, pv[[2]], [1.0])
    assert abs(t1 - lib.choice_loglik(m, sol, obs, ivec0=2, nvec=1)[0]) <= 1e-12 * abs(t1)


def test_device_variant_confines_nan_to_the_malformed_individual():
    m, lib, sol, _ = _solved()
    obs, start = _panel()
    obs = obs.copy()
    j = int(np.nonzero(np.diff(start) > 2)[0][3])  # an individual with several rows; its second row gets state 0
    obs[start[j] + 1, 1] = 0.0
    nobs, k = obs.shape
    nind, (nmix, ntypes) = start.size - 1, TVEC.shape
    # a fifth mixture with a type vector out of range under zero weight: skipped
    tv = np.ascontiguousarray(np.vstack([TVEC, [1, 9, 2]]), dtype=np.int32)
    w = np.ascontiguousarray(np.vstack([W, [0.2, 0.0, 0.5]]))
    nmix += 1
    obsf = np.ascontiguousarray(obs.ravel(order="F"))
    st = np.ascontiguousarray(start, dtype=np.int32)
    tot = np.zeros(nmix)
    indll = np.full((3, nind), 7.0)
    mixll = np.full((nmix, nind), 7.0)
    post = np.full((nmix, ntypes, nind), 7.0)
    lib.mixture_loglik_device(m, sol, obsf.ctypes.data, nobs, k, st.ctypes.data, nind, tv.ctypes.data, w.ctypes.data,
                              ntypes, nmix, tot.ctypes.data, sigma_c=0.1, d_indll=indll.ctypes.data,
                              d_mixll=mixll.ctypes.data, d_post=post.ctypes.data)
    others = np.arange(nind) != j
    assert np.all(np.isnan(indll[:, j])) and np.all(np.isfinite(indll[:, others]))
    assert np.all(np.isnan(mixll[:, j])) and np.all(np.isfinite(mixll[:, others]))
    assert np.all(np.isnan(tot))
    assert np.all(np.isnan(post[:, :, j][w > 0])) and np.all(post[:, :, j][w == 0] == 0.0)
    assert np.all(np.isfinite(post[:, :, others]))
    # the other individuals have the host entry point's values; the zero-weight type out of range does not matter
    good = obs.copy()
    good[start[j] + 1, 1] = 1.0
    _, i0, m0, p0 = lib.mixture_loglik(m, sol, good, start, np.vstack([TVEC, [1, 0, 2]]), w, sigma_c=0.1,
                                       individuals=True, posterior=True)
    assert np.array_equal(mc.bits(indll[:, others]), mc.bits(i0[:, others]))
    assert np.array_equal(mc.bits(mixll[:, others]), mc.bits(m0[:, others]))
    assert np.array_equal(mc.bits(post[:, :, others]), mc.bits(p0[:, :, others]))
    # totals accumulate into the caller's buffer
    tot2 = np.ones(nmix)
    good_f = np.ascontiguousarray(good.ravel(order="F"))
    lib.mixture_loglik_device(m, sol, good_f.ctypes.data, nobs, k, st.ctypes.data, nind, tv.ctypes.data, w.ctypes.data,
                              ntypes, nmix, tot2.ctypes.data, sigma_c=0.1)
    t0 = lib.mixture_loglik(m, sol, good, start, np.vstack([TVEC, [1, 0, 2]]), w, sigma_c=0.1)
    assert np.array_equal(mc.bits(tot2), mc.bits(1.0 + t0))


def test_an_unavailable_decision_makes_its_individual_minus_infinity():
    from build import build  # tools/hostemu/build.py
    m = examples.model2()
    m.sigma_eps = 0.2
    m.prepare()
    lib = capi.ModelLibrary(build(m))
    sol = lib.solve(m)
    assert sol.status()[0] == 0, sol.status()
    # individual 0 works in the absorbing retired state (decision 2 is not available there); 1 has ordinary rows;
    # 2 is empty; 3 has one row
    obs = np.array([[m.t0, 2, 5.0, 1], [m.t0 + 1, 1, 20.0, 2], [m.t0, 2, 5.0, 2], [m.t0 + 1, 2, 8.0, 1],
                    [m.t0, 2, 6.0, 1]], dtype=float)
    start = [0, 2, 4, 4, 5]
    tot, indll, mixll, post = mc.check_against_oracle(lib, m, sol, obs, start, [[0, 0], [0, 0]], [[1.0, 1.0], [0.0, 2.0]])
    assert indll[0, 0] == -np.inf and np.all(np.isfinite(indll[0, 1:])) and indll[0, 2] == 0.0
    assert np.all(mixll[:, 0] == -np.inf) and np.all(np.isfinite(mixll[:, 1:]))
    assert np.all(np.isnan(post[0, :, 0])) and np.isnan(post[1, 1, 0]) and post[1, 0, 0] == 0.0
    assert np.all(tot == -np.inf)


def test_refusals():
    from build import build  # tools/hostemu/build.py
    m, lib, sol, _ = _solved()
    obs, start = _panel()
    nobs, nind = obs.shape[0], start.size - 1

    def refused(fn, *words):
        with pytest.raises(capi.EgdstError) as e:
            fn()
        assert e.value.code == 2 and all(w in str(e.value) for w in words), str(e.value)

    def mix(o=obs, s=start, tv=TVEC, w=W, **kw):
        return lib.mixture_loglik(m, sol, o, s, tv, w, **kw)

    bad = start.copy()
    bad[0] = 1
    refused(lambda: mix(s=bad), "start[0] = 1")
    bad = start.copy()
    bad[5] = bad[6] + 1
    refused(lambda: mix(s=bad), "decreases at individual 5")
    bad = start.copy()
    bad[-1] -= 1
    refused(lambda: mix(s=bad), "start[%d]" % nind, "nobs = %d" % nobs)
    tv = TVEC.copy()
    tv[2, 1] = 3
    refused(lambda: mix(tv=tv), "mixture 2, type 1", "vector 3 is not in 0..2")
    refused(lambda: mix(tv=TVEC - 1, ivec0=1, nvec=2), "mixture 0, type 0", "vector -1")
    w = W.copy()
    w[1, 2] = -0.5
    refused(lambda: mix(w=w), "mixture 1, type 2", "negative or not finite")
    w[1, 2] = np.inf
    refused(lambda: mix(w=w), "mixture 1, type 2", "negative or not finite")
    w = W.copy()
    w[3] = 0.0
    refused(lambda: mix(w=w), "mixture 3 sum to 0")
    refused(lambda: mix(tv=np.zeros((1, 0)), w=np.zeros((1, 0))), "ntypes and nmix")
    refused(lambda: mix(tv=np.zeros((65536, 1)), w=np.ones((65536, 1))), "65535 mixtures")
    # the checks of the choice log-likelihood, with their messages
    o = obs.copy()
    o[4, 3] = 0
    refused(lambda: mix(o=o), "obs row 4", "decision")
    refused(lambda: mix(o=obs[:, :3]), "4 or 5")
    refused(lambda: mix(sigma_c=-1.0), "sigma_c")
    refused(lambda: mix(ivec0=2, nvec=2), "out of range")
    imported = lib.import_solution(m, sol.M, sol.D)
    refused(lambda: lib.mixture_loglik(m, imported, obs, start, [0], [1.0]), "imported")
    # the device variant checks the sizes
    z = np.zeros(4)
    refused(lambda: lib.mixture_loglik_device(m, sol, z.ctypes.data, 0, 4, z.ctypes.data, -1, z.ctypes.data, z.ctypes.data,
                                              1, 1, z.ctypes.data), "nind < 0")
    refused(lambda: lib.mixture_loglik_device(m, sol, z.ctypes.data, 0, 4, z.ctypes.data, 0, z.ctypes.data, z.ctypes.data,
                                              0, 1, z.ctypes.data), "ntypes and nmix")
    # an image without taste shocks
    m2 = examples.retirement2(T=6, ngridm=40, ngridmax=200, ny=4)
    m2.prepare()
    lib2 = capi.ModelLibrary(build(m2))
    sol2 = lib2.solve(m2)
    refused(lambda: lib2.mixture_loglik(m2, sol2, obs[:, :4], start, [0], [1.0]), "sigma_eps")
