"""Central-difference mixture scores (egdst_mixture_scores) on the host emulator of the kernels, retirement2_smooth
(T=6) with a three-parameter stencil (duw, wage, interest; 7 vectors) and two type vectors: the oracle of
tests/score_checks.py on a ragged panel, bit-identity of every entry across component subsets, orders and vector
windows, a forward difference, type-weight scores against the posterior identity, NaN scores for an individual with
an unavailable decision, the device variant's NaN confinement, the refusals, and the EgdstModel entry points."""
import shutil
import sys
import os

import numpy as np
import pytest

from egdst_b200 import capi, examples
from tests import score_checks as sc
from tests.mixture_loglik_checks import bits

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "tools", "hostemu"))

pytestmark = pytest.mark.skipif(shutil.which("g++") is None, reason="g++ not available")

_CACHE = {}
FREE = ["duw", "wage", "interest"]
TYPES = (0.35, 0.65)  # duw of the two type vectors 7 and 8
SIGMA_C = 0.1


def _model():
    m = examples.retirement2_smooth(sigma_eps=0.2, T=6, ngridm=100, ngridmax=300, ny=5)
    m.prepare()
    return m


def _solved():
    """The stencil of FREE around the defaults (vectors 0..6, centre first) and the two type vectors, one batch."""
    if "sol" not in _CACHE:
        from build import build  # tools/hostemu/build.py
        m = _model()
        lib = capi.ModelLibrary(build(m))
        names = [p["ref"] for p in m.param]
        idx = [names.index(f) for f in FREE]
        pv, mplus, mminus, hinv = sc.stencil(m.param_vector(), idx)
        types = np.tile(m.param_vector(), (len(TYPES), 1))
        types[:, names.index("duw")] = TYPES
        sol = lib.solve_batch(m, np.vstack([pv, types]))
        for v in range(sol.nvec):
            assert sol.status(v)[0] == 0, (v, sol.status(v))
        _CACHE["sol"] = (m, lib, sol, pv, mplus, mminus, hinv)
    return _CACHE["sol"]


def _panel(n=240):
    """Draw panel of n agents under the centre vector, made ragged: every 7th agent has no record (empty individual),
    every 5th keeps only its first record (one-row individual)."""
    if "panel" not in _CACHE:
        m, lib, sol = _solved()[:3]
        rng = np.random.default_rng(5)
        init = np.column_stack([np.ones(n), m.a0 + 0.6 * (m.mmax - m.a0) * rng.random(n)])
        sol.set_choice_draws(True)
        try:
            sims, _ = lib.simulate_philox(m, sol, init, seed=78, ivec=0)
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


def _stencil_call(comps=(0, 1, 2), **kw):
    m, lib, sol, _, mplus, mminus, hinv = _solved()
    obs, start = _panel()
    tv, w = sc.one_type(7)
    c = list(comps)
    return lib.mixture_scores(m, sol, obs, start, tv, w, mplus[c], mminus[c], hinv[c], sigma_c=SIGMA_C, scores=True, **kw)


def test_oracle_on_a_ragged_panel():
    m, lib, sol, _, mplus, mminus, hinv = _solved()
    obs, start = _panel()
    tv, w = sc.one_type(7)
    tot, grad, opg, s, mixll = sc.check_against_oracle(lib, m, sol, obs, start, tv, w, mplus, mminus, hinv, sigma_c=SIGMA_C)
    assert np.all(np.isfinite(s)) and np.all(np.isfinite(opg)) and np.all(np.isfinite(tot))
    assert np.all(s[:, np.diff(start) == 0] == 0.0)
    assert start.size - 1 > 2 * 16  # several blocks of the emulator's 16-individual chunk
    # the OPG is positive definite and the gradient is that of the totals
    assert np.all(np.linalg.eigvalsh(opg) > 0)
    np.testing.assert_allclose(grad, (tot[mplus] - tot[mminus]) * hinv, rtol=1e-9, atol=1e-9)
    # a plain one-type likelihood: the mixture totals are the choice log-likelihood's
    np.testing.assert_allclose(tot, lib.choice_loglik(m, sol, obs, sigma_c=SIGMA_C, nvec=7), rtol=1e-12, atol=0)


def test_entries_do_not_depend_on_the_other_components():
    tot, grad, opg, s = _stencil_call()
    for order in ([2, 0, 1], [1], [2, 1], [0, 1, 2, 2, 0]):
        t2, g2, o2, s2 = _stencil_call(order)
        assert sc.same(t2, tot)
        for a, p in enumerate(order):
            assert sc.same(g2[a], grad[p]) and sc.same(s2[a], s[p]), (order, p)
            for b, q in enumerate(order):
                assert sc.same(o2[a, b], opg[p, q]), (order, p, q)


def test_entries_do_not_depend_on_the_window():
    m, lib, sol, _, mplus, mminus, hinv = _solved()
    obs, start = _panel()
    tot, grad, opg, s = _stencil_call()
    # the same differences through the window 1..6 (without the centre) and through all nine vectors
    tv, w = sc.one_type(6)
    t1, g1, o1, s1 = lib.mixture_scores(m, sol, obs, start, tv, w, mplus - 1, mminus - 1, hinv, sigma_c=SIGMA_C, ivec0=1,
                                        nvec=6, scores=True)
    assert sc.same(g1, grad) and sc.same(o1, opg) and sc.same(s1, s) and sc.same(t1, tot[1:])
    tv, w = sc.one_type(9)
    t9, g9, o9, s9 = lib.mixture_scores(m, sol, obs, start, tv, w, mplus, mminus, hinv, sigma_c=SIGMA_C, scores=True)
    assert sc.same(g9, grad) and sc.same(o9, opg) and sc.same(s9, s) and sc.same(t9[:7], tot)


def test_forward_difference():
    m, lib, sol, pv, mplus, mminus, hinv = _solved()
    obs, start = _panel()
    tv, w = sc.one_type(7)
    names = [p["ref"] for p in m.param]
    j = names.index("duw")
    hf = 1.0 / (pv[1, j] - pv[0, j])
    _, gf, of, sf, _ = sc.check_against_oracle(lib, m, sol, obs, start, tv, w, [1], [0], [hf], sigma_c=SIGMA_C)
    _, gc, _, scen = _stencil_call([0])
    # the forward difference has the central one's leading term
    np.testing.assert_allclose(sf[0], scen[0], rtol=0, atol=1e-3 * np.abs(scen[0]).max())
    np.testing.assert_allclose(gf, gc, rtol=1e-2)


def test_type_weight_scores_are_the_posterior_identity():
    m, lib, sol = _solved()[:3]
    obs, start = _panel()
    pi, h = 0.3, 1e-4
    tv = [[7, 8]] * 3
    w = [[pi, 1 - pi], [pi + h, 1 - pi - h], [pi - h, 1 - pi + h]]
    hinv = 1.0 / ((pi + h) - (pi - h))
    _, _, _, s, _ = sc.check_against_oracle(lib, m, sol, obs, start, tv, w, [1], [2], [hinv], sigma_c=SIGMA_C)
    _, post = lib.mixture_loglik(m, sol, obs, start, [7, 8], [pi, 1 - pi], sigma_c=SIGMA_C, posterior=True)
    want = post[0, 0] / pi - post[0, 1] / (1 - pi)
    np.testing.assert_allclose(s[0], want, rtol=1e-6, atol=1e-6)


def test_an_unavailable_decision_gives_nan_scores():
    from build import build  # tools/hostemu/build.py
    m = examples.model2()
    m.sigma_eps = 0.2
    m.prepare()
    lib = capi.ModelLibrary(build(m))
    sol = lib.solve(m)
    assert sol.status()[0] == 0, sol.status()
    # individual 0 works in the absorbing retired state (decision 2 is not available there); 2 is empty
    obs = np.array([[m.t0, 2, 5.0, 1], [m.t0 + 1, 1, 20.0, 2], [m.t0, 2, 5.0, 2], [m.t0 + 1, 2, 8.0, 1],
                    [m.t0, 2, 6.0, 1]], dtype=float)
    start = [0, 2, 4, 4, 5]
    # two one-type mixtures of the same vector (weights 1 and 2 normalise alike): -inf under both for individual 0
    tot, grad, opg, s, mixll = sc.check_against_oracle(lib, m, sol, obs, start, [[0], [0]], [[1.0], [2.0]], [0, 1], [1, 0],
                                                       [1.0, -2.0])
    assert np.all(mixll[:, 0] == -np.inf)
    assert np.all(np.isnan(s[:, 0])) and np.all(s[:, 1:] == 0.0)
    assert np.all(np.isnan(grad)) and np.all(np.isnan(opg))


def test_device_variant_confines_nan_to_the_bad_component():
    m, lib, sol, _, mplus, mminus, hinv = _solved()
    obs, start = _panel()
    nobs, k = obs.shape
    nind, npar = start.size - 1, 4
    tv, w = sc.one_type(7)
    tv = np.ascontiguousarray(tv, dtype=np.int32)
    # component 3 names mixture 99: NaN, never a read out of bounds
    mp = np.ascontiguousarray(np.append(mplus, 99), dtype=np.int32)
    mm = np.ascontiguousarray(np.append(mminus, 0), dtype=np.int32)
    h = np.ascontiguousarray(np.append(hinv, 1.0))
    obsf = np.ascontiguousarray(obs.ravel(order="F"))
    st = np.ascontiguousarray(start, dtype=np.int32)
    tot, grad, opg = np.ones(7), np.ones(npar), np.ones((npar, npar))
    s = np.full((npar, nind), 7.0)
    lib.mixture_scores_device(m, sol, obsf.ctypes.data, nobs, k, st.ctypes.data, nind, tv.ctypes.data, w.ctypes.data, 1, 7,
                              npar, mp.ctypes.data, mm.ctypes.data, h.ctypes.data, tot.ctypes.data, grad.ctypes.data,
                              opg.ctypes.data, sigma_c=SIGMA_C, d_scores=s.ctypes.data)
    t0, g0, o0, s0 = _stencil_call()
    assert np.all(np.isnan(s[3])) and sc.same(s[:3], s0)
    assert np.isnan(grad[3]) and np.all(np.isnan(opg[3])) and np.all(np.isnan(opg[:, 3]))
    # the caller's buffers are added into
    assert sc.same(grad[:3], 1.0 + g0) and sc.same(opg[:3, :3], 1.0 + o0) and sc.same(tot, 1.0 + t0)


def test_refusals():
    from build import build  # tools/hostemu/build.py
    m, lib, sol, _, mplus, mminus, hinv = _solved()
    obs, start = _panel()
    tv, w = sc.one_type(7)

    def refused(fn, *words):
        with pytest.raises(capi.EgdstError) as e:
            fn()
        assert e.value.code == 2 and all(x in str(e.value) for x in words), str(e.value)

    def call(mp=mplus, mm=mminus, h=hinv, **kw):
        return lib.mixture_scores(m, sol, obs, start, kw.pop("tv", tv), kw.pop("w", w), mp, mm, h, **kw)

    refused(lambda: call([1] * 33, [2] * 33, [1.0] * 33), "npar = 33", "1..32")
    refused(lambda: call([], [], []), "npar = 0")
    refused(lambda: call([1, 7, 5], mminus), "component 1", "mplus 7 is not in 0..6")
    refused(lambda: call(mplus, [2, 4, -1]), "component 2", "mminus -1")
    for bad in (0.0, np.inf, np.nan):
        refused(lambda: call(h=[hinv[0], bad, hinv[2]]), "component 1", "hinv", "0 or not finite")
    # the checks of the mixture log-likelihood, with their messages
    bad = start.copy()
    bad[0] = 1
    refused(lambda: lib.mixture_scores(m, sol, obs, bad, tv, w, mplus, mminus, hinv), "start[0] = 1")
    refused(lambda: call(tv=tv + 3, nvec=7), "mixture 4, type 0", "vector 7 is not in 0..6")
    o = obs.copy()
    o[4, 3] = 0
    refused(lambda: lib.mixture_scores(m, sol, o, start, tv, w, mplus, mminus, hinv), "obs row 4", "decision")
    refused(lambda: call(sigma_c=-1.0), "sigma_c")
    # the device variant checks the sizes
    z = np.zeros(4)
    zi = np.zeros(4, dtype=np.int32)
    refused(lambda: lib.mixture_scores_device(m, sol, z.ctypes.data, 0, 4, zi.ctypes.data, 0, zi.ctypes.data, z.ctypes.data,
                                              1, 1, 33, zi.ctypes.data, zi.ctypes.data, z.ctypes.data, z.ctypes.data,
                                              z.ctypes.data, z.ctypes.data), "npar = 33")
    refused(lambda: lib.mixture_scores_device(m, sol, z.ctypes.data, 0, 4, zi.ctypes.data, 0, zi.ctypes.data, z.ctypes.data,
                                              1, 1, 1, zi.ctypes.data, zi.ctypes.data, z.ctypes.data, z.ctypes.data,
                                              z.ctypes.data, 0), "invalid arguments")
    # an image without taste shocks
    m2 = examples.retirement2(T=6, ngridm=40, ngridmax=200, ny=4)
    m2.prepare()
    lib2 = capi.ModelLibrary(build(m2))
    sol2 = lib2.solve(m2)
    refused(lambda: lib2.mixture_scores(m2, sol2, obs[:, :4], start, [0], [1.0], [0], [0], [1.0]), "sigma_eps")


def test_model_scores_and_fit():
    m, lib, sol, _, mplus, mminus, hinv = _solved()
    obs, start = _panel()
    m.__dict__["_lib"] = lib
    m.__dict__["needtocompile"] = False
    total, grad, opg = m.scores(obs, start, FREE, sigma_c=SIGMA_C)
    tot, g, o, _ = _stencil_call()
    assert sc.same(total, tot[0]) and sc.same(grad, g) and sc.same(opg, o)
    with pytest.raises(ValueError):
        m.scores(obs, start, ["duw", "nosuch"])
    with pytest.raises(ValueError):
        m.scores(obs, start, ["duw", "duw"])
    # BHHH in duw from 0.6 on the panel drawn at 0.5; the model's values are left as they were
    before = m.param_vector()
    m.setparam("duw", 0.6)
    try:
        est, se, tot1, g1, o1, it = m.fit(obs, start, ["duw"], sigma_c=SIGMA_C, maxiter=20)
        assert m.getparam("duw") == 0.6
    finally:
        m.setparam(before)
    assert 1 <= it <= 20 and tot1 > tot[0] - 1e-9 * abs(tot[0])
    assert abs(est[0] - 0.5) < 4 * se[0], (est, se)
    assert g1[0] ** 2 / o1[0, 0] < 1e-8 and se[0] == pytest.approx(1.0 / np.sqrt(o1[0, 0]), rel=1e-12)
    # an empty panel has zero scores: the OPG is singular
    with pytest.raises(np.linalg.LinAlgError):
        m.fit(obs[:0], np.zeros(3, dtype=np.int32), ["duw"])
