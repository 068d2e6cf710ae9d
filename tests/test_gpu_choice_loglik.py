"""Choice log-likelihood of the smoothing mode (egdst_choice_loglik) on the GPU: the row values against numpy at full
size, large launches against small ones, recovery of the disutility of work from a simulated panel, and the limit
sigma_eps -> 0 (tests/choice_loglik_checks.py)."""
import numpy as np
import pytest
import torch

from egdst_b200 import capi, examples
from tests import choice_draw_checks as cd
from tests import choice_loglik_checks as cl

pytestmark = pytest.mark.gpu


def _solved(sigma_eps, **kw):
    m = examples.retirement2_smooth(sigma_eps=sigma_eps, **kw)
    m.compile()
    lib = m._capi()
    sol = lib.solve(m, strict=True)
    return m, lib, sol


def _init(m, n, seed=1):
    rng = np.random.default_rng(seed)
    return np.column_stack([np.ones(n), m.a0 + 0.6 * (m.mmax - m.a0) * rng.random(n)])


@pytest.mark.parametrize("sigma_eps", [0.2, 0.05])
def test_rows_are_the_log_choice_probabilities(sigma_eps):
    m, lib, sol = _solved(sigma_eps)
    n = 20000
    rs = np.random.default_rng(7).random(4 * m.nt * n)
    sol.set_choice_draws(True)
    sims = lib.simulate(m, sol, _init(m, n), rs)
    sol.set_choice_draws(False)
    cl.check_mechanism(cd.ChoiceCells(sol, m), lib, sims, min_rows=10000)


def test_large_launches_hold_the_rows_of_small_ones():
    m, lib, sol = _solved(0.2)
    obs, _ = cl.recovery_panel(lib, m, sol, 100_000, seed=11)
    assert obs.shape[0] >= 2_000_000, obs.shape
    dev = torch.device("cuda", 0)
    desc = capi.Desc(m)
    small = 1024
    out = []
    for o in (obs, obs[:small]):
        n = o.shape[0]
        d_obs = torch.from_numpy(np.ascontiguousarray(o.ravel(order="F"))).to(dev)
        d_tot = torch.zeros(1, dtype=torch.float64, device=dev)
        d_row = torch.full((n,), 7.0, dtype=torch.float64, device=dev)
        lib.choice_loglik_device(m, sol, d_obs.data_ptr(), n, 5, d_tot.data_ptr(), sigma_c=0.05, d_rowll=d_row.data_ptr(), desc=desc)
        torch.cuda.synchronize()
        out.append((d_tot.cpu().numpy(), d_row.cpu().numpy()))
    (tb, rb), (ts, rs) = out
    assert np.array_equal(rb[:small].view(np.int64), rs.view(np.int64))
    assert not np.isnan(rb).any()
    cl.check_total(tb[0], rb)
    cl.check_total(ts[0], rs)


def test_recovery_of_the_disutility_of_work():
    m, lib, sol = _solved(0.2)
    obs, _ = cl.recovery_panel(lib, m, sol, 200_000, seed=2024)
    names = [p["ref"] for p in m.param]
    j = np.arange(-4, 5)
    pv = np.array([list(m.param_vector())] * j.size)
    duw0 = pv[0, names.index("duw")]
    assert duw0 == 0.5
    pv[:, names.index("duw")] = duw0 * (1.0 + 0.05 * j)
    bsol = lib.solve_batch(m, pv)
    for v in range(j.size):
        assert bsol.status(v)[0] == 0, (v, bsol.status(v))
    tot = lib.choice_loglik(m, bsol, obs, sigma_c=0.0)
    assert np.all(np.isfinite(tot)), tot
    assert int(np.argmax(tot)) == 4, tot
    assert np.all(np.diff(tot[:5]) > 0) and np.all(np.diff(tot[4:]) < 0), tot


def test_vanishing_taste_shocks_give_the_modal_choice_probability_one():
    m, lib, sol = _solved(1e-8)
    n = 20000
    rs = np.random.default_rng(9).random(4 * m.nt * n)
    modal = lib.simulate(m, sol, _init(m, n, seed=3), rs)
    obs = capi.observations_from_sims(m, modal, consumption=False)
    assert obs.shape[0] > 100_000
    _, r = lib.choice_loglik(m, sol, obs, rows=True)
    assert np.mean(r[0] >= -1e-9) >= 0.999, np.mean(r[0] >= -1e-9)
