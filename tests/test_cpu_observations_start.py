"""capi.observations_from_sims with start=True: the offsets of each agent's rows, with agents that die early or have
no live record (empty individuals); the default return is unchanged."""
import numpy as np

from egdst_b200 import capi, examples


def _sims():
    m = examples.retirement2_smooth(T=6)
    rng = np.random.default_rng(5)
    nsim, nt, nso = 9, m.T - m.t0 + 1, m.nsimout()
    sims = rng.random((nsim, nt, nso)) * 4.0
    sims[:, :, 4] = rng.integers(0, 2, (nsim, nt))  # decision index
    sims[:, :, 5] = rng.integers(0, 2, (nsim, nt))  # state index
    sims[1, 3:] = np.nan   # dies after three periods
    sims[2] = np.nan       # skipped: no live record
    sims[5, :, 0] = np.nan  # no cash in any period
    sims[6, 1:] = np.nan   # one record
    sims[8] = np.nan       # the last agent is empty
    return m, sims


def test_offsets_follow_the_agents():
    m, sims = _sims()
    obs, start = capi.observations_from_sims(m, sims, start=True)
    assert start.dtype == np.int32 and start.shape == (sims.shape[0] + 1,)
    nt = sims.shape[1]
    assert list(np.diff(start)) == [nt, 3, 0, nt, nt, 0, 1, nt, 0]
    assert start[0] == 0 and start[-1] == obs.shape[0]
    assert np.array_equal(obs, capi.observations_from_sims(m, sims))
    for a in range(sims.shape[0]):
        rows = obs[start[a]:start[a + 1]]
        assert np.array_equal(rows[:, 2], sims[a, :rows.shape[0], 0])
        assert np.array_equal(rows[:, 0], m.t0 + np.arange(rows.shape[0]))


def test_without_consumption_and_without_records():
    m, sims = _sims()
    obs, start = capi.observations_from_sims(m, sims, consumption=False, start=True)
    assert obs.shape[1] == 4 and start[-1] == obs.shape[0]
    empty = np.full_like(sims, np.nan)
    obs, start = capi.observations_from_sims(m, empty, start=True)
    assert obs.shape == (0, 5) and np.array_equal(start, np.zeros(sims.shape[0] + 1))
    assert isinstance(capi.observations_from_sims(m, sims), np.ndarray)
