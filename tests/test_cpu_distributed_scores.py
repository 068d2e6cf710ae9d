"""Host logic of the sharded mixture scores (distributed.mixture_scores_sharded), world size 2 on CPU (gloo): the
blocks of individuals tile the panel with rebased offsets, and the one all-reduce of totals, gradient and OPG gives the
single-process result."""
import os
import socket

import numpy as np
import pytest

from egdst_b200 import distributed as D

NMIX, NPAR = 3, 2


def _panel():
    rng = np.random.default_rng(9)
    sizes = rng.integers(0, 6, 41)
    sizes[[3, 20, 21]] = 0
    start = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
    n = int(start[-1])
    obs = np.column_stack([rng.integers(20, 30, n), np.ones(n), rng.random(n) * 5, rng.integers(1, 3, n)]).astype(float)
    return obs, start


def _fake(block, sblock):
    """Stand-in for the CUDA call: per-individual mixture values from the rows, their totals, and the scores' sums."""
    assert sblock[0] == 0 and sblock[-1] == block.shape[0] and np.all(np.diff(sblock) >= 0)
    ind = np.array([np.sum(-block[sblock[i]:sblock[i + 1], 2]) for i in range(sblock.size - 1)])
    mix = np.array([(x + 1) * ind + x * ind ** 2 for x in range(NMIX)]).reshape(NMIX, ind.size)
    s = np.array([mix[1] - mix[0], (mix[2] - mix[0]) * 0.5])
    return mix.sum(axis=1), s.sum(axis=1), s @ s.T


def _worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    obs, start = _panel()
    tot, grad, opg, (lo, hi) = D.mixture_scores_sharded(None, None, None, obs, start, None, None, None, None, None, fn=_fake)
    q.put((rank, lo, hi, tot, grad, opg))
    dist.barrier()
    dist.destroy_process_group()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.timeout(120)
def test_world2_gloo_matches_single_process():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=90) for _ in procs], key=lambda x: x[0])
    for p in procs:
        p.join(30)
        assert p.exitcode == 0
    obs, start = _panel()
    want = _fake(obs, start)
    tot, grad, opg, (lo, hi) = D.mixture_scores_sharded(None, None, None, obs, start, None, None, None, None, None, fn=_fake,
                                                        rank=0, world=1)
    assert (lo, hi) == (0, 41)
    assert (res[0][1], res[0][2], res[1][1], res[1][2]) == (0, 21, 21, 41)
    for r in res + [(0, 0, 0, tot, grad, opg)]:
        assert r[5].shape == (NPAR, NPAR)
        for got, exp in zip(r[3:], want):
            np.testing.assert_allclose(got, exp, rtol=1e-12, atol=0)
