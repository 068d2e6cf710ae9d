"""Host logic of the sharded mixture log-likelihood (distributed.mixture_loglik_sharded), world size 2 on CPU (gloo):
the blocks of individuals tile the panel, each block's rows follow the offsets, and the all-reduced totals equal the
single-process result."""
import os
import socket

import numpy as np
import pytest

from egdst_b200 import distributed as D

NMIX = 2


def _panel():
    rng = np.random.default_rng(8)
    sizes = rng.integers(0, 6, 41)
    sizes[[3, 20, 21]] = 0
    start = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
    n = int(start[-1])
    obs = np.column_stack([rng.integers(20, 30, n), np.ones(n), rng.random(n) * 5, rng.integers(1, 3, n)]).astype(float)
    return obs, start


def _fake(block, sblock):
    """Stand-in for the CUDA call: per-individual sums of a function of each row, and their totals per mixture."""
    assert sblock[0] == 0 and sblock[-1] == block.shape[0] and np.all(np.diff(sblock) >= 0)
    ind = np.array([np.sum(-block[sblock[i]:sblock[i + 1], 2]) for i in range(sblock.size - 1)])
    mix = np.array([(x + 1) * ind for x in range(NMIX)]).reshape(NMIX, ind.size)
    return mix.sum(axis=1), mix, block[:, 2].copy()


def _worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    obs, start = _panel()
    tot, parts, (lo, hi) = D.mixture_loglik_sharded(None, None, None, obs, start, None, None, fn=_fake)
    q.put((rank, lo, hi, tot, parts))
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
    want, (mix, cash), (lo, hi) = D.mixture_loglik_sharded(None, None, None, obs, start, None, None, fn=_fake, rank=0, world=1)
    assert (lo, hi) == (0, 41)
    assert (res[0][1], res[0][2], res[1][1], res[1][2]) == (0, 21, 21, 41)
    # the blocks tile the individuals and their rows follow start
    np.testing.assert_array_equal(np.hstack([r[4][0] for r in res]), mix)
    np.testing.assert_array_equal(res[0][4][1], obs[:start[21], 2])
    np.testing.assert_array_equal(res[1][4][1], obs[start[21]:, 2])
    for r in res:
        np.testing.assert_allclose(r[3], want, rtol=1e-13, atol=0)
