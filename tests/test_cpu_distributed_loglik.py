"""Host logic of the sharded choice log-likelihood (distributed.choice_loglik_sharded), world size 2 on CPU (gloo): the
observation blocks tile the panel and the all-reduced totals equal the single-process result."""
import os
import socket

import numpy as np
import pytest

from egdst_b200 import distributed as D

NVEC = 3


def _obs():
    rng = np.random.default_rng(3)
    return np.column_stack([rng.integers(20, 30, 101), np.ones(101), rng.random(101) * 5, rng.integers(1, 3, 101)]).astype(float)


def _fake_loglik(block):
    """Stand-in for the CUDA call: per-vector sums of a function of each row."""
    return np.array([np.sum(-(v + 1) * block[:, 2] - block[:, 3]) for v in range(NVEC)])


def _worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    tot, (lo, hi) = D.choice_loglik_sharded(None, None, None, _obs(), loglik_fn=_fake_loglik)
    q.put((rank, lo, hi, tot))
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
    want, (lo, hi) = D.choice_loglik_sharded(None, None, None, _obs(), loglik_fn=_fake_loglik, rank=0, world=1)
    assert (lo, hi) == (0, 101)
    assert (res[0][1], res[0][2], res[1][1], res[1][2]) == (0, 51, 51, 101)
    for r in res:
        np.testing.assert_allclose(r[3], want, rtol=1e-13, atol=0)
