"""Multi-GPU sharding of the workloads that shard (SURVEY 8(e)): forward simulation over agents, batched solves over
parameter vectors, the choice log-likelihood over observations, and the mixture log-likelihood and its scores over
individuals.
One process per GPU; ``torch.distributed`` is plumbing only -- the single
collective on the data path is one all-reduce of the simulated-moment buffer (NCCL over NVLink on GPUs, gloo in
the CPU tests of the host logic).  A single model's backward induction does not shard ("replicas only"): every
rank solves it redundantly, bit-identically, which is cheaper than broadcasting the 16 MB arena every period.

Agents are numbered globally; the counter-based Philox stream is keyed by (seed; global agent id, period), so
simulated paths do not depend on the number of GPUs or on how agents are split.
"""
from __future__ import annotations

from typing import Callable, Optional, Tuple

import numpy as np


def shard_range(n: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous block partition of ``n`` items: rank r owns [lo, hi); sizes differ by at most one."""
    if world < 1 or not (0 <= rank < world):
        raise ValueError("invalid rank/world")
    base, rem = divmod(int(n), world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def _dist():
    import torch.distributed as dist
    return dist if dist.is_available() and dist.is_initialized() else None


def all_reduce_moments(moments, group=None):
    """Sum the moment buffer [3, nsimout, nt] (sum x, sum x^2, alive count) over all ranks, in place.
    ``moments`` is a torch tensor (CUDA with nccl, CPU with gloo) or a numpy array (gloo only)."""
    dist = _dist()
    if dist is None or dist.get_world_size(group) == 1:
        return moments
    import torch
    if isinstance(moments, np.ndarray):
        t = torch.from_numpy(moments)
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
        return moments
    dist.all_reduce(moments, op=dist.ReduceOp.SUM, group=group)
    return moments


def moments_to_stats(moments: np.ndarray):
    """(mean, variance, count) per [nsimout, nt] from the summed moment buffer."""
    s1, s2, n = moments[0], moments[1], moments[2]
    with np.errstate(invalid="ignore", divide="ignore"):
        mean = np.where(n > 0, s1 / n, np.nan)
        var = np.where(n > 0, s2 / n - mean * mean, np.nan)
    return mean, var, n


def simulate_sharded(lib, model, sol, init: np.ndarray, seed: int, rank: Optional[int] = None, world: Optional[int] = None,
                     want_sims: bool = True, simulate_fn: Optional[Callable] = None, group=None):
    """Simulate this rank's block of the global agent list ``init`` [nsim, 2] and all-reduce the moments.
    Returns (sims of the local block or None, global moments [3, nsimout, nt], (lo, hi)).
    ``simulate_fn(init_block, agent0) -> (sims, moments)`` replaces the CUDA call in the CPU tests."""
    dist = _dist()
    if world is None:
        world = dist.get_world_size(group) if dist else 1
    if rank is None:
        rank = dist.get_rank(group) if dist else 0
    init = np.atleast_2d(np.asarray(init, dtype=np.float64))
    lo, hi = shard_range(init.shape[0], rank, world)
    block = init[lo:hi]
    if simulate_fn is None:
        def simulate_fn(b, agent0):
            return lib.simulate_philox(model, sol, b, seed, agent0=agent0, want_sims=want_sims, want_moments=True)
    if hi > lo:
        sims, mom = simulate_fn(block, lo)
    else:
        sims, mom = None, np.zeros((3, model.nsimout(), model.nt))
    mom = np.ascontiguousarray(mom, dtype=np.float64)
    all_reduce_moments(mom, group)
    return sims, mom, (lo, hi)


def solve_batch_sharded(lib, model, params: np.ndarray, init: np.ndarray, seed: int, rank: Optional[int] = None,
                        world: Optional[int] = None, solve_sim_fn: Optional[Callable] = None, group=None):
    """Estimation sweep (SURVEY 8(d) S3): the parameter vectors [nvec, nparam] are block-partitioned over the ranks;
    each rank solves its vectors in one batched pass, simulates ``init`` under every vector and contributes the
    per-vector moments [nvec, 3, nsimout, nt]; one all-reduce (sum, other ranks' rows are zero) assembles the table
    on every rank.  ``solve_sim_fn(params_block, first_index) -> moments_block`` replaces the CUDA path in CPU tests."""
    dist = _dist()
    if world is None:
        world = dist.get_world_size(group) if dist else 1
    if rank is None:
        rank = dist.get_rank(group) if dist else 0
    params = np.atleast_2d(np.asarray(params, dtype=np.float64))
    nvec = params.shape[0]
    lo, hi = shard_range(nvec, rank, world)
    nso, nt = model.nsimout(), model.nt
    table = np.zeros((nvec, 3, nso, nt), dtype=np.float64)
    if hi > lo:
        if solve_sim_fn is None:
            def solve_sim_fn(pblock, first):
                sol = lib.solve_batch(model, pblock)
                # the same agents (global ids 0..nsim-1) and the same shocks under every parameter vector, one launch
                return lib.sim_moments(model, sol, init, seed, agent0=0)
        table[lo:hi] = solve_sim_fn(params[lo:hi], lo)
    flat = table.reshape(-1)
    all_reduce_moments(flat, group)
    return table, (lo, hi)


def choice_loglik_sharded(lib, model, sol, obs: np.ndarray, sigma_c: float = 0.0, rank: Optional[int] = None,
                          world: Optional[int] = None, loglik_fn: Optional[Callable] = None, group=None):
    """Choice log-likelihood of the observations ``obs`` [nobs, k] under every parameter vector of ``sol``: each rank
    evaluates its contiguous block of rows and one all-reduce of the [nvec] totals gives every rank the sum.
    Returns (totals [nvec], (lo, hi)).  ``loglik_fn(obs_block) -> totals`` replaces the CUDA call in the CPU tests."""
    dist = _dist()
    if world is None:
        world = dist.get_world_size(group) if dist else 1
    if rank is None:
        rank = dist.get_rank(group) if dist else 0
    obs = np.atleast_2d(np.asarray(obs, dtype=np.float64))
    lo, hi = shard_range(obs.shape[0], rank, world)
    if loglik_fn is None:
        def loglik_fn(block):
            return lib.choice_loglik(model, sol, block, sigma_c=sigma_c)
    tot = np.ascontiguousarray(loglik_fn(obs[lo:hi]), dtype=np.float64)
    all_reduce_moments(tot, group)
    return tot, (lo, hi)


def mixture_loglik_sharded(lib, model, sol, obs: np.ndarray, start: np.ndarray, tvec, weights, sigma_c: float = 0.0,
                           individuals: bool = False, posterior: bool = False, rank: Optional[int] = None,
                           world: Optional[int] = None, fn: Optional[Callable] = None, group=None):
    """Mixture log-likelihood (``ModelLibrary.mixture_loglik``) of the observations ``obs`` grouped by individual with
    offsets ``start`` [nind + 1]: each rank evaluates its contiguous block of individuals [lo, hi), i.e. the rows
    start[lo]..start[hi]-1 with the offsets rebased to 0, and one all-reduce of the [nmix] totals gives every rank the
    sum.  Returns (totals [nmix], per-individual outputs of the rank's block (the tuple after the totals that
    ``mixture_loglik`` returns with ``individuals`` / ``posterior``; empty without them), (lo, hi)).
    ``fn(obs_block, start_block)`` (returning what ``mixture_loglik`` returns) replaces the CUDA call in the CPU tests."""
    dist = _dist()
    if world is None:
        world = dist.get_world_size(group) if dist else 1
    if rank is None:
        rank = dist.get_rank(group) if dist else 0
    obs = np.atleast_2d(np.asarray(obs, dtype=np.float64))
    start = np.asarray(start, dtype=np.int64)
    lo, hi = shard_range(start.size - 1, rank, world)
    r0, r1 = int(start[lo]), int(start[hi])
    if fn is None:
        def fn(block, sblock):
            return lib.mixture_loglik(model, sol, block, sblock, tvec, weights, sigma_c=sigma_c, individuals=individuals,
                                      posterior=posterior)
    res = fn(obs[r0:r1], (start[lo:hi + 1] - r0).astype(np.int32))
    tot, parts = (res[0], tuple(res[1:])) if isinstance(res, tuple) else (res, ())
    tot = np.ascontiguousarray(tot, dtype=np.float64)
    all_reduce_moments(tot, group)
    return tot, parts, (lo, hi)


def mixture_scores_sharded(lib, model, sol, obs: np.ndarray, start: np.ndarray, tvec, weights, mplus, mminus, hinv,
                           sigma_c: float = 0.0, rank: Optional[int] = None, world: Optional[int] = None,
                           fn: Optional[Callable] = None, group=None):
    """Mixture scores (``ModelLibrary.mixture_scores``) over individuals sharded as in ``mixture_loglik_sharded``: each
    rank evaluates its contiguous block of individuals with the offsets rebased to 0, and its totals [nmix], grad
    [npar] and opg [npar * npar] are concatenated and all-reduced once (the OPG is a sum over individuals).  Returns
    (totals [nmix], grad [npar], opg [npar, npar], (lo, hi)).  ``fn(obs_block, start_block)`` (returning (totals,
    grad, opg)) replaces the CUDA call in the CPU tests."""
    dist = _dist()
    if world is None:
        world = dist.get_world_size(group) if dist else 1
    if rank is None:
        rank = dist.get_rank(group) if dist else 0
    obs = np.atleast_2d(np.asarray(obs, dtype=np.float64))
    start = np.asarray(start, dtype=np.int64)
    lo, hi = shard_range(start.size - 1, rank, world)
    r0, r1 = int(start[lo]), int(start[hi])
    if fn is None:
        def fn(block, sblock):
            return lib.mixture_scores(model, sol, block, sblock, tvec, weights, mplus, mminus, hinv, sigma_c=sigma_c)
    tot, grad, opg = fn(obs[r0:r1], (start[lo:hi + 1] - r0).astype(np.int32))
    nmix, npar = np.size(tot), np.size(grad)
    buf = np.ascontiguousarray(np.concatenate([np.ravel(tot), np.ravel(grad), np.ravel(opg)]), dtype=np.float64)
    all_reduce_moments(buf, group)
    return buf[:nmix], buf[nmix:nmix + npar], buf[nmix + npar:].reshape(npar, npar), (lo, hi)
