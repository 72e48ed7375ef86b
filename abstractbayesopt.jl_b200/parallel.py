"""Multi-GPU host logic: one process per GPU.  Candidates (and NLML restarts) are sharded by
contiguous index range with no data-path collective; the posterior is broadcast once per BO
iteration with NCCL (abo_gp_sync) and the per-rank top-k lists are merged with the
(value desc, index asc, NaN first) order of sortperm(scores; rev=true) (acq_utils.jl:51) so the
selected candidates do not depend on the number of ranks (SURVEY §8e)."""
from __future__ import annotations

import numpy as np


def shard_range(m: int, rank: int, world: int):
    """Rank r owns candidates [r*m/G, (r+1)*m/G)."""
    return (rank * m) // world, ((rank + 1) * m) // world


def _ordkey(v: np.ndarray) -> np.ndarray:
    """Julia isless order on Float64 as uint64 keys (NaN largest, -0.0 < 0.0)."""
    v = np.ascontiguousarray(v, dtype=np.float64)
    u = v.view(np.uint64)
    neg = (u >> np.uint64(63)).astype(bool)
    key = np.where(neg, ~u, u | np.uint64(1 << 63))
    return np.where(np.isnan(v), np.uint64(0xFFFFFFFFFFFFFFFF), key)


def merge_topk(idx_lists, val_lists, k: int):
    """Merge per-rank (global index, value) lists into the global stable descending top-k."""
    idx = np.concatenate([np.asarray(a, dtype=np.int64) for a in idx_lists]) if idx_lists else np.empty(0, np.int64)
    val = np.concatenate([np.asarray(a, dtype=np.float64) for a in val_lists]) if val_lists else np.empty(0)
    if idx.size == 0:
        return idx, val
    key = _ordkey(val)
    order = np.lexsort((idx, np.iinfo(np.uint64).max - key))
    order = order[:min(k, order.size)]
    return idx[order], val[order]


def sharded_topk(acq, surrogate, candidates, k: int, group=None):
    """Every rank holds the full candidate array (or can index its shard), evaluates its shard
    with the fused sweep, and all ranks end up with the same global top-k (global indices)."""
    import torch.distributed as dist
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    lo, hi = shard_range(len(candidates), rank, world)
    ctx = getattr(surrogate, "ctx", None)
    shard_topk = getattr(acq, "shard_topk", None)
    if shard_topk is not None:
        # an acquisition whose parameters depend on the whole set (MaxValueEntropySearch: the sampled minimum values)
        # exchanges what it needs through `gather` before it sweeps its shard
        _, ti, tv = shard_topk(surrogate, candidates[lo:hi], k, lambda v: _allgather(v, world, group, ctx))
    else:
        _, ti, tv = acq.topk(surrogate, candidates[lo:hi], k)
    mine = (np.asarray(ti, dtype=np.int64) + lo, np.asarray(tv))
    if world == 1:
        return merge_topk([mine[0]], [mine[1]], k)
    if _nccl_spans(ctx, world):
        # abo_topk_allgather: one NCCL all-gather of the (count, index, value) records + the same
        # (value desc, index asc, NaN first) merge inside the library
        return ctx.topk_allgather(k, mine[0], mine[1])
    gathered = [None] * world
    dist.all_gather_object(gathered, mine, group=group)
    return merge_topk([g[0] for g in gathered], [g[1] for g in gathered], k)


def _allgather(values, world: int, group=None, ctx=None):
    """Every rank's equally long float64 array, in rank order: NCCL through `ctx` when it spans the job, else the
    torch.distributed group."""
    values = np.ascontiguousarray(values, dtype=np.float64)
    if world == 1:
        return [values]
    if _nccl_spans(ctx, world):
        return list(ctx.allgather_f64(values, world))
    import torch.distributed as dist
    gathered = [None] * world
    dist.all_gather_object(gathered, values, group=group)
    return [np.asarray(g, dtype=np.float64) for g in gathered]


def _nccl_spans(ctx, world: int) -> bool:
    """True when `ctx` carries an NCCL communicator over exactly `world` ranks (init_nccl_context was called
    on it).  Otherwise the torch.distributed group does the exchange (gloo in the CPU tests)."""
    if ctx is None or not hasattr(ctx, "ranks"):
        return False
    try:
        return ctx.ranks()[1] == world
    except Exception:
        return False


def sharded_restarts(evaluate, logparams, group=None, nccl_ctx=None):
    """NLML restarts sharded R/G per rank (SURVEY 8e): rank r evaluates rows [r*R/G, (r+1)*R/G) of
    `logparams` with `evaluate(rows) -> (val[R_r], grad[R_r, 2], info[R_r])` (abo_nlml_batch on its GPU) and
    every rank ends up with the full (val, grad, info) in restart order.  The exchange is one
    all-gather of 4 doubles per restart: NCCL through the context when `nccl_ctx` has a
    communicator, else the torch.distributed group (gloo in the CPU tests)."""
    import torch.distributed as dist
    theta = np.asarray(logparams, dtype=np.float64).reshape(-1, 2)
    R = theta.shape[0]
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    lo, hi = shard_range(R, rank, world)
    val, grad, info = evaluate(theta[lo:hi])
    if world == 1:
        return np.asarray(val), np.asarray(grad), np.asarray(info)
    per = -(-R // world)                                   # equal-sized blocks, padded
    block = np.zeros((per, 4))
    block[:hi - lo, 0] = val; block[:hi - lo, 1:3] = np.asarray(grad).reshape(-1, 2); block[:hi - lo, 3] = info
    if _nccl_spans(nccl_ctx, world):
        allb = nccl_ctx.allgather_f64(block, world).reshape(world, per, 4)
    else:
        gathered = [None] * world
        dist.all_gather_object(gathered, block, group=group)
        allb = np.stack(gathered)
    out = np.concatenate([allb[r, :shard_range(R, r, world)[1] - shard_range(R, r, world)[0]] for r in range(world)])
    return out[:, 0].copy(), out[:, 1:3].copy(), out[:, 3].astype(np.int32)


def sharded_nlml_batch(model, logparams, xs, ys, group=None, use_nccl=True):
    """nlml + gradient for all restarts with the restarts split across the ranks' GPUs."""
    from .surrogates import nlml_batch
    from ._lib import default_context
    ctx = model.ctx or default_context()
    return sharded_restarts(lambda th: nlml_batch(model, th, xs, ys), logparams, group=group,
                            nccl_ctx=ctx if use_nccl else None)


def init_nccl_context(ctx, group=None):
    """Give `ctx` an NCCL rank matching the torch.distributed group: rank 0 creates the NCCL
    unique id, it is broadcast through the existing process group (any backend)."""
    import torch.distributed as dist
    from ._lib import nccl_unique_id
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    box = [nccl_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(box, src=0, group=group)
    ctx.init_rank(rank, world, box[0])


def sync_posterior(model, root: int = 0):
    """Broadcast the conditioned surrogate (L, L^-1, X, alpha, hyper-parameters) from `root`
    to every rank over NCCL / NVLink.  Non-root models must already hold a handle of the same
    (kernel, d, p) — e.g. created by update() on any data, or by `empty_like`."""
    model.gpx.sync(root)
    return model
