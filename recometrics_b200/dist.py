"""Multi-GPU evaluation: one process per GPU, users block-partitioned, item factors replicated.

The path has no exchange step (every user is an independent unit, SURVEY 8(e)): each rank evaluates
its contiguous block of users against its own full copy of ``B`` and the per-user metric rows are
gathered to the destination rank.  ``torch.distributed`` (NCCL on GPUs, gloo in the CPU tests) is
plumbing for that gather only.
"""
import numpy as np

from .frontend import calc_reco_metrics_ex, item_popularity

__all__ = ["shard_bounds", "gather_metric_rows", "reduce_exposure", "reduce_popularity", "calc_reco_metrics_sharded"]


def shard_bounds(m, world_size, rank):
    """Contiguous user block [begin, end) of `rank` (work per eligible user is ~2*p*n regardless of
    the user, so equal counts balance)."""
    m, world_size, rank = int(m), int(world_size), int(rank)
    if not (0 <= rank < world_size):
        raise ValueError("rank outside [0, world_size)")
    return (m * rank) // world_size, (m * (rank + 1)) // world_size


def gather_metric_rows(local, m, group=None, dst=0):
    """Gather per-user rows to rank `dst`.

    `local` maps metric name -> array holding THIS rank's rows only (shape [rows] or [rows, K]), for
    the block given by :func:`shard_bounds`.  Returns the assembled dict (full m rows) on `dst`,
    None elsewhere.  Blocks are padded to a common height so one collective moves each metric."""
    import torch
    import torch.distributed as dist

    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    backend = dist.get_backend(group)
    dev = torch.device("cuda", torch.cuda.current_device()) if backend == "nccl" else torch.device("cpu")
    bounds = [shard_bounds(m, world, r) for r in range(world)]
    hmax = max(e - b for b, e in bounds)
    out = {} if rank == dst else None
    for name in sorted(local.keys()):
        arr = np.ascontiguousarray(local[name])
        b, e = bounds[rank]
        if arr.shape[0] != e - b:
            raise ValueError("rank %d: metric %s has %d rows, its block has %d" % (rank, name, arr.shape[0], e - b))
        tail = arr.shape[1:]
        pad = np.full((hmax,) + tail, np.nan, dtype=arr.dtype)
        pad[: e - b] = arr
        t = torch.from_numpy(pad).to(dev)
        if backend == "nccl":
            bufs = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(bufs, t, group=group)
        else:
            bufs = [torch.empty_like(t) for _ in range(world)] if rank == dst else None
            dist.gather(t, bufs, dst=dst, group=group)
        if rank == dst:
            full = np.empty((m,) + tail, dtype=arr.dtype)
            for r, (rb, re_) in enumerate(bounds):
                full[rb:re_] = bufs[r][: re_ - rb].cpu().numpy()
            out[name] = full
    return out


def reduce_exposure(local_counts, group=None, dst=0, local_users=0):
    """Sum the ranks' item counts (``EvalResult.exposure`` of each rank's block; int64 [n], the same n everywhere) to rank
    `dst`.  Counts are additive, so the sum is exactly what one call over all users counts; the catalogue statistics are
    computed from it by the library's own host function.  `local_users`: this rank's counted users
    (``EvalResult.catalogue["users"]``).  Returns ``(counts, catalogue)`` on `dst`, None elsewhere."""
    import torch
    import torch.distributed as dist

    from . import _capi

    rank = dist.get_rank(group)
    dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend(group) == "nccl" else torch.device("cpu")
    counts = np.ascontiguousarray(local_counts, dtype=np.int64)
    t = torch.from_numpy(np.append(counts, np.int64(local_users))).to(dev)       # one collective: counts, then users
    dist.reduce(t, dst=dst, op=dist.ReduceOp.SUM, group=group)
    if rank != dst:
        return None
    total = t.cpu().numpy()
    return total[:-1].copy(), _capi.exposure_stats(total[:-1], users=int(total[-1]))


def reduce_popularity(local_counts, group=None):
    """Sum the ranks' item popularity counts (:func:`recometrics_b200.item_popularity` of each rank's block of ``X_train``
    rows; int64 [n], the same n everywhere) on every rank: one ``all_reduce``.  The sum is the popularity over all users,
    exactly, so every rank's Novelty@K / AvgPop@K rows are those of one call over all users.  Returns numpy int64 [n]."""
    import torch
    import torch.distributed as dist

    dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend(group) == "nccl" else torch.device("cpu")
    t = torch.from_numpy(np.ascontiguousarray(local_counts, dtype=np.int64).copy()).to(dev)
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t.cpu().numpy()


def calc_reco_metrics_sharded(X_train, X_test, A, B, k=5, group=None, dst=0, return_exposure=False, **kwargs):
    """Evaluate with every rank of `group` taking its block of users on its current CUDA device.

    Every rank passes the same (full) inputs; only the block's rows of A and of the CSR matrices are
    copied to that rank's GPU, B entirely.  Returns the reference-style dict on `dst` (None elsewhere).
    ``return_exposure``: returns ``(dict, item_counts, catalogue)`` on `dst` instead, the ranks' item exposure summed by
    :func:`reduce_exposure`.  ``novelty`` / ``avg_popularity`` without ``item_popularity``: every rank counts its block's
    ``X_train`` rows and :func:`reduce_popularity` adds them up, so the rows equal those of one call over all users.
    ``unexpectedness`` / ``serendipity`` (see :func:`calc_reco_metrics_ex`) pass through ``kwargs`` as they are: a user's
    values read only that user's own ``X_train`` and ``X_test`` rows, so the ranks' rows need no reduction step."""
    import torch.distributed as dist

    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    m = X_test.shape[0]
    b, e = shard_bounds(m, world, rank)
    if (kwargs.get("novelty") or kwargs.get("avg_popularity")) and kwargs.get("item_popularity") is None:
        local = item_popularity(X_train, user_range=(b, e)) if X_train is not None else np.zeros(X_test.shape[1], dtype=np.int64)
        kwargs["item_popularity"] = reduce_popularity(local, group=group)
    res = calc_reco_metrics_ex(X_train, X_test, A, B, k=k, user_range=(b, e), return_exposure=return_exposure, **kwargs)
    K = res.metrics["K"]
    local = {name: v[b:e] for name, v in res.metrics.items() if name != "K"}
    full = gather_metric_rows(local, m, group=group, dst=dst)
    if full is not None:
        full["K"] = K
    if not return_exposure:
        return full
    expo = reduce_exposure(res.exposure, group=group, dst=dst, local_users=res.catalogue["users"])
    return None if expo is None else (full,) + expo
