"""Multi-GPU partitioning of the hot path (one process per GPU).

The unit of work is an independent chain: chains are sharded across ranks with
NO data-path collective.  torch.distributed is used only for (a) the timing
barrier / max-over-ranks of bench.py and (b) gathering the tracked scalars and
samples onto rank 0 at the end of a run.  Philox streams are keyed on the GLOBAL
chain index so results do not depend on how chains are sharded.
"""
import numpy as np


def chain_shard(nchains_total, world_size, rank):
    """(first global chain index, number of chains) of `rank`; remainders go to the low ranks."""
    if not (0 <= rank < world_size):
        raise ValueError("rank out of range")
    base, rem = divmod(int(nchains_total), int(world_size))
    count = base + (1 if rank < rem else 0)
    start = rank * base + min(rank, rem)
    return start, count


def philox_stream0(nchains_total, world_size, rank):
    """first Philox stream id of this rank (stream id == global chain index)"""
    return chain_shard(nchains_total, world_size, rank)[0]


def gather_chains(local, nchains_total, group=None):
    """Gather per-chain arrays [nlocal, ...] from every rank into [nchains_total, ...] on rank 0
    (None elsewhere), ordered by global chain index.  Works on any backend (gloo / nccl)."""
    import torch
    import torch.distributed as dist

    if not dist.is_available() or not dist.is_initialized():
        return np.asarray(local)
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    t = torch.as_tensor(np.ascontiguousarray(local))
    if dist.get_backend(group) == "nccl":
        t = t.cuda()
    counts = [chain_shard(nchains_total, world, r)[1] for r in range(world)]
    maxc = max(counts)
    pad = torch.zeros((maxc,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    pad[: t.shape[0]] = t
    bufs = [torch.empty_like(pad) for _ in range(world)] if rank == 0 else None
    dist.gather(pad, bufs, dst=0, group=group)
    if rank != 0:
        return None
    return np.concatenate([b[:c].cpu().numpy() for b, c in zip(bufs, counts)], axis=0)


def max_over_ranks(value, group=None):
    """max of a python float over ranks (device timing of bench.py)"""
    import torch
    import torch.distributed as dist

    if not dist.is_available() or not dist.is_initialized():
        return float(value)
    t = torch.tensor([float(value)], dtype=torch.float64)
    if dist.get_backend(group) == "nccl":
        t = t.cuda()
    dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    return float(t.item())


def gather_summary(partials, nchains_total, group=None, chain_arrays=True):
    """Streaming posterior summaries of chains sharded over ranks: `partials` = this rank's
    `sampler.summary_partials()` ({target: partial record dict}); rank 0 receives every rank's records and returns
    {target: diagnostics.Summary} over all `nchains_total` logical chains (per-chain arrays in global chain order, as
    `gather_chains`; `chain_arrays=False` leaves them out and sends only the records), None elsewhere."""
    from .diagnostics import finalize

    def strip(p):
        return p if chain_arrays else {k: v for k, v in p.items() if k not in ("chain_mean", "chain_var")}

    mine = {k: strip(p) for k, p in partials.items()}
    import torch.distributed as dist

    if not dist.is_available() or not dist.is_initialized():
        got = [mine]
    else:
        rank = dist.get_rank(group)
        got = [None] * dist.get_world_size(group) if rank == 0 else None
        dist.gather_object(mine, got, dst=0, group=group)
        if rank != 0:
            return None
    out = {}
    for k in got[0]:
        parts = [g[k] for g in got]
        total = sum(int(p["nchains"]) for p in parts)
        if total != int(nchains_total):
            raise ValueError(f"gather_summary: the ranks hold {total} chains of {k}, expected {nchains_total}")
        out[k] = finalize(parts, chain_arrays=chain_arrays)
    return out
