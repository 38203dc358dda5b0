"""Multi-GPU sampling: one process per GPU, pocket graphs partitioned across ranks.

The path shards naturally (SURVEY.md section 8e): complexes are independent, weights (145 MB bf16) and the
[T,3,20,20] transition tables are replicated, and the sampling noise is keyed by the GLOBAL graph id, so a
rank only needs its slice of the batch -- there is NO collective on the data path.  torch.distributed is
used for exactly two things: gathering the decoded result strings (a few bytes per graph) and the
max-over-ranks timing reduction of bench.py.
"""
from __future__ import annotations

from typing import Callable, Dict, Tuple

import torch


def shard_bounds(n: int, world: int, rank: int) -> Tuple[int, int]:
    """Contiguous block partition of n graphs; the first n % world ranks hold one extra graph."""
    if not (0 <= rank < world):
        raise ValueError("rank out of range")
    base, extra = divmod(n, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def shard_batch(batch: Dict, world: int, rank: int):
    """Slices every per-graph entry of a reference-style batch dict (sample.py:183-190, incl. the nested
    structure_ids lists).  Returns (sub_batch, graph_id0) -- graph_id0 keys the counter-based RNG."""
    n = batch["ligand_seq"].shape[0]
    lo, hi = shard_bounds(n, world, rank)

    def cut(v):
        if torch.is_tensor(v):
            return v[lo:hi] if v.ndim > 0 and v.shape[0] == n else v
        if isinstance(v, dict):
            return {k: cut(x) for k, x in v.items()}
        if isinstance(v, (list, tuple)) and len(v) == n:
            return v[lo:hi]
        return v

    return {k: cut(v) for k, v in batch.items()}, lo


def max_over_ranks(value: float, device=None, group=None) -> float:
    """Timing reduction: every multi-GPU number is the slowest rank's."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return float(value)
    t = torch.tensor([float(value)], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    return float(t.item())


def denoise_sharded(batch, model, noise_schedule, transition, diverse, denoise_fn: Callable = None, group=None, **kw):
    """Strong-scaling front end with the return contract of reference denoise() (sample.py:181-229): every rank
    samples its block of graphs on its own GPU, then the decoded (ids, true, pred, recovery) lists are
    all-gathered in rank order, so each rank returns exactly what a single-GPU call on the whole batch returns:
    the start state x_T of the WHOLE batch is drawn once (rank 0's `generate_discrete_noise`, broadcast as class indices --
    a one-off B*L-byte exchange before the loop, not a data-path collective) unless the caller passes `x_T`, and the Philox
    noise is keyed by global graph ids taken as ONE block from the process-wide stream on every rank.
    `num_samples=K > 1` (K sequences per pocket): the ranks share out the POCKETS -- rank r samples pockets [lo, hi), which are graphs
    [lo*K, hi*K) of the one-GPU call: its slice of x_T and noise_E_steps and its graph ids start there."""
    import torch.distributed as dist
    from . import _cabi
    from .sample import check_num_samples
    if denoise_fn is None:
        from .sample import denoise as denoise_fn
    K = check_num_samples(kw.get("num_samples", 1))
    if not (dist.is_available() and dist.is_initialized()):
        return denoise_fn(batch, model, noise_schedule, transition, diverse, **kw)
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    n, L, C = batch["ligand_seq"].shape
    sub, lo = shard_batch(batch, world, rank)
    hi = lo + sub["ligand_seq"].shape[0]
    x_T = kw.pop("x_T", None)
    if x_T is None:
        box = [torch.randint(0, C, (n * K, L)).to(torch.uint8) if rank == 0 else None]
        dist.broadcast_object_list(box, src=0, group=group)
        x_T = torch.nn.functional.one_hot(box[0].long(), C).float()
    kw["x_T"] = x_T[lo * K:hi * K]
    if K > 1 and kw.get("noise_E_steps") is not None:
        kw["noise_E_steps"] = kw["noise_E_steps"][:, lo * K * L:hi * K * L]
    base = kw.pop("graph_id0", None)
    gid0 = lo * K + (_cabi.GRAPH_IDS.take(n * K) if base is None else base)
    part = denoise_fn(sub, model, noise_schedule, transition, diverse, graph_id0=gid0, **kw) if sub["ligand_seq"].shape[0] else ([], [], [], [])
    parts = [None] * world
    dist.all_gather_object(parts, part, group=group)
    out = ([], [], [], [])
    for p in parts:
        for dst, src in zip(out, p):
            dst.extend(src)
    return out


def p_sample_loop_sharded(model, ligand_mask, ligand_angle_noise, receptor_seq, receptor_mask, receptor_angle, total_timesteps, betas,
                          sample_fn: Callable = None, group=None, **kw):
    """structure_model p_sample_loop (reference structure_model/sample.py:104-144) over the ranks of `group`: every rank samples
    its contiguous block of complexes on its own GPU (noise keyed by the global graph id), then the CPU [T, b_r, L, F] histories
    are all-gathered and concatenated along the batch axis in rank order -- each rank returns what one GPU returns for the
    whole batch.  No collective on the data path; the only exchange is the result tensor the reference returns anyway."""
    import torch.distributed as dist
    if sample_fn is None:
        from .structure_model import p_sample_loop as sample_fn
    if not (dist.is_available() and dist.is_initialized()):
        return sample_fn(model, ligand_mask, ligand_angle_noise, receptor_seq, receptor_mask, receptor_angle, total_timesteps, betas, **kw)
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    n = ligand_angle_noise.shape[0]
    lo, hi = shard_bounds(n, world, rank)
    noise_steps = kw.pop("noise_steps", None)
    if noise_steps is not None:
        kw["noise_steps"] = noise_steps[:, lo:hi]
    base = kw.pop("graph_id0", None)
    if base is None:
        from . import _cabi
        base = _cabi.GRAPH_IDS.take(n)
    gid0 = lo + base
    part = None
    if hi > lo:
        part = sample_fn(model, ligand_mask[lo:hi], ligand_angle_noise[lo:hi], receptor_seq[lo:hi], receptor_mask[lo:hi],
                         receptor_angle[lo:hi], total_timesteps, betas, graph_id0=gid0, **kw)
    parts = [None] * world
    dist.all_gather_object(parts, part, group=group)
    return torch.cat([p for p in parts if p is not None], dim=1)
