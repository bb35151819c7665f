"""Multi-GPU plumbing, one process per GPU: rays shard by index (contiguous blocks, or the beams of a scan dealt
round-robin); the only exchange of the path is the weighted sum of reference src/solve.jl:233-240 -> one small all-reduce
of [dP_dV | deposited_power | sum w]. Per-ray outputs are gathered into the launch order of the whole bundle."""
from __future__ import annotations

import numpy as np


def shard_range(n_rays: int, rank: int, world_size: int) -> tuple[int, int]:
    """Contiguous block [lo, hi) of rank; sizes differ by at most one."""
    base, rem = divmod(int(n_rays), int(world_size))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def shard_block_cyclic(n_rays: int, block: int, rank: int, world_size: int):
    """Ray indices of rank when blocks of `block` consecutive rays (one beam of a scan) are dealt round-robin:
    block b goes to rank b % world_size. Contiguous sharding of an angle scan gives every rank a different range of
    launcher angles, i.e. rays of different lengths (measured: 6.2x on 8 GPUs instead of the ideal 8); dealing the
    beams out evens the work. Returns a sorted int64 array; the ranks' arrays partition range(n_rays)."""
    n_blocks = -(-int(n_rays) // int(block))
    mine = np.arange(rank, n_blocks, world_size, dtype=np.int64)
    idx = (mine[:, None] * block + np.arange(block, dtype=np.int64)[None, :]).ravel()
    return idx[idx < n_rays]


def shard_indices(n_rays: int, rank: int, world_size: int, sharding: str = "contiguous", block: int = 1):
    """Global ray indices of `rank` (sorted int64): "contiguous" blocks or "block_cyclic" (see shard_block_cyclic)."""
    if sharding == "contiguous":
        lo, hi = shard_range(n_rays, rank, world_size)
        return np.arange(lo, hi, dtype=np.int64)
    if sharding == "block_cyclic":
        return shard_block_cyclic(n_rays, block, rank, world_size)
    raise ValueError("sharding must be 'contiguous' or 'block_cyclic'")


def allreduce_profile(t):
    """In-place sum over ranks of a tensor [n_psi+2] (NCCL on GPUs, gloo in CPU tests); no-op when not initialised."""
    import torch.distributed as dist

    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return t


def _world():
    import torch.distributed as dist

    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def trace_sharded(trace_fn, ray_positions, ray_directions, ray_weights, *, n_beams=1, per_ray=None, sharding="contiguous",
                  block=1, device=None, gather_rays=True):
    """make_beam's parallel region and reduction (reference src/solve.jl:219-240) over the ranks of the initialised process
    group. `trace_fn(pos, dirs, w)` traces this rank's rays — on a GPU box `lambda p, d, w: tj.trace_bundle(plasma, p, d, w,
    ...)` — and returns a dict with dP_dV [n_psi], deposited_power, P_final / n_points / status [n_local].
    per_ray: a dict of further per-ray arrays over the whole bundle (beam_id, f, mode, ...); each is cut to this rank's rays
    and passed to trace_fn as a keyword argument of that name.
    n_beams > 1: trace_fn returns dP_dV [n_beams, n_psi] and deposited_power [n_beams], per_ray holds "beam_id", and the
    reduced vector is the device profile layout [n_beams][n_psi | deposited | sum w] with the weights summed per beam. A
    plasma set then runs as `lambda p, d, w, beam_id: tj.trace_bundle(plasmas, p, d, w, ..., beam_id=beam_id, n_beams=K,
    beam_plasma=bp)`.
    Returns the all-reduced dP_dV, deposited_power and sum of weights (per beam when n_beams > 1), this rank's `local`
    result and `idx`, and (when gather_rays) the per-ray outputs of the WHOLE bundle in launch order, identical on every
    rank."""
    import torch
    import torch.distributed as dist

    rank, world = _world()
    pos, dirs, w = np.asarray(ray_positions), np.asarray(ray_directions), np.asarray(ray_weights)
    n = len(w)
    per_ray = {k: np.asarray(v) for k, v in (per_ray or {}).items()}
    for k, v in per_ray.items():
        if len(v) != n:
            raise ValueError(f"per_ray[{k!r}] must have one entry per ray ({n}), got {len(v)}")
    n_beams = int(n_beams)
    if n_beams > 1:
        bid = per_ray.get("beam_id")
        if bid is None:
            raise ValueError("n_beams > 1 needs per_ray['beam_id'] (the beam of every ray)")
        if n and (bid.min() < 0 or bid.max() >= n_beams):
            raise ValueError(f"beam_id must lie in [0, {n_beams})")
    idx = shard_indices(n, rank, world, sharding, block)
    local = trace_fn(pos[idx], dirs[idx], w[idx], **{k: v[idx] for k, v in per_ray.items()})
    if n_beams > 1:
        sw = np.bincount(per_ray["beam_id"][idx], weights=w[idx], minlength=n_beams)
        vec = np.concatenate([np.reshape(local["dP_dV"], (n_beams, -1)), np.reshape(local["deposited_power"], (n_beams, 1)),
                              sw[:, None]], axis=1).ravel()
    else:
        vec = np.concatenate([np.ravel(local["dP_dV"]), [float(local["deposited_power"]), float(np.sum(w[idx]))]])
    t = torch.from_numpy(vec.copy())
    if device is not None:
        t = t.to(device)
    allreduce_profile(t)
    vec_sum = t.cpu().numpy()
    if n_beams > 1:
        rows = vec_sum.reshape(n_beams, -1)
        out = dict(dP_dV=rows[:, :-2].copy(), deposited_power=rows[:, -2].copy(), sum_weights=rows[:, -1].copy(), local=local,
                   idx=idx, local_vector=vec)
    else:
        out = dict(dP_dV=vec_sum[:-2], deposited_power=float(vec_sum[-2]), sum_weights=float(vec_sum[-1]), local=local, idx=idx,
                   local_vector=vec)
    if gather_rays:
        mine = {k: np.asarray(local[k]) for k in ("P_final", "n_points", "status") if k in local}
        parts = [None] * world
        if world > 1:
            dist.all_gather_object(parts, (idx, mine))
        else:
            parts = [(idx, mine)]
        for k in mine:
            full = np.zeros(n, dtype=mine[k].dtype)
            for pidx, pm in parts:
                full[pidx] = pm[k]
            out[k] = full
    return out
