"""Multi-GPU plumbing, one process per GPU: rays shard by index (contiguous blocks, or the beams of a scan dealt
round-robin); the only exchange of the path is the weighted sum of reference src/solve.jl:233-240 -> one small all-reduce
of [dP_dV | deposited_power | sum w]. Per-ray outputs are gathered into the launch order of the whole bundle."""
from __future__ import annotations

import numpy as np

from ._lib import exact_bins, profile_vector, split_profile_vector


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


class _ExactReduction:
    """trace_sharded(exact_sum=True): the integer all-reduce of the ranks' exact words, between each rank's trace and its
    conversion (trace_bundle's reduce_exact). Every rank makes the same collective calls in the same order whether it
    traced, had no rays or failed, so a failure on one rank makes every rank raise instead of leaving the others waiting:
      1. agreement, one all-reduce (MIN) of [ok, n_words, -n_words, rank if traced, -empty]: all ranks reached the sum,
         the shortest and longest accumulator, the lowest rank that traced, whether some rank had no rays;
      2. the integer sum (SUM, int64) of the words; a rank without rays adds zeros of the agreed length;
      3. a second agreement [ok] after every rank's conversion and results;
      4. only when some rank had no rays: a broadcast of the converted vector from the lowest rank that traced (a copy of
         bits; an empty rank has no bundle to convert)."""
    _NONE = 1 << 62  # neutral under MIN

    def __init__(self, rank, world, device):
        import torch
        import torch.distributed as dist

        self.torch, self.dist, self.rank = torch, dist, rank
        self.on = world > 1
        self.nccl = self.on and dist.get_backend() == "nccl"
        if self.nccl:
            self.dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        else:
            self.dev = torch.device("cpu")
        self.entered = self.summed = False
        self.agreed = None

    def _min(self, vals):
        t = self.torch.tensor(vals, dtype=self.torch.int64, device=self.dev)
        if self.on:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
        return t.tolist()

    def _agree(self, ok, n_words=None, empty=False):
        N = self._NONE
        ok_all, lo, neg_hi, src, neg_empty = self._min([int(ok), N if n_words is None else n_words,
                                                        N if n_words is None else -n_words, N if empty else self.rank,
                                                        -int(empty)])
        if not ok_all:
            raise RuntimeError("trace_sharded(exact_sum=True): trace_fn failed on a rank before the exact sum (that rank "
                               "raised its own error); no rank summed")
        if lo != -neg_hi:
            raise RuntimeError(f"trace_sharded(exact_sum=True): the ranks' exact accumulators differ in length ({lo} to "
                               f"{-neg_hi} words): every rank must trace with the same psi levels and n_beams")
        self.agreed = (lo, src, neg_empty < 0)

    def _agree_after(self, ok):
        if not self._min([int(ok)])[0]:
            raise RuntimeError("trace_sharded(exact_sum=True): a rank failed after the exact sum, converting it or reading "
                               "its results (that rank raised its own error)")

    def _sum(self, words):
        if not self.on:
            return
        if self.nccl:
            self.dist.all_reduce(words, op=self.dist.ReduceOp.SUM)
        else:
            h = words.cpu()
            self.dist.all_reduce(h, op=self.dist.ReduceOp.SUM)
            words.copy_(h)

    def reduce_exact(self, words):
        self.entered = True
        self._agree(1, int(words.numel()))
        self._sum(words)
        self.summed = True

    def run(self, trace_fn, args, per_ray, n_beams):
        """(local result, this rank's exact vector, the reduced vector) of trace_fn on this rank's rays args"""
        torch = self.torch
        if len(args[2]) == 0:
            self._agree(1, empty=True)
            n_words, src, _ = self.agreed
            self._sum(torch.zeros(n_words, dtype=torch.int64, device=self.dev))
            self._agree_after(1)
            vec = np.zeros(exact_bins(n_words))
            out = torch.zeros(len(vec), dtype=torch.float64, device=self.dev)
            self.dist.broadcast(out, src)
            local = dict(P_final=np.zeros(0), P_deposited_ray=np.zeros(0), n_points=np.zeros(0, dtype=np.int32),
                         status=np.zeros(0, dtype=np.int32))
            return local, vec, out.cpu().numpy()
        try:
            local = trace_fn(*args, **per_ray, reduce_exact=self.reduce_exact)
            if not self.summed:
                raise RuntimeError("trace_sharded(exact_sum=True): trace_fn did not call reduce_exact; pass it on as "
                                   "trace_bundle(..., exact_sum=True, reduce_exact=reduce_exact)")
        except BaseException:
            if not self.entered:
                try:
                    self._agree(0)
                except RuntimeError:
                    pass  # every rank learns of the failure; this one raises its own error
            elif self.summed:
                try:
                    self._agree_after(0)
                except RuntimeError:
                    pass
            raise
        self._agree_after(1)
        vec_sum = profile_vector(local["dP_dV"], local["deposited_power"], local["sum_weights"], n_beams)
        if self.agreed[2]:
            t = torch.from_numpy(vec_sum.copy()).to(self.dev)
            self.dist.broadcast(t, self.agreed[1])
        return local, np.asarray(local["local_vector"]), vec_sum


def trace_sharded(trace_fn, ray_positions, ray_directions, ray_weights, *, n_beams=1, per_ray=None, sharding="contiguous",
                  block=1, device=None, gather_rays=True, exact_sum=False):
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
    rank.
    exact_sum=True: the ranks' exact deposition sums are added as integers, not as finished double profiles, so dP_dV,
    deposited_power and sum_weights are bit-identical for any world size and either sharding, at a fixed lanes_per_ray
    (the automatic width depends on the shard's size), and equal those of one trace_bundle(..., exact_sum=True) of the
    whole bundle. trace_fn then receives one more keyword argument, `reduce_exact`, and must pass it on:
    `lambda p, d, w, reduce_exact: tj.trace_bundle(plasma, p, d, w, ..., exact_sum=True, reduce_exact=reduce_exact)`; its
    result must carry trace_bundle's `sum_weights` and `local_vector`, which is then this rank's own exact vector. A rank
    whose shard is empty (block-cyclic sharding with fewer blocks than ranks) does not call trace_fn. If trace_fn raises on
    any rank, or the ranks' accumulators differ in length, every rank raises; none waits forever in a collective."""
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
    if exact_sum:
        if n == 0:
            raise ValueError("trace_sharded(exact_sum=True) needs at least one ray")
        local, vec, vec_sum = _ExactReduction(rank, world, device).run(
            trace_fn, (pos[idx], dirs[idx], w[idx]), {k: v[idx] for k, v in per_ray.items()}, n_beams)
    else:
        local = trace_fn(pos[idx], dirs[idx], w[idx], **{k: v[idx] for k, v in per_ray.items()})
        if n_beams > 1:
            sw = np.bincount(per_ray["beam_id"][idx], weights=w[idx], minlength=n_beams)
        else:
            sw = np.sum(w[idx])  # numpy's pairwise sum: a bincount would change the last bits
        vec = profile_vector(local["dP_dV"], local["deposited_power"], sw, n_beams)
        t = torch.from_numpy(vec.copy())
        if device is not None:
            t = t.to(device)
        allreduce_profile(t)
        vec_sum = t.cpu().numpy()
    dP_dV, deposited_power, sum_weights = split_profile_vector(vec_sum, n_beams)
    out = dict(dP_dV=dP_dV, deposited_power=deposited_power, sum_weights=sum_weights, local=local, idx=idx, local_vector=vec)
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
