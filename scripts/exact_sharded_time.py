"""Cost of the exact cross-process sum of trace_sharded(..., exact_sum=True) against the double all-reduce of the float
route, one process per GPU under torchrun (NCCL):

    torchrun --nproc_per_node N scripts/exact_sharded_time.py [--reps 20] [--out profiles/r06_exact_sharded.json]

Each rank traces its shard once in exact mode on a resident bundle; then, on the same bundles, the two reductions are
alternated and timed (host clock between a barrier + device synchronise and the synchronise that ends the reduction):
  - float: dist.all_reduce of the device profile, n_beams x (n_psi + 2) doubles (bench.py's route);
  - exact: the agreement all-reduce, the int64 all-reduce of the accumulator's words and torj_bundle_finalize_exact (the
    code trace_sharded runs: distributed._ExactReduction.reduce_exact).
The words and the profile are restored from a copy before every repeat (untimed), so each repeat reduces the trace's own
values. Workloads: bench.py's 1 M-ray sweep, this rank's block-cyclic shard, with one profile row and with the 1 024
per-beam rows (65.6 MB of words against 8.2 MB of doubles), and the 65 543-ray bench beam sharded contiguously. Also
recorded: the k_trace time of each trace, and whether every rank's converted profile has the same bits. With N = 1 the
all-reduces are no-ops and only the conversion is timed. Rank 0 merges its row into --out under the key N and reads the
card name and power limit in the same run."""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def main():
    import torch
    import torch.distributed as dist

    import torj_jl_b200 as tj
    from torj_jl_b200 import _lib
    from torj_jl_b200.distributed import _ExactReduction, shard_indices
    from torj_jl_b200.solve import device_tensor

    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_exact_sharded.json"))
    args = ap.parse_args()
    rank, local, world = (int(os.environ.get(k, d)) for k, d in (("RANK", 0), ("LOCAL_RANK", 0), ("WORLD_SIZE", 1)))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L, ctx = tj.lib(), _lib.context(local)
    tj.abs_Al_init(bench.N_GL, ctx)
    _lib.check(L.torj_ctx_set_exact_sum(ctx, 1))
    pl = tj.Plasma(*tj.solovev_arrays(bench.GRID, bench.GRID).values())
    psi = np.linspace(0.0, 1.0, bench.N_PSI)
    opt = _lib.default_options(lanes_per_ray=1)  # fixed: a shard and the whole bundle then run the same per-ray arithmetic

    pos, dirs, w = bench.sweep_bundle()
    idx = shard_indices(len(w), rank, world, "block_cyclic", 1025)
    beam = (idx // 1025).astype(np.int32)
    bpos, bdirs, bw = bench.beam_bundle("beam64k", 0)
    bidx = shard_indices(len(bw), rank, world, "contiguous")
    workloads = [("sweep1m shard, 1 profile row", pos[idx], dirs[idx], w[idx], None, 1),
                 ("sweep1m shard, 1024 per-beam rows", pos[idx], dirs[idx], w[idx], beam, 1024),
                 ("beam64k shard", bpos[bidx], bdirs[bidx], bw[bidx], None, 1)]

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        _lib.check(L.torj_ctx_sync(ctx))

    rows = []
    for name, p, d, ww, bid, nb in workloads:
        posT, dirT = np.ascontiguousarray(p.T), np.ascontiguousarray(d.T)
        ww = np.ascontiguousarray(ww, dtype=np.float64)
        fr, md = np.array([95e9]), np.array([1], dtype=np.int32)
        bh = _lib.c_vp()
        _lib.check(L.torj_bundle_create(ctx, len(ww), posT.ctypes.data_as(_lib.c_dp), dirT.ctypes.data_as(_lib.c_dp),
                                        ww.ctypes.data_as(_lib.c_dp), fr.ctypes.data_as(_lib.c_dp),
                                        md.ctypes.data_as(_lib.c_ip), 0, C.byref(bh)))
        try:
            if bid is not None:
                _lib.check(L.torj_bundle_set_beams(bh, nb, np.ascontiguousarray(bid).ctypes.data_as(_lib.c_ip)))
            _lib.check(L.torj_bundle_trace(bh, pl.handle(ctx), C.byref(opt), bench.S_MAX, len(psi),
                                           psi.ctypes.data_as(_lib.c_dp)))
            _lib.check(L.torj_ctx_sync(ctx))
            ms = C.c_double()
            _lib.check(L.torj_ctx_last_trace_ms(ctx, C.byref(ms)))
            wp, nw = _lib.c_vp(), C.c_int64()
            _lib.check(L.torj_bundle_device_exact_words(bh, C.byref(wp), C.byref(nw)))
            words = device_tensor(wp.value, nw.value, "<i8")
            prof = device_tensor(L.torj_bundle_device_profile(bh), nb * (len(psi) + 2), "<f8")
            assert words.device == dev and prof.device == dev
            words0, prof0 = words.clone(), prof.clone()
            t = {"float": [], "exact": []}
            for rep in range(args.reps + 1):  # rep 0 warms both routes up
                for route in ("float", "exact"):
                    words.copy_(words0)
                    prof.copy_(prof0)
                    sync_all()
                    t0 = time.perf_counter()
                    if route == "float":
                        if world > 1:
                            dist.all_reduce(prof)
                        torch.cuda.current_stream().synchronize()
                    else:
                        _ExactReduction(rank, world, dev).reduce_exact(words)
                        torch.cuda.current_stream().synchronize()
                        _lib.check(L.torj_bundle_finalize_exact(bh))
                        _lib.check(L.torj_ctx_sync(ctx))
                    t1 = time.perf_counter()
                    if rep > 0:
                        t[route].append((t1 - t0) * 1e3)
            dep = np.zeros(nb)
            _lib.check(L.torj_bundle_results(bh, None, dep.ctypes.data_as(_lib.c_dp), None, None, None, None, None))
            digest = hashlib.sha256(prof.cpu().numpy().tobytes()).hexdigest()
            digests = [None] * world
            if world > 1:
                dist.all_gather_object(digests, digest)
            else:
                digests = [digest]
            kt = [None] * world
            if world > 1:
                dist.all_gather_object(kt, ms.value)
            else:
                kt = [ms.value]
        finally:
            L.torj_bundle_destroy(bh)
        row = dict(workload=name, n_rays_rank0=len(ww) if rank == 0 else None, n_beams=nb, words_bytes=nw.value * 8,
                   profile_bytes=nb * (len(psi) + 2) * 8, float_ms=float(np.median(t["float"])),
                   exact_ms=float(np.median(t["exact"])), float_all=t["float"], exact_all=t["exact"],
                   ktrace_ms_per_rank=kt, ranks_same_profile_bits=len(set(digests)) == 1)
        row["exact_extra_ms"] = row["exact_ms"] - row["float_ms"]
        rows.append(row)
        if rank == 0:
            print(f"N={world} {name:36s} float {row['float_ms']:8.3f} ms  exact {row['exact_ms']:8.3f} ms  "
                  f"(words {row['words_bytes'] / 1e6:.1f} MB, doubles {row['profile_bytes'] / 1e6:.1f} MB); k_trace max "
                  f"{max(kt):.1f} ms; same bits on every rank: {row['ranks_same_profile_bits']}", flush=True)
    if rank == 0:
        out = {}
        if os.path.exists(args.out):
            with open(args.out) as f:
                out = json.load(f)
        out.setdefault("runs", {})[str(world)] = dict(card=card(), reps=args.reps, gpus=world, rows=rows)
        out["note"] = ("medians of the timed repeats; float and exact routes alternated on the same resident bundles, "
                       "host clock from a barrier + synchronise to the end of the reduction; lanes_per_ray = 1")
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
        print("card:", out["runs"][str(world)]["card"])
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
