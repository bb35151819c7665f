"""trace_sharded with several beams and per-ray arrays on CPU: two and three gloo ranks run the product's sharding,
all-reduce of the [n_beams][n_psi | deposited | sum w] vector and per-ray assembly around a closed-form multi-beam fake
backend (no GPU, no oracle). The assembled result must equal the backend applied to the unsharded bundle, for contiguous
and block-cyclic sharding, ragged beam sizes included; a single-beam call must keep its keys and local vector."""
import os
import sys

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_PSI = 29
N_BEAMS = 5
SIZES = (23, 7, 31, 1, 19)  # ragged beams, one of a single ray


def fake_trace(pos, dirs, w, beam_id, f):
    """Every per-ray output is a function of the ray (its frequency included) alone; each beam's profile row is the
    weighted sum over its rays, as the device profile is."""
    key = pos[:, 0] * 3.0 + pos[:, 2] - dirs[:, 1] + 1e-11 * f
    P_final = np.exp(-np.abs(key))
    shell = (np.floor(np.abs(key) * 7.0).astype(int)) % N_PSI
    prof = np.zeros((N_BEAMS, N_PSI))
    np.add.at(prof, (beam_id, shell), w * (1.0 - P_final))
    dep = np.zeros(N_BEAMS)
    np.add.at(dep, beam_id, w * (1.0 - P_final))
    return dict(dP_dV=prof, deposited_power=dep, P_final=P_final, n_points=(2 + np.floor(100 * np.abs(key))).astype(np.int32),
                status=(np.abs(key) > 5.0).astype(np.int32) * 2)


def single_trace(pos, dirs, w):
    r = fake_trace(pos, dirs, w, np.zeros(len(w), dtype=np.int32), np.full(len(w), 95e9))
    return dict(r, dP_dV=r["dP_dV"][0], deposited_power=float(r["deposited_power"][0]))


def bundle():
    n = sum(SIZES)
    k = np.arange(n, dtype=np.float64)
    pos = np.stack([np.sin(k), np.cos(0.3 * k), 0.01 * k], axis=1)
    dirs = np.stack([np.cos(k), np.sin(0.7 * k), np.ones(n)], axis=1)
    w = (1.0 + (k % 5)) / np.sum(1.0 + (k % 5))
    beam_id = np.repeat(np.arange(N_BEAMS, dtype=np.int32), SIZES)
    f = 90e9 + 1e9 * (k % 7)
    return pos, dirs, w, beam_id, f


CASES = (("contig", dict(sharding="contiguous")), ("cyclic", dict(sharding="block_cyclic", block=7)),
         ("cyclic1", dict(sharding="block_cyclic", block=1)))
KEYS = ("dP_dV", "deposited_power", "sum_weights", "P_final", "n_points", "status")


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from torj_jl_b200.distributed import trace_sharded

    pos, dirs, w, beam_id, f = bundle()
    res = {}
    for name, kw in CASES:
        r = trace_sharded(fake_trace, pos, dirs, w, n_beams=N_BEAMS, per_ray=dict(beam_id=beam_id, f=f), **kw)
        assert len(r["idx"]) == len(r["local"]["P_final"])
        for k in KEYS:
            res[f"{name}_{k}"] = np.asarray(r[k])
        res[f"{name}_idx_{rank}"] = r["idx"]
    r = trace_sharded(single_trace, pos, dirs, w, sharding="block_cyclic", block=7)
    assert set(r) == {"dP_dV", "deposited_power", "sum_weights", "local", "idx", "local_vector", "P_final", "n_points",
                      "status"}
    assert isinstance(r["deposited_power"], float) and isinstance(r["sum_weights"], float)
    idx = r["idx"]
    mine = single_trace(pos[idx], dirs[idx], w[idx])
    want = np.concatenate([np.ravel(mine["dP_dV"]), [float(mine["deposited_power"]), float(np.sum(w[idx]))]])
    assert np.array_equal(r["local_vector"], want)
    res["single_dP_dV"] = r["dP_dV"]
    np.savez(os.path.join(out_dir, f"rank{rank}.npz"), **res)
    dist.barrier()
    dist.destroy_process_group()


def _check(tmp_path, world):
    port = 31500 + (os.getpid() % 2000) + world
    mp.spawn(_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    ranks = [np.load(tmp_path / f"rank{r}.npz") for r in range(world)]
    pos, dirs, w, beam_id, f = bundle()
    full = fake_trace(pos, dirs, w, beam_id, f)
    sw = np.array([w[beam_id == q].sum() for q in range(N_BEAMS)])
    for name, _ in CASES:
        owned = np.sort(np.concatenate([ranks[r][f"{name}_idx_{r}"] for r in range(world)]))
        assert np.array_equal(owned, np.arange(len(w)))                 # the shards partition the bundle
        for g in ranks:                                                 # every rank holds the same assembled result
            assert g[f"{name}_dP_dV"].shape == (N_BEAMS, N_PSI)
            assert np.abs(g[f"{name}_dP_dV"] - full["dP_dV"]).max() <= 1e-13
            assert np.abs(g[f"{name}_deposited_power"] - full["deposited_power"]).max() <= 1e-13
            assert np.abs(g[f"{name}_sum_weights"] - sw).max() <= 1e-13
            for k in ("P_final", "n_points", "status"):
                assert np.array_equal(g[f"{name}_{k}"], full[k]), (name, k)
    single = single_trace(pos, dirs, w)
    for g in ranks:
        assert np.abs(g["single_dP_dV"] - single["dP_dV"]).max() <= 1e-13


def test_two_rank_multibeam_sharded_trace_equals_unsharded(tmp_path):
    _check(tmp_path, 2)


def test_three_rank_multibeam_sharded_trace_equals_unsharded(tmp_path):
    _check(tmp_path, 3)


def test_multibeam_needs_beam_id():
    sys.path.insert(0, ROOT)
    from torj_jl_b200.distributed import trace_sharded

    pos, dirs, w, beam_id, f = bundle()
    with pytest.raises(ValueError, match="beam_id"):
        trace_sharded(fake_trace, pos, dirs, w, n_beams=N_BEAMS, per_ray=dict(f=f))
    with pytest.raises(ValueError, match=r"\[0, 5\)"):
        trace_sharded(fake_trace, pos, dirs, w, n_beams=N_BEAMS, per_ray=dict(beam_id=beam_id + 1, f=f))
    with pytest.raises(ValueError, match="one entry per ray"):
        trace_sharded(fake_trace, pos, dirs, w, n_beams=N_BEAMS, per_ray=dict(beam_id=beam_id, f=f[:-1]))
