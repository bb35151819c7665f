"""trace_sharded(..., exact_sum=True) on CPU: two and three gloo ranks run the exact-sum protocol (agreement, integer
all-reduce of the words, empty ranks, failures) around a closed-form fake of trace_bundle(..., reduce_exact=fn). The fake
books integer words per beam and converts them with a fixed rule, so the reduced profile must equal the fake applied to
the unsharded bundle bit for bit, under contiguous and block-cyclic sharding, with ragged beams and with a rank that has no
rays. A failure on one rank must make every rank raise, and no worker may be left behind."""
import json
import multiprocessing
import os
import sys
from datetime import timedelta

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_PSI = 13
N_BEAMS = 4
SIZES = (23, 7, 31, 20)  # ragged beams
ROW = N_PSI + 2
SCALE = 2.0 ** 40        # the fake's quantum: 2^-40
JOIN_S = 120


def bundle():
    n = sum(SIZES)
    k = np.arange(n, dtype=np.float64)
    pos = np.stack([np.sin(k), np.cos(0.3 * k), 0.01 * k], axis=1)
    dirs = np.stack([np.cos(k), np.sin(0.7 * k), np.ones(n)], axis=1)
    w = (1.0 + (k % 5)) / 3.0
    beam_id = np.repeat(np.arange(N_BEAMS, dtype=np.int32), SIZES)
    return pos, dirs, w, beam_id


def _per_ray(pos, dirs):
    key = pos[:, 0] * 3.0 + pos[:, 2] - dirs[:, 1]
    P_final = np.exp(-np.abs(key))
    shell = (np.floor(np.abs(key) * 7.0).astype(int)) % N_PSI
    return key, P_final, shell


def _convert(words, n_beams):
    """the fake's fixed conversion: bin value = its first word times the quantum, shells over a fixed dV"""
    v = words[2:2 + n_beams * ROW * 8].reshape(n_beams, ROW, 8)[:, :, 0].astype(np.float64) / SCALE
    v[:, :N_PSI] /= 1.0 + np.arange(N_PSI)
    return v.ravel()


def fake_trace(pos, dirs, w, beam_id=None, *, reduce_exact=None, extra_words=0, n_beams=N_BEAMS):
    """trace_bundle(..., exact_sum=True, reduce_exact=...) in closed form: integer bookings w (1 - P_final) into a shell and
    the deposited bin, w into the weight bin, 2 status words in front, 8 words per bin."""
    beam_id = np.zeros(len(w), dtype=np.int64) if beam_id is None else np.asarray(beam_id, dtype=np.int64)
    key, P_final, shell = _per_ray(pos, dirs)
    words = np.zeros(2 + n_beams * ROW * 8 + extra_words, dtype=np.int64)
    dep = np.round(w * (1.0 - P_final) * SCALE).astype(np.int64)
    np.add.at(words, 2 + (beam_id * ROW + shell) * 8, dep)
    np.add.at(words, 2 + (beam_id * ROW + N_PSI) * 8, dep)
    np.add.at(words, 2 + (beam_id * ROW + N_PSI + 1) * 8, np.round(w * SCALE).astype(np.int64))
    words[0] = 3 * len(w)
    local_vector = _convert(words, n_beams)
    if reduce_exact is not None:
        t = torch.from_numpy(words)
        reduce_exact(t)
        words = t.numpy()
    rows = _convert(words, n_beams).reshape(n_beams, ROW)
    one = n_beams == 1
    return dict(dP_dV=rows[0, :N_PSI] if one else rows[:, :N_PSI], deposited_power=float(rows[0, N_PSI]) if one else rows[:, N_PSI],
                sum_weights=float(rows[0, -1]) if one else rows[:, -1], local_vector=local_vector, P_final=P_final,
                n_points=(2 + np.floor(100 * np.abs(key))).astype(np.int32), status=(np.abs(key) > 5.0).astype(np.int32) * 2)


def _single(pos, dirs, w, *, reduce_exact=None):
    return fake_trace(pos, dirs, w, reduce_exact=reduce_exact, n_beams=1)


# name, trace_sharded keywords, multi-beam
CASES = (("contig", dict(sharding="contiguous"), True), ("cyclic", dict(sharding="block_cyclic", block=7), True),
         ("beams", dict(sharding="block_cyclic", block=40), True),  # 81 rays, 3 blocks
         ("fewblocks", dict(sharding="block_cyclic", block=50), True),  # 2 blocks: the third rank has no rays
         ("single", dict(sharding="block_cyclic", block=11), False))
KEYS = ("dP_dV", "deposited_power", "sum_weights", "P_final", "n_points", "status")


def _errors(fn):
    try:
        fn()
    except Exception as e:  # noqa: BLE001 — the test compares every rank's error
        return f"{type(e).__name__}: {e}"
    return None


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world, timeout=timedelta(seconds=60))
    from torj_jl_b200.distributed import trace_sharded

    pos, dirs, w, beam_id = bundle()
    res, errs = {}, {}
    for name, kw, multi in CASES:
        if multi:
            r = trace_sharded(fake_trace, pos, dirs, w, n_beams=N_BEAMS, per_ray=dict(beam_id=beam_id), exact_sum=True, **kw)
        else:
            r = trace_sharded(_single, pos, dirs, w, exact_sum=True, **kw)
        for k in KEYS:
            res[f"{name}_{k}"] = np.asarray(r[k])
        res[f"{name}_idx_{rank}"] = r["idx"]
        res[f"{name}_local_vector_{rank}"] = r["local_vector"]

    def raising(p, d, ww, beam_id, *, reduce_exact):
        if rank == 1:
            raise ValueError("rank 1 cannot trace")
        return fake_trace(p, d, ww, beam_id, reduce_exact=reduce_exact)

    def longer(p, d, ww, beam_id, *, reduce_exact):
        return fake_trace(p, d, ww, beam_id, reduce_exact=reduce_exact, extra_words=8 * rank)

    def late(p, d, ww, beam_id, *, reduce_exact):
        r = fake_trace(p, d, ww, beam_id, reduce_exact=reduce_exact)
        if rank == 0:
            raise ValueError("rank 0 failed converting")
        return r

    def forgets(p, d, ww, beam_id, *, reduce_exact):
        return fake_trace(p, d, ww, beam_id)

    for name, fn in (("raising", raising), ("longer", longer), ("late", late), ("forgets", forgets)):
        for sharding, block in (("contiguous", 1), ("block_cyclic", 50)):  # block 50: with 3 ranks one is empty
            errs[f"{name}_{sharding}"] = _errors(lambda: trace_sharded(
                fn, pos, dirs, w, n_beams=N_BEAMS, per_ray=dict(beam_id=beam_id), exact_sum=True, sharding=sharding,
                block=block))
    # the protocol is still in step after the refusals: a valid call gives the earlier bits
    r = trace_sharded(fake_trace, pos, dirs, w, n_beams=N_BEAMS, per_ray=dict(beam_id=beam_id), exact_sum=True)
    res["again_dP_dV"] = r["dP_dV"]
    np.savez(os.path.join(out_dir, f"rank{rank}.npz"), **res)
    with open(os.path.join(out_dir, f"rank{rank}.json"), "w") as f:
        json.dump(errs, f)
    dist.barrier()
    dist.destroy_process_group()


def _run(tmp_path, world):
    """spawn the ranks; every process is joined, or terminated and joined when one fails or the time runs out"""
    port = 33500 + (os.getpid() % 2000) + 7 * world
    ctx = multiprocessing.get_context("spawn")
    procs = [ctx.Process(target=_worker, args=(r, world, port, str(tmp_path))) for r in range(world)]
    try:
        for p in procs:
            p.start()
        for p in procs:
            p.join(JOIN_S)
    finally:
        for p in procs:
            if p.is_alive():
                p.terminate()
            p.join(10)
    assert all(not p.is_alive() for p in procs)
    assert [p.exitcode for p in procs] == [0] * world
    return ([np.load(tmp_path / f"rank{r}.npz") for r in range(world)],
            [json.load(open(tmp_path / f"rank{r}.json")) for r in range(world)])


def bits(a):
    return np.ascontiguousarray(np.atleast_1d(np.asarray(a, dtype=np.float64))).view(np.uint64)


def _check(tmp_path, world):
    ranks, errs = _run(tmp_path, world)
    pos, dirs, w, beam_id = bundle()
    full = fake_trace(pos, dirs, w, beam_id)
    single = _single(pos, dirs, w)
    for name, kw, multi in CASES:
        want = full if multi else single
        idx = [ranks[r][f"{name}_idx_{r}"] for r in range(world)]
        assert np.array_equal(np.sort(np.concatenate(idx)), np.arange(len(w)))  # the shards partition the bundle
        if name == "fewblocks" and world == 3:
            assert len(idx[2]) == 0
        for r, g in enumerate(ranks):                                            # every rank, empty ones too
            for k in ("dP_dV", "deposited_power", "sum_weights"):
                assert np.array_equal(bits(g[f"{name}_{k}"]), bits(want[k])), (name, k, r)
            for k in ("P_final", "n_points", "status"):
                assert np.array_equal(g[f"{name}_{k}"], want[k]), (name, k, r)
            mine = fake_trace(pos[idx[r]], dirs[idx[r]], w[idx[r]], beam_id[idx[r]] if multi else None,
                              n_beams=N_BEAMS if multi else 1)
            assert np.array_equal(bits(g[f"{name}_local_vector_{r}"]), bits(mine["local_vector"])), (name, r)
        assert bits(want["dP_dV"]).any()
    for g in ranks:
        assert np.array_equal(bits(g["again_dP_dV"]), bits(full["dP_dV"]))
    for sharding in ("contiguous", "block_cyclic"):
        e = [x[f"raising_{sharding}"] for x in errs]
        assert e[1] == "ValueError: rank 1 cannot trace"
        assert all(x is not None and "failed on a rank before the exact sum" in x for i, x in enumerate(e) if i != 1)
        e = [x[f"longer_{sharding}"] for x in errs]
        assert len(set(e)) == 1 and "differ in length" in e[0]
        e = [x[f"late_{sharding}"] for x in errs]
        assert e[0] == "ValueError: rank 0 failed converting"
        assert all("failed after the exact sum" in x for x in e[1:])
        e = [x[f"forgets_{sharding}"] for x in errs]  # an empty rank has no trace_fn to blame
        assert "did not call reduce_exact" in e[0]
        assert all(x is not None and ("did not call reduce_exact" in x or "before the exact sum" in x) for x in e)


def test_two_rank_exact_sharded_trace_is_bit_identical(tmp_path):
    _check(tmp_path, 2)


def test_three_rank_exact_sharded_trace_is_bit_identical(tmp_path):
    _check(tmp_path, 3)


def test_one_process_exact_sharded_trace_is_bit_identical():
    sys.path.insert(0, ROOT)
    from torj_jl_b200.distributed import trace_sharded

    pos, dirs, w, beam_id = bundle()
    full = fake_trace(pos, dirs, w, beam_id)
    r = trace_sharded(fake_trace, pos, dirs, w, n_beams=N_BEAMS, per_ray=dict(beam_id=beam_id), exact_sum=True)
    for k in ("dP_dV", "deposited_power", "sum_weights"):
        assert np.array_equal(bits(r[k]), bits(full[k])), k
    assert np.array_equal(bits(r["local_vector"]), bits(full["local_vector"]))
    with pytest.raises(ValueError, match="at least one ray"):
        trace_sharded(fake_trace, pos[:0], dirs[:0], w[:0], exact_sum=True)
