"""Exact sums across processes on the GPU: trace_bundle(..., exact_sum=True, reduce_exact=fn) and
distributed.trace_sharded(..., exact_sum=True).

Profiles are compared as bits. Ranks are spawned processes, each with its own context; under gloo they all share device 0,
so the protocol runs on one GPU. With two or more visible GPUs the same cases also run under NCCL, one rank per GPU.
lanes_per_ray is fixed in every case: the automatic width depends on the bundle's size, so a shard could pick another."""
import ctypes as C
import multiprocessing
import os
import sys
from datetime import timedelta

import numpy as np
import pytest
import torch

import torj_jl_b200 as tj
from torj_jl_b200 import _lib

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_PSI, S_MAX = 200, 1.0
PSI = np.linspace(0.0, 1.0, N_PSI)
JOIN_S = 600
KEYS = ("dP_dV", "deposited_power", "sum_weights")


def bits(a):
    return np.ascontiguousarray(np.atleast_1d(np.asarray(a, dtype=np.float64))).view(np.uint64)


def same_bits(a, b):
    return np.array_equal(bits(a), bits(b))


def plasmas():
    """built like MultiGPU's per-device copies (torj_plasma_create_from_data), so its results compare bit for bit"""
    return [tj.Plasma(*tj.solovev_arrays(129, 129, **kw).values(), build="device") for kw in ({}, dict(Te0=6e3))]


def beams(n_beams):
    """n_beams beams of 1 025 rays at different steering angles"""
    P, D, W, B = [], [], [], []
    for b, pol in enumerate(np.linspace(15.0, 40.0, n_beams)):
        p, d, w = tj.launch_peripheral_rays(np.array([2.5, 0.0, 0.4]), tj.pol_tor_angles_2_vector(np.deg2rad(pol), 0.02 * b),
                                            0.0174, 1 / 3.99, 95e9, N_rings=7, min_azimuthal_points=20)
        P.append(p); D.append(d); W.append(w); B.append(np.full(len(w), b, dtype=np.int32))
    return np.concatenate(P), np.concatenate(D), np.concatenate(W), np.concatenate(B)


def cases():
    """name -> (bundle, keywords of trace_bundle, keywords of trace_sharded, compare with MultiGPU)"""
    ALB = _lib.default_options(lanes_per_ray=1)
    pos, dirs, w, bid = beams(4)
    n1 = int((bid == 0).sum())
    warm = tj.launch_peripheral_rays(np.array([2.5, 0.0, 0.4]), tj.pol_tor_angles_2_vector(np.deg2rad(30.0), 0.0), 0.0174,
                                     1 / 3.99, 95e9)
    return {
        "beam": ((pos[:n1], dirs[:n1], w[:n1], None), dict(options=ALB), dict(sharding="contiguous"), True),
        "set": ((pos, dirs, w, bid), dict(options=ALB, n_beams=4, beam_plasma=np.array([1, 0, 0, 1], dtype=np.int32)),
                dict(sharding="block_cyclic", block=n1, n_beams=4), True),
        "two_beams": ((pos[:2 * n1], dirs[:2 * n1], w[:2 * n1], bid[:2 * n1]), dict(options=ALB, n_beams=2),
                      dict(sharding="block_cyclic", block=n1, n_beams=2), True),
        "warm": ((*warm, None), dict(options=_lib.default_options(absorption_model=1, lanes_per_ray=32), s_max=0.6),
                 dict(sharding="contiguous"), False),
    }


def _plasma_arg(pls, kw):
    return pls if "beam_plasma" in kw else pls[0]


def _warm_plasma():
    return tj.Plasma(*tj.solovev_arrays(129, 129, Te0=10e3).values(), build="device")


def single(name, pls):
    (pos, dirs, w, bid), kw, _, _ = cases()[name]
    kw = dict(kw)
    s_max = kw.pop("s_max", S_MAX)
    pl = _warm_plasma() if name == "warm" else _plasma_arg(pls, kw)
    return tj.trace_bundle(pl, pos, dirs, w, 95e9, 1, s_max, PSI, beam_id=bid, exact_sum=True, **kw)


def _worker(rank, world, backend, port, out_dir):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), LOCAL_RANK=str(rank if backend == "nccl" else 0))
    device = None
    if backend == "nccl":
        torch.cuda.set_device(rank)
        device = torch.device("cuda", rank)
    dist.init_process_group(backend, rank=rank, world_size=world, timeout=timedelta(seconds=120))
    import torj_jl_b200 as tj
    from torj_jl_b200.distributed import trace_sharded

    tj.abs_Al_init(24)
    pls = plasmas()
    res = {}
    for name, ((pos, dirs, w, bid), kw, skw, _) in cases().items():
        kw = dict(kw)
        s_max = kw.pop("s_max", S_MAX)
        pl = _warm_plasma() if name == "warm" else _plasma_arg(pls, kw)
        kw.pop("n_beams", None)
        nb = skw.get("n_beams", 1)

        def trace_fn(p, d, ww, beam_id=None, *, reduce_exact):
            return tj.trace_bundle(pl, p, d, ww, 95e9, 1, s_max, PSI, beam_id=beam_id, n_beams=nb, exact_sum=True,
                                   reduce_exact=reduce_exact, **kw)

        r = trace_sharded(trace_fn, pos, dirs, w, per_ray=dict(beam_id=bid) if bid is not None else None, device=device,
                          exact_sum=True, **skw)
        for k in KEYS + ("P_final", "status", "local_vector"):
            res[f"{name}_{k}"] = np.asarray(r[k])
        res[f"{name}_n_local"] = len(r["idx"])
    # one rank's weights beyond 2^40: refused on that rank before its trace, every rank raises, nobody waits
    (pos, dirs, w, _), kw, skw, _ = cases()["beam"]
    big = w.copy()
    big[-1] = 2.0 ** 41  # the last ray belongs to the last rank

    def trace_fn(p, d, ww, *, reduce_exact):
        return tj.trace_bundle(pls[0], p, d, ww, 95e9, 1, S_MAX, PSI, exact_sum=True, reduce_exact=reduce_exact, **kw)

    try:
        trace_sharded(trace_fn, pos, dirs, big, device=device, exact_sum=True, **skw)
        res["refusal"] = "none"
    except Exception as e:  # noqa: BLE001
        res["refusal"] = f"{type(e).__name__}: {e}"
    r = trace_sharded(trace_fn, pos, dirs, w, device=device, exact_sum=True, **skw)
    res["after_refusal_dP_dV"] = r["dP_dV"]
    np.savez(os.path.join(out_dir, f"{backend}{world}_rank{rank}.npz"), **res)
    dist.barrier()
    dist.destroy_process_group()


def _spawn(tmp_path, world, backend):
    port = 35500 + (os.getpid() % 2000) + 11 * world + (5 if backend == "nccl" else 0)
    ctx = multiprocessing.get_context("spawn")
    procs = [ctx.Process(target=_worker, args=(r, world, backend, port, str(tmp_path))) for r in range(world)]
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
    return [dict(np.load(tmp_path / f"{backend}{world}_rank{r}.npz")) for r in range(world)]


@pytest.fixture(scope="module", autouse=True)
def _abs_al_init():
    tj.abs_Al_init(24)


@pytest.fixture(scope="module")
def pls():
    return plasmas()


@pytest.fixture(scope="module")
def reference(pls):
    """one process tracing each whole bundle, and MultiGPU over the visible devices"""
    ref = {name: single(name, pls) for name in cases()}
    mg = tj.MultiGPU()
    try:
        mg.abs_Al_init(24)
        print(f"\n{torch.cuda.device_count()} visible GPU(s); MultiGPU over {mg.n_devices}")
        for name, ((pos, dirs, w, bid), kw, skw, multi) in cases().items():
            if multi:
                kw = dict(kw)
                ref[name]["multi"] = mg.trace_bundle(_plasma_arg(pls, kw), pos, dirs, w, 95e9, 1, S_MAX, PSI, beam_id=bid,
                                                     exact_sum=True, **kw)
    finally:
        mg.close()
    return ref


def test_identity_reduction_equals_plain_exact_trace(pls):
    pos, dirs, w, bid = beams(3)
    for pl, kw in ((pls[0], dict(trajectories=(1000, 60))),
                   (pls, dict(beam_id=bid, n_beams=3, beam_plasma=np.array([1, 0, 1], dtype=np.int32),
                              trajectories=(2000, 100)))):
        opt = _lib.default_options(lanes_per_ray=1)
        plain = tj.trace_bundle(pl, pos, dirs, w, 95e9, 1, S_MAX, PSI, options=opt, exact_sum=True, **kw)
        seen = []

        def ident(words):
            seen.append((words.is_cuda, words.dtype, words.numel()))
        r = tj.trace_bundle(pl, pos, dirs, w, 95e9, 1, S_MAX, PSI, options=opt, exact_sum=True, reduce_exact=ident, **kw)
        nb = kw.get("n_beams", 1)
        assert seen == [(True, torch.int64, 2 + nb * (N_PSI + 2) * 8)]
        assert set(plain) <= set(r) and {"sum_weights", "local_vector"} <= set(r)
        for k in plain:
            if k == "counters":
                assert r[k] == plain[k]
            else:
                a, b = np.atleast_1d(np.asarray(r[k])), np.atleast_1d(np.asarray(plain[k]))
                assert a.dtype == b.dtype and np.array_equal(a.view(np.uint8), b.view(np.uint8)), k
        rows = r["local_vector"].reshape(nb, -1)
        assert same_bits(rows[:, :N_PSI].ravel(), np.ravel(plain["dP_dV"]))
        assert same_bits(rows[:, N_PSI], plain["deposited_power"])
        assert same_bits(rows[:, -1], r["sum_weights"])
        assert np.allclose(np.atleast_1d(r["sum_weights"]), [w[bid == q].sum() for q in range(nb)] if nb > 1 else [w.sum()],
                           rtol=1e-14)


def test_exact_words_refusals(pls):
    (pos, dirs, w, _), kw, _, _ = cases()["beam"]
    opt = kw["options"]
    ref = tj.trace_bundle(pls[0], pos, dirs, w, 95e9, 1, S_MAX, PSI, options=opt, exact_sum=True)
    L, ctx = tj.lib(), _lib.context()
    ptr, nw = _lib.c_vp(), C.c_int64()
    assert L.torj_bundle_device_exact_words(None, C.byref(ptr), C.byref(nw)) != 0
    assert b"bundle is NULL" in L.torj_last_error()
    assert L.torj_bundle_finalize_exact(None) != 0 and b"bundle is NULL" in L.torj_last_error()
    m = tj.solve.marshal_bundle(pos, dirs, w, 95e9, 1, PSI, None, 1)
    bh = _lib.c_vp()
    p = tj.solve._p
    _lib.check(L.torj_bundle_create(ctx, m["n"], p(m["pos"]), p(m["dir"]), p(m["w"]), p(m["f"]),
                                    m["mode"].ctypes.data_as(_lib.c_ip), 0, C.byref(bh)))
    try:
        for fn in (lambda: L.torj_bundle_device_exact_words(bh, C.byref(ptr), C.byref(nw)), lambda: L.torj_bundle_finalize_exact(bh)):
            assert fn() != 0 and b"nothing traced yet" in L.torj_last_error()
        _lib.check(L.torj_ctx_set_exact_sum(ctx, 0))
        _lib.check(L.torj_bundle_trace(bh, pls[0].handle(ctx), C.byref(opt), S_MAX, N_PSI, p(PSI)))
        for fn in (lambda: L.torj_bundle_device_exact_words(bh, C.byref(ptr), C.byref(nw)), lambda: L.torj_bundle_finalize_exact(bh)):
            assert fn() != 0 and b"did not book exact sums" in L.torj_last_error()
        _lib.check(L.torj_ctx_set_exact_sum(ctx, 1))
        _lib.check(L.torj_bundle_trace(bh, pls[0].handle(ctx), C.byref(opt), S_MAX, N_PSI, p(PSI)))
        _lib.check(L.torj_bundle_device_exact_words(bh, C.byref(ptr), C.byref(nw)))
        assert ptr.value and nw.value == 2 + (N_PSI + 2) * 8
        _lib.check(L.torj_bundle_finalize_exact(bh))  # converting the same words twice gives the same profile
        prof, dep = np.zeros(N_PSI), np.zeros(1)
        _lib.check(L.torj_bundle_results(bh, p(prof), p(dep), None, None, None, None, None))
        assert same_bits(prof, ref["dP_dV"]) and same_bits(dep, ref["deposited_power"])
    finally:
        L.torj_bundle_destroy(bh)
    r = tj.trace_bundle(pls[0], pos, dirs, w, 95e9, 1, S_MAX, PSI, options=opt, exact_sum=True,
                        reduce_exact=lambda words: None)
    assert same_bits(r["dP_dV"], ref["dP_dV"]) and same_bits(r["deposited_power"], ref["deposited_power"])


def _check_ranks(ranks, reference, world):
    for name, ((pos, dirs, w, bid), kw, skw, multi) in cases().items():
        want = reference[name]
        sw = [w[bid == q].sum() for q in range(skw["n_beams"])] if "n_beams" in skw else [w.sum()]
        if name == "two_beams" and world == 3:
            assert ranks[2][f"{name}_n_local"] == 0  # two beams over three ranks: the third has no rays
        for r, g in enumerate(ranks):
            for k in ("dP_dV", "deposited_power"):
                assert same_bits(g[f"{name}_{k}"], want[k]), (name, k, r)
                if multi:
                    assert same_bits(g[f"{name}_{k}"], want["multi"][k]), (name, k, r, "MultiGPU")
            assert np.allclose(np.atleast_1d(g[f"{name}_sum_weights"]), sw, rtol=1e-14)
            assert same_bits(g[f"{name}_sum_weights"], ranks[0][f"{name}_sum_weights"])
            assert same_bits(g[f"{name}_P_final"], want["P_final"]) and np.array_equal(g[f"{name}_status"], want["status"])
        assert sum(g[f"{name}_n_local"] for g in ranks) == len(w)
    e = [str(g["refusal"]) for g in ranks]
    assert "2^40" in e[-1], e
    assert all("failed on a rank before the exact sum" in x for x in e[:-1]), e
    for g in ranks:
        assert same_bits(g["after_refusal_dP_dV"], reference["beam"]["dP_dV"])


@pytest.mark.parametrize("world", [2, 3])
def test_gloo_ranks_on_one_gpu_equal_one_trace(tmp_path, reference, world):
    _check_ranks(_spawn(tmp_path, world, "gloo"), reference, world)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="NCCL ranks need two or more visible GPUs")
def test_nccl_ranks_one_per_gpu_equal_one_trace(tmp_path, reference):
    world = min(torch.cuda.device_count(), 3)
    _check_ranks(_spawn(tmp_path, world, "nccl"), reference, world)
