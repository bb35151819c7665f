"""bench.py --dump-outputs: the results of the last timed step as .npy files, so that two builds can be compared output for
output on the same inputs.  CPU: the writer (float64, size budget, seeded ray sample) and the argument checks.  GPU: what
the bench writes equals a direct trace of the same bundle."""
import glob
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

import bench


class FakeBundle:
    def __init__(self, n, n_beams, seed):
        g = np.random.default_rng(seed)
        self.r = dict(dP_dV=g.random((n_beams, bench.N_PSI)), deposited_power=g.random(n_beams), P_final=g.random(n),
                      P_deposited_ray=g.random(n), n_points=g.integers(0, 500, n, dtype=np.int32),
                      status=g.integers(0, 4, n, dtype=np.int32), counters=g.integers(0, 10**9, 8))

    def results(self):
        return self.r


def _load(d):
    return {os.path.basename(p)[:-4]: np.load(p) for p in glob.glob(os.path.join(d, "*.npy"))}


def test_dump_outputs_concatenates_bundles_and_samples_rays_within_the_budget(tmp_path):
    bs = [FakeBundle(3000, 2, 1), FakeBundle(1000, 3, 2)]
    bench.dump_outputs(str(tmp_path / "all"), bs, 0, 1)
    a = _load(tmp_path / "all")
    assert set(a) == {"dP_dV", "deposited_power", "P_final", "P_deposited_ray", "n_points", "status", "counters"}
    assert all(v.dtype == np.float64 for v in a.values())
    assert a["dP_dV"].shape == (5, bench.N_PSI) and np.array_equal(a["dP_dV"][2:], bs[1].r["dP_dV"])
    assert np.array_equal(a["n_points"], np.concatenate([b.r["n_points"] for b in bs]))
    assert np.array_equal(a["counters"], bs[0].r["counters"] + bs[1].r["counters"])

    budget = 100_000
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), bs, 0, 1, budget=budget)
    s1, s2 = _load(tmp_path / "s1"), _load(tmp_path / "s2")
    assert sum(v.nbytes for v in s1.values()) <= budget
    idx = s1["ray_index"].astype(int)
    assert np.array_equal(s1["ray_index"], s2["ray_index"]) and np.all(np.diff(idx) > 0) and len(idx) < 4000
    assert np.array_equal(s1["P_final"], a["P_final"][idx]) and np.array_equal(s1["status"], a["status"][idx])
    assert np.array_equal(s1["dP_dV"], a["dP_dV"])

    bench.dump_outputs(str(tmp_path / "ranks"), bs[:1], 1, 2)
    assert set(_load(tmp_path / "ranks")) == {f"rank1_{k}" for k in a}


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_bench_rejects_arguments_it_cannot_honour(argv):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True)
    assert r.returncode == 2 and "error" in r.stderr


@pytest.mark.gpu
def test_bench_dump_equals_a_direct_trace_of_the_same_bundle(tmp_path):
    import torj_jl_b200 as tj
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--small", "--steps", "2", "--warmup", "1", "--no-cpu-baseline",
                        "--no-parity", "--no-exact", "--dump-outputs", str(out)], capture_output=True, text=True, cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr[-4000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["warmup"] == 1
    d = _load(out)
    assert sum(v.nbytes for v in d.values()) <= 64_000_000 and all(v.dtype == np.float64 for v in d.values())
    tj.abs_Al_init(bench.N_GL)
    pos, dirs, w = bench.beam_bundle("small")
    ref = tj.trace_bundle(tj.Plasma(*tj.solovev_arrays(bench.GRID, bench.GRID).values()), pos, dirs, w, 95e9, 1, bench.S_MAX,
                          np.linspace(0.0, 1.0, bench.N_PSI))
    assert np.array_equal(d["n_points"], ref["n_points"]) and np.array_equal(d["status"], ref["status"])
    assert np.abs(d["P_final"] - ref["P_final"]).max() < 1e-11
    assert np.abs(d["P_deposited_ray"] - ref["P_deposited_ray"]).max() < 1e-11
    assert np.abs(d["dP_dV"][0] - ref["dP_dV"]).max() <= 1e-9 * np.abs(ref["dP_dV"]).max()
    assert abs(d["deposited_power"][0] - ref["deposited_power"]) < 1e-11
    assert d["counters"][0] == ref["counters"]["n_acc"] == line["roofline"]["counters"]["n_acc"]
