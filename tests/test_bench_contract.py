"""The JSON lines bench.py printed in the committed driver-style runs (profiles/r02_bench_*.json) carry every key of the
measurement contract, agree with each other about the workload, and are internally consistent (value = cells / time,
roofline.frac = achieved / peak, the reference arm ran the same config); and what --dump-outputs writes."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import MESHES, ROOT, rel_l2

PROFILES = os.path.join(ROOT, "profiles")
BENCH = os.path.join(ROOT, "bench.py")


def load(name):
    with open(os.path.join(PROFILES, name)) as fh:
        return json.loads([l for l in fh.read().splitlines() if l.startswith("{")][-1])


@pytest.mark.parametrize("n", [1, 2, 4, 8])
def test_our_arm_line(n):
    d = load("r02_bench_%dgpu.json" % n)
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
              "data", "config", "roofline", "e2e", "gpu_launches", "clocks", "setup_s", "time_to_solution"):
        assert k in d, k
    assert d["n_gpus"] == n and d["warmup"] >= 3 and d["higher_is_better"] is True and d["dtype"] == "f64" and d["vs_baseline"] is None
    assert d["scaling"] == "strong" and "workload" in d["config"] and d["config"]["cells"] == 1073741824
    assert abs(d["value"] / (d["config"]["cells"] / (d["ms_per_step"] * 1e-3)) - 1) < 1e-9
    r = d["roofline"]
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert k in r, k
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12
    e = d["e2e"]
    # whole-job bytes (the committed N > 1 lines were printed before bench.py switched from rank 0's share to the job total)
    assert e["unit"] == d["unit"] and e["h2d_bytes_per_step"] == e["d2h_bytes_per_step"]
    assert e["h2d_bytes_per_step"] in (8 * d["config"]["cells"], 8 * d["config"]["cells"] // n)
    assert e["value"] < d["value"]  # host copies inside the timed region: never the device-resident number repeated
    assert d["gpu_launches"] > 0
    c = d["clocks"]
    assert not set(c["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    assert c["sm_mhz"] > 0.9 * c["sm_max_mhz"]
    if n == 1:
        b = d["cpu_baseline"]
        assert b["kind"] == "reference" and b["cores"] == 1 and b["value"] > 0 and b["sample"]
    else:
        p = d["multi_gpu_parity"]
        assert p["ok"] and p["max_rel_l2"] < p["tolerance"] <= 1e-10


def test_scaling_curve_is_on_one_mesh_and_reference_arm_matches():
    lines = {n: load("r02_bench_%dgpu.json" % n) for n in (1, 2, 4, 8)}
    ref = load("r02_bench_reference_arm.json")
    w = lines[1]["config"]["workload"]
    assert all(l["config"]["workload"] == w and l["metric"] == lines[1]["metric"] for l in lines.values())
    assert ref["impl"] == "reference" and ref["config"] == lines[1]["config"] and ref["metric"] == lines[1]["metric"] and ref["unit"] == lines[1]["unit"]
    assert ref["e2e"]["h2d_bytes_per_step"] == 0 and ref["e2e"]["value"] == ref["value"] and ref["cpu_baseline"]["value"] == ref["value"]
    eff = {n: lines[n]["value"] / (n * lines[1]["value"]) for n in (2, 4, 8)}
    assert eff[2] > 0.9 and eff[4] > 0.85 and eff[8] > 0.8, eff  # north star: >= 0.8 at 8 GPUs on a >= 1 B-cell mesh
    assert lines[1]["roofline"]["vcycle_frac"] >= 0.6              # north star: >= 60 % of the HBM roofline per V-cycle


def test_dump_outputs_writes_the_whole_result_or_a_fixed_sample(tmp_path):
    """bench.py --dump-outputs: float64, all of u up to DUMP_MAX_VALUES cells, above that the same sorted sample every run"""
    spec = importlib.util.spec_from_file_location("bench_mod", BENCH)
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)

    class Vec:
        def __init__(self, n):
            self.n = n

        def download(self):
            return np.arange(self.n, dtype=np.float64)

    bench.DUMP_MAX_VALUES = 64
    bench.dump_outputs(str(tmp_path / "whole"), Vec(64))
    assert np.array_equal(np.load(tmp_path / "whole" / "u.npy"), np.arange(64.0))
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), Vec(1000))
    a, b = np.load(tmp_path / "a" / "u.npy"), np.load(tmp_path / "b" / "u.npy")
    assert a.dtype == np.float64 and a.size == 64 and np.array_equal(a, b)
    assert np.all(np.diff(a) > 0) and a[-1] < 1000  # distinct cells in index order


@pytest.mark.parametrize("argv,env", [(["--impl", "reference"], {}), ([], {"WORLD_SIZE": "2"})])
def test_dump_outputs_is_refused_where_there_is_no_single_gpu_result(tmp_path, argv, env):
    """the reference arm computes no u, and under torchrun every rank holds only its own patches"""
    out = tmp_path / "dump"
    res = subprocess.run([sys.executable, BENCH, "--dump-outputs", str(out)] + argv, env=dict(os.environ, **env),
                         capture_output=True, text=True, timeout=120)
    assert res.returncode == 2 and "--dump-outputs" in res.stderr, res.stderr
    assert not out.exists()


@pytest.mark.gpu
def test_dump_outputs_is_the_timed_cycles_result(tmp_path):
    """main() hands --dump-outputs to the timed measurement: on a workload small enough to be written whole (config
    `small`, 2,097,152 cells), u.npy is one V-cycle of the workload's right-hand side, checked against the oracle"""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import gmg_oracle as go
    res = subprocess.run([sys.executable, BENCH, "--config", "small", "--cycle-only", "--no-other-configs", "--no-cpu-baseline",
                          "--steps", "2", "--warmup", "3", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout + res.stderr
    u = np.load(tmp_path / "u.npy")
    levels = go.build_hierarchy(os.path.join(MESHES, "3uni.bin"), 3, 16, 1)
    f, _ = go.trig_rhs(levels[0])
    assert u.dtype == np.float64 and u.size == f.size == 2097152
    assert rel_l2(u, go.vcycle(levels, f)) < 1e-12
