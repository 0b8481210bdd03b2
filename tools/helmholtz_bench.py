#!/usr/bin/env python
"""Helmholtz problems (Hierarchy.set_helmholtz) against the Poisson problem and against the smoother-only shift
(Hierarchy.set_lambda alone), fp64, V(1,1) cycles with the default options (fused schedule, CUDA graphs).

    python tools/helmholtz_bench.py [--configs D,B] [--reps 10] [--warmup 3] [--parent DIR] [--out FILE]

Per config (bench.py's CONFIGS, one GPU) and state: Poisson (lambda = 0), Helmholtz and smoother-only at lambda h^2 =
-1e-2 and -1 on the finest cells of level 0:
  vcycle_ms      one vcycle, CUDA events around each call, median over --reps after --warmup
  gmg_solve      cycles and wall ms of gmg_solve to 1e-10 from zero, trig right-hand side
  first_solve_ms set_helmholtz (or set_lambda) plus the first gmg_solve after it, host clock around both ending in a device
                 synchronise; next_solve_ms is the same solve again (graphs captured)
--parent DIR (a built checkout of the commit before the Helmholtz operator) adds the record that the lambda = 0 path did
not move:
  bench          bench.py --gpus 1 (config D, --bench-runs times, alternating parent and this tree): DOF/s and ms per step
  res_usage      cuobjdump -res-usage of the kernels the change touched, both libraries: registers, stack, local bytes
The card name, power limit and maximum SM clock come from a read-only nvidia-smi query in the same run.  Prints one JSON
line (and writes it to --out)."""
import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402  (CONFIGS, Env, build_hierarchy)
from fmg_bench import gpu_info, timed  # noqa: E402


def measure(env, cfg, reps, warmup):
    pps = env.pps
    n = bench.CONFIGS[cfg][3]
    h, mesh, _, setup_s = bench.build_hierarchy(env, cfg)
    hmin = float(mesh.level_arrays(n)[0]["spacings"].min())
    opts = pps.CycleOpts.default()
    f, u = h.new_vec(0), h.new_vec(0)
    h.init_trig_rhs(f)
    states = [("poisson", 0.0, "helmholtz")]
    for c in (-1e-2, -1.0):
        states += [("helmholtz_%g" % c, c / hmin ** 2, "helmholtz"), ("smoother_only_%g" % c, c / hmin ** 2, "lambda")]
    out = {}
    for name, lam, how in states:
        h.set_helmholtz(0.0)
        env.ctx.sync()
        t0 = time.perf_counter()
        (h.set_helmholtz if how == "helmholtz" else h.set_lambda)(lam)
        u.set(0.0)
        its, rel = h.gmg_solve(f, u, opts, tol=1e-10, max_it=200)
        env.ctx.sync()
        first = (time.perf_counter() - t0) * 1e3
        u.set(0.0)
        env.ctx.sync()
        t0 = time.perf_counter()
        h.gmg_solve(f, u, opts, tol=1e-10, max_it=200)
        env.ctx.sync()
        nxt = (time.perf_counter() - t0) * 1e3
        for _ in range(warmup):
            h.vcycle(f, u, opts)
        t = [timed(env.ctx, lambda: h.vcycle(f, u, opts)) for _ in range(reps)]
        out[name] = {"lambda": lam, "lambda_h2": lam * hmin ** 2, "vcycle_ms": statistics.median(t), "vcycle_ms_min_max": [min(t), max(t)],
                     "gmg_solve": {"cycles": its, "rel_residual": rel, "ms": nxt}, "first_solve_ms": first, "next_solve_ms": nxt}
    for x in (f, u):
        x.close()
    h.close()
    mesh.close()
    return {"workload": bench.CONFIGS[cfg][5], "setup_s": setup_s, "h_min": hmin, "reps": reps, "states": out}


CHANGED = ("apply_tma_kernel", "apply3d32_tma_kernel", "jacobi_update_kernel", "smooth_kernel", "smooth3d16_kernel", "smooth3d32c_kernel",
           "smooth3d32n_kernel", "smooth2d32_kernel")


def res_usage(tree):
    """{demangled kernel name: [registers, stack bytes, local bytes]} of the touched kernels of tree's libtgpu.so"""
    cuobjdump = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")
    lib = os.path.join(tree, "pressurepoissonsolver_b200", "libtgpu.so")
    txt = subprocess.run([cuobjdump, "-res-usage", lib], capture_output=True, text=True, check=True).stdout
    out, fn = {}, None
    for line in txt.splitlines():
        m = re.match(r"\s*Function (\S+):", line)
        if m:
            fn = m.group(1)
            continue
        m = re.search(r"REG:(\d+) STACK:(\d+) SHARED:\d+ LOCAL:(\d+)", line)
        if m and fn:
            out[fn] = [int(x) for x in m.groups()]
            fn = None
    names = subprocess.run(["c++filt"], input="\n".join(out), capture_output=True, text=True).stdout.split("\n")
    # (the name without its argument list: the change added arguments to some kernels)
    short = {k: re.sub(r"\(.*$", "", d) for k, d in zip(out, names)}
    return {short[k]: v for k, v in out.items() if any(c in short[k] for c in CHANGED)}


def lambda0_record(parent, runs, steps, warmup):
    cmd = [sys.executable, "bench.py", "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup), "--no-cpu-baseline",
           "--no-other-configs"]
    bench_runs = []
    for k in range(runs):
        for arm, tree in (("parent", parent), ("change", ROOT)):
            res = subprocess.run(cmd, cwd=tree, capture_output=True, text=True, check=True)
            r = json.loads(res.stdout.strip().splitlines()[-1])
            bench_runs.append({"arm": arm, "run": k, "dof_per_s": r["value"], "ms_per_step": r["ms_per_step"]})
    a, b = res_usage(parent), res_usage(ROOT)
    usage = {k: {"parent": a.get(k), "change": b.get(k)} for k in sorted(set(a) | set(b))}
    return {"bench": {"command": " ".join(cmd[1:]), "runs": bench_runs}, "res_usage": usage,
            "local_bytes_max_change": max(v[2] for v in b.values())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="D,B")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--parent", default=None)
    ap.add_argument("--bench-runs", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    env = bench.Env()
    if env.world != 1:
        sys.exit("helmholtz_bench runs on one GPU")
    res = {"gpu": gpu_info(), "cycle": "V(1,1), fused schedule, CUDA graphs", "configs": {}}
    for cfg in args.configs.split(","):
        res["configs"][cfg] = measure(env, cfg, args.reps, args.warmup)
    if args.parent:
        env.ctx.close()  # (bench.py runs in processes of its own)
        res["lambda0_path"] = lambda0_record(os.path.abspath(args.parent), args.bench_runs, 20, 5)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    if not args.parent:
        env.ctx.close()


if __name__ == "__main__":
    main()
