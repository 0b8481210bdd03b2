#!/usr/bin/env python
"""Full multigrid (Hierarchy.fmg) against one V-cycle and against the stationary solve, fp64, V(1,1) cycles, trig
right-hand side with its Dirichlet data passed as a boundary vector.

    python tools/fmg_bench.py [--configs B,D] [--reps 10] [--warmup 3] [--out FILE]

Per config (bench.py's CONFIGS, one GPU):
  time       ms of one vcycle and of one fmg with cycles = 1 and 2, alternated, CUDA events around each call, median over
             --reps after --warmup each (CUDA graphs: every call after the first replays)
  error      ||u - u_exact||_2 / ||u_exact||_2 of fmg (cycles 1, 2) and of u_h = gmg_solve to 1e-12 from zero
  solve      gmg_solve to 1e-10 from the fmg (cycles = 2) result and from zero: cycles and wall ms (the fmg ms not included)
The card name, power limit and maximum SM clock come from a read-only nvidia-smi query in the same run.  Prints one JSON
line (and writes it to --out)."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (CONFIGS, Env, build_hierarchy)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True, check=True).stdout.strip().splitlines()
    name, power, clock = [x.strip() for x in q[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def trig_boundary(h, mesh, n):
    """the exact solution of the 3D trig problem (apps/3d/steady.cpp) on the boundary face centres, boundary-vector layout"""
    d = mesh.level_arrays(n)[0]
    patch, side = h.boundary_sides()
    st, sp = d["starts"][patch], d["spacings"][patch]
    k = (np.arange(n) + 0.5)
    out = np.empty((patch.size, n * n))
    for s in range(6):
        sel = np.nonzero(side == s)[0]
        a = s // 2
        rem = [b for b in range(3) if b != a]  # face order: rem[0] fastest
        x = [None] * 3
        x[a] = (st[sel, a] + (sp[sel, a] * n if s % 2 else 0.0))[:, None, None]
        x[rem[0]] = st[sel, rem[0], None, None] + sp[sel, rem[0], None, None] * k[None, None, :]
        x[rem[1]] = st[sel, rem[1], None, None] + sp[sel, rem[1], None, None] * k[None, :, None]
        X, Y, Z = (c + 0.3 for c in x)
        g = np.sin(np.pi * X) * np.cos(2.0 / 3 * np.pi * Y) * np.sin(5.0 / 6 * np.pi * Z)
        out[sel] = np.broadcast_to(g, (sel.size, n, n)).reshape(sel.size, -1)
    return out


def timed(ctx, fn):
    ctx.sync()
    ctx.timer_start()
    fn()
    return ctx.timer_stop()


def measure(env, cfg, reps, warmup):
    pps = env.pps
    D, _, _, n, _, _ = bench.CONFIGS[cfg]
    assert D == 3
    h, mesh, _, setup_s = bench.build_hierarchy(env, cfg)
    opts = pps.CycleOpts.default()
    f, exact, u, w, e = (h.new_vec(0) for _ in range(5))
    h.init_trig_rhs(f, exact)
    b = h.new_boundary_vec(trig_boundary(h, mesh, n))
    xnorm = exact.two_norm()

    def err(v):
        e.copy(v)
        e.add_scaled(-1.0, exact)
        return e.two_norm() / xnorm

    calls = {"vcycle": lambda: h.vcycle(f, u, opts), "fmg1": lambda: h.fmg(f, w, b, opts, 1), "fmg2": lambda: h.fmg(f, w, b, opts, 2)}
    for _ in range(warmup):
        for fn in calls.values():
            fn()
    t = {k: [] for k in calls}
    for _ in range(reps):
        for k, fn in calls.items():
            t[k].append(timed(env.ctx, fn))
    times = {k + "_ms": statistics.median(v) for k, v in t.items()}
    times.update({k + "_ms_min_max": [min(v), max(v)] for k, v in t.items()})
    times["fmg1_over_vcycle"] = times["fmg1_ms"] / times["vcycle_ms"]
    times["fmg2_over_vcycle"] = times["fmg2_ms"] / times["vcycle_ms"]
    times["reps"] = reps
    # errors against the exact solution
    h.fmg(f, w, b, opts, 1)
    error = {"fmg1": err(w)}
    h.fmg(f, w, b, opts, 2)
    error["fmg2"] = err(w)
    h.fmg(f, w, None, opts, 2)
    error["fmg2_without_boundary_data"] = err(w)
    u.set(0.0)
    its_h, rel_h = h.gmg_solve(f, u, opts, tol=1e-12, max_it=100)
    error.update(u_h=err(u), u_h_cycles=its_h, u_h_rel_residual=rel_h)
    error["fmg2_over_u_h"] = error["fmg2"] / error["u_h"]
    # stationary solve to 1e-10 from the FMG result and from zero
    solve = {}
    for name, start in (("from_fmg2", lambda: h.fmg(f, u, b, opts, 2)), ("from_zero", lambda: u.set(0.0))):
        start()
        env.ctx.sync()
        t0 = time.perf_counter()
        its, rel = h.gmg_solve(f, u, opts, tol=1e-10, max_it=100)
        env.ctx.sync()
        solve[name] = {"cycles": its, "ms": (time.perf_counter() - t0) * 1e3, "rel_residual": rel, "error": err(u)}
    for x in (f, exact, u, w, e, b):
        x.close()
    h.close()
    mesh.close()
    return {"workload": bench.CONFIGS[cfg][5], "setup_s": setup_s, "time": times, "error": error, "gmg_solve_to_1e-10": solve}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="B,D")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    env = bench.Env()
    if env.world != 1:
        sys.exit("fmg_bench runs on one GPU")
    res = {"gpu": gpu_info(), "cycle": "V(1,1), fused schedule, CUDA graphs", "configs": {}}
    for cfg in args.configs.split(","):
        res["configs"][cfg] = measure(env, cfg, args.reps, args.warmup)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    env.ctx.close()


if __name__ == "__main__":
    main()
