#!/usr/bin/env python
"""Stationary multigrid from an initial guess: Hierarchy.vcycle_update / gmg_solve against the hand-written loop
u += V(f - A u) (residual -> two_norm -> vcycle -> add), fp64, V(1,1) cycles, trig right-hand side.

    python tools/gmg_solve_bench.py [--configs B,D] [--reps 20] [--warmup 3] [--out FILE]
    torchrun --nproc_per_node N tools/gmg_solve_bench.py --configs D

Per config (bench.py's CONFIGS, same partition when run under torchrun):
  per_iteration  ms of one vcycle_update (rel. residual included) and of one loop step (residual + two_norm + vcycle + add),
                 alternated, CUDA events around each call (it ends in a host read), median over --reps after --warmup each
  from_zero      gmg_solve and the loop to 1e-10 relative to ||f|| from u = 0: cycles and wall ms
  warm_start     solve f, then f' = f + 1e-3 ||f|| g / ||g|| (g: one cycle applied to seeded white noise, a smooth field):
                 gmg_solve cycles and wall ms from the previous u and from zero
The card name, power limit and maximum SM clock come from a read-only nvidia-smi query.  Rank 0 prints one JSON line
(and writes it to --out)."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (CONFIGS, Env, build_hierarchy)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True, check=True).stdout.strip().splitlines()
    name, power, clock = [x.strip() for x in q[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock, "gpus_on_node": len(q)}


def loop_step(h, f, u, r, e, fnorm, opts):
    h.residual(0, f, u, r)
    rel = r.two_norm() / fnorm
    h.vcycle(r, e, opts)
    u.add(e)
    return rel


def loop_solve(h, f, u, r, e, opts, tol=1e-10, max_it=100):
    fnorm = f.two_norm()
    its = 0
    while True:
        h.residual(0, f, u, r)
        rel = r.two_norm() / fnorm
        if rel <= tol or its == max_it:
            return its, rel
        h.vcycle(r, e, opts)
        u.add(e)
        its += 1


def wall(env, fn):
    env.ctx.sync()
    env.barrier()
    t0 = time.perf_counter()
    out = fn()
    env.ctx.sync()
    return (time.perf_counter() - t0) * 1e3, out


def measure(env, cfg, reps, warmup):
    import numpy as np
    pps = env.pps
    h, mesh, part, setup_s = bench.build_hierarchy(env, cfg)
    opts = pps.CycleOpts.default()
    f, u, v, r, e = (h.new_vec(0) for _ in range(5))
    h.init_trig_rhs(f)
    fnorm = f.two_norm()
    # per iteration, alternating, both from the same iterate sequence's neighbourhood (u, v advance independently)
    for _ in range(warmup):
        h.vcycle_update(f, u, opts)
        loop_step(h, f, v, r, e, fnorm, opts)
    t_upd, t_loop = [], []
    for _ in range(reps):
        env.ctx.sync()
        env.barrier()
        env.ctx.timer_start()
        h.vcycle_update(f, u, opts)
        t_upd.append(env.reduce_max(env.ctx.timer_stop())[0])
        env.barrier()
        env.ctx.timer_start()
        loop_step(h, f, v, r, e, fnorm, opts)
        t_loop.append(env.reduce_max(env.ctx.timer_stop())[0])
    per_it = {"vcycle_update_ms": statistics.median(t_upd), "loop_step_ms": statistics.median(t_loop),
              "vcycle_update_ms_min_max": [min(t_upd), max(t_upd)], "loop_step_ms_min_max": [min(t_loop), max(t_loop)], "reps": reps}
    per_it["speedup"] = per_it["loop_step_ms"] / per_it["vcycle_update_ms"]
    # from zero (one short solve first: gmg_solve allocates its work vectors on the first call)
    h.gmg_solve(f, u, opts, tol=1e-10, max_it=1)
    u.set(0.0)
    ms_g, (its_g, rel_g) = wall(env, lambda: h.gmg_solve(f, u, opts, tol=1e-10, max_it=100))
    v.set(0.0)
    ms_l, (its_l, rel_l) = wall(env, lambda: loop_solve(h, f, v, r, e, opts))
    ms_g, ms_l = env.reduce_max(ms_g, ms_l)
    from_zero = {"gmg_solve": {"cycles": its_g, "ms": ms_g, "rel_residual": rel_g}, "loop": {"cycles": its_l, "ms": ms_l, "rel_residual": rel_l}}
    # warm start: u holds the solution of f
    noise = np.random.default_rng(1000 + env.rank).standard_normal(h.ncells(0))
    g, gs = h.new_vec(0, noise), h.new_vec(0)
    del noise
    h.vcycle(g, gs, opts)
    scale = 1e-3 * fnorm / gs.two_norm()
    g.copy(f)
    g.add_scaled(scale, gs)  # g = f' now
    ms_w, (its_w, rel_w) = wall(env, lambda: h.gmg_solve(g, u, opts, tol=1e-10, max_it=100))
    v.set(0.0)
    ms_z, (its_z, rel_z) = wall(env, lambda: h.gmg_solve(g, v, opts, tol=1e-10, max_it=100))
    ms_w, ms_z = env.reduce_max(ms_w, ms_z)
    warm = {"from_previous_u": {"cycles": its_w, "ms": ms_w, "rel_residual": rel_w}, "from_zero": {"cycles": its_z, "ms": ms_z, "rel_residual": rel_z}}
    for x in (f, u, v, r, e, g, gs):
        x.close()
    h.close()
    if part is not None:
        part.close()
    mesh.close()
    return {"workload": bench.CONFIGS[cfg][5], "setup_s": setup_s, "per_iteration": per_it, "from_zero": from_zero, "warm_start": warm}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="B,D")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    env = bench.Env()
    res = {"gpu": gpu_info() if env.rank == 0 else None, "gpus": env.world, "cycle": "V(1,1), fused schedule, CUDA graphs", "configs": {}}
    for cfg in args.configs.split(","):
        res["configs"][cfg] = measure(env, cfg, args.reps, args.warmup)
    if env.rank == 0:
        line = json.dumps(res)
        print(line)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as fh:
                fh.write(line + "\n")
    env.ctx.close()
    if env.dist is not None:
        env.dist.destroy_process_group()


if __name__ == "__main__":
    main()
