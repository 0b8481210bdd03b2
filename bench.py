#!/usr/bin/env python
"""bench.py - fp64 GMG V-cycle DOF/s (BASELINE.json metric) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config D|B|A|C|...] [--dump-outputs DIR]

A "step" is one V(1,1) cycle (GMG::Cycle::apply, zero initial guess) over the whole finest level.

`--dump-outputs DIR` (one GPU) writes the result u of the last timed step to DIR/u.npy (float64): all of it when it has at
most DUMP_MAX_VALUES cells, otherwise the cells at a fixed seeded sample of indices (sorted).  The right-hand side is a
function of the workload only, so two builds run with the same arguments can be compared output for output.

Workload at EVERY N (1, 2, 4, 8): BASELINE config D as named - the >= 1 B-cell 3D uniform octree, 4uni.bin --divide 2,
32,768 patches of 32^3 = 1,073,741,824 cells, 6 levels, trig manufactured right-hand side resident in HBM - so that the
driver's 1 -> 8 curve is a strong-scaling curve on one mesh.  The other BASELINE configs (A, B, C, E) and the same mesh
with 16^3 patches (D16) are measured in the same run and reported under `other_configs` (N = 1: child processes;
N = 8: config C at --divide 4 and the config E weak-scaling point, in process).

`--impl reference` times the reference's own CPU implementation of the path (oracle/_ref/ref_gmg: the unmodified
reference GMG sources on single-rank shims) on a bounded sample of the same workload and prints the same `config`.
One JSON line is printed by rank 0; DESIGN.md section 5 describes every key.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
MESHES = os.path.join(ROOT, "tests", "golden", "meshes")
GOLDEN = os.path.join(ROOT, "tests", "golden")
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "ref_gmg")
HEADLINE = "D"

# name -> D, mesh file, --divide, n, global finest-level cells, description
CONFIGS = {
    "A": (2, "2d2uni.bin", 6, 32, 16777216, "config A: apps/2d/steady2d GMG, uniform quadtree 2d2uni.bin --divide 6, 16384 patches of 32^2 (16,777,216 cells), 8 levels, trig RHS"),
    "B": (3, "4uni.bin", 1, 16, 16777216, "config B: apps/3d/steady GMG, uniform octree 4uni.bin --divide 1, 4096 patches of 16^3 (16,777,216 cells), 5 levels, trig RHS"),
    "C": (3, "2refine.bin", 3, 16, 31457280, "config C: apps/3d/steady GMG, refined octree 2refine.bin --divide 3, 7680 patches of 16^3 (31,457,280 cells), 6 levels, trig RHS"),
    "C4": (3, "2refine.bin", 4, 16, 251658240, "config C for 8 GPUs: refined octree 2refine.bin --divide 4, 61,440 patches of 16^3 (251,658,240 cells), 7 levels, trig RHS"),
    "D": (3, "4uni.bin", 2, 32, 1073741824, "config D: 3D uniform octree 4uni.bin --divide 2, 32,768 patches of 32^3 (1,073,741,824 cells), 6 levels, trig RHS"),
    "D16": (3, "4uni.bin", 3, 16, 1073741824, "config D's mesh with 16^3 patches: uniform octree 4uni.bin --divide 3, 262,144 patches of 16^3 (1,073,741,824 cells), 7 levels, trig RHS"),
    "D2": (3, "3uni.bin", 1, 32, 16777216, "3uni.bin --divide 1, 512 patches of 32^3 (16,777,216 cells), 4 levels, trig RHS"),
    "E": (2, "2d_multi_refine_8.bin", 4, 32, 41943040, "config E: apps/2d/steady2d GMG, deeply refined quadtree multi_refine_8.bin (tree levels 3-9) --divide 4, 40,960 patches of 32^2 (41,943,040 cells), 13 levels, trig RHS"),
    "E5": (2, "2d_multi_refine_8.bin", 5, 32, 167772160, "config E, one more --divide: 163,840 patches of 32^2 (167,772,160 cells), 14 levels, trig RHS"),
    "GMGEX": (3, "3d_multi_refine_8.bin", 2, 16, 73662464, "the reference's shipped GMG example (apps/3d/config/gmg_example.ini: Neumann boundaries, problem gauss, 16^3 patches, meshes/multi_refine_8.bin) --divide 2: 17,984 patches of 16^3 (73,662,464 cells), 11 levels"),
    "small": (3, "3uni.bin", 1, 16, 2097152, "3uni.bin --divide 1, 512 patches of 16^3 (2,097,152 cells), 4 levels, trig RHS"),
    "small32": (3, "3uni.bin", 0, 32, 2097152, "3uni.bin, 64 patches of 32^3 (2,097,152 cells), 3 levels, trig RHS"),
}
# config E weak scaling: the mesh family grows by a factor 4 per --divide, so the 1- and 4-GPU points are an exact weak pair
# (41.9 M cells per GPU); the 2- and 8-GPU points run the same two meshes at half the cells per GPU (a 2:1-balanced mesh with
# twice the cells does not exist in this family).  cells_per_gpu and DOF/s per GPU are reported with every point.
E_WEAK = {1: ("E", None), 2: ("E", None), 4: ("E5", None), 8: ("E5", None)}
# workloads with Neumann conditions on the whole domain boundary: name -> manufactured problem (apps/3d/steady.cpp:230-282)
NEUMANN = {"GMGEX": "gauss"}
ALGO_BYTES_PER_CELL_VISIT = 48.0  # SURVEY 8(d): pre-smooth 16 + residual/restrict 16 + post-smooth 16
CYCLE = "V(1,1), 1 coarse sweep, all levels down to the root patch"
DUMP_MAX_VALUES = 1 << 22  # 32 MB of float64
DUMP_SEED = 0
DFT_CAVEAT = ("patch solver = the reference's first-party DftPatchSolver (dense n x n transform matrices through a naive dgemv_ shim): "
              "O(n) work per cell per axis, i.e. slower than the FftwPatchSolver path with a real FFTW, which is not installed here")


def config_block(cfg, n_gpus):
    """identical in both arms (the driver compares them): a function of the workload name and N only"""
    D, mesh, div, n, cells, desc = CONFIGS[cfg]
    return {"workload": desc, "cycle": CYCLE, "cells": cells,
            "l2": "inputs larger than L2 (f and u are %.0f MB each over all GPUs, L2 is 126 MB per GPU)" % (cells * 8 / 1e6),
            "parallelism": "1 GPU" if n_gpus == 1 else "%d GPUs: patches split along a Morton curve, peer-to-peer halo-face exchange over NVLink, strong scaling on the mesh of N = 1" % n_gpus}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(cfg):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed ncu --set full
    capture (profiles/ncu_traffic.json, written by hand from the summaries next to it)"""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(p):
        t = json.load(open(p)).get(cfg)
        if t:
            return t.get("bytes_per_launch"), t.get("source")
    return None, None


class ClockSampler(threading.Thread):
    """samples nvidia-smi clocks / throttle reasons while the timed region runs"""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.rows = index, False, []

    def run(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


# ------------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference's own code on the host cores
# ------------------------------------------------------------------------------------------------------------
def cpu_sample_for(cfg):
    """bounded sample of a workload for the CPU runs: the same mesh family, patch size and cycle, cut down to 2.1 M cells
    (a 1/512 sub-cube of config D; per-DOF cost of the reference is size-independent to ~5 %, measured 3.56e6 DOF/s at 2.1 M
    cells vs 3.42e6 at 16.8 M cells in the build container)"""
    D, mesh, div, n, cells, desc = CONFIGS[cfg]
    if D == 3 and n == 32:
        return "small32"
    if D == 3:
        return "small"
    return cfg


def cpu_reference_run(cfg_name, reps, warmup, replicas):
    """times the reference's own CPU implementation (oracle/_ref/ref_gmg) of one V-cycle; `replicas` concurrent single-rank
    processes stand in for the MPI ranks the reference would use (no MPI runtime here): an optimistic, comm-free bound."""
    D, mesh, div, n, cells, desc = CONFIGS[cfg_name]
    cmd = [REF_BIN, str(D), os.path.join(MESHES, mesh), str(div), str(n), "dft", "time:%d:%d" % (reps, warmup)]
    t0 = time.time()
    procs = [subprocess.Popen(cmd, stdout=subprocess.PIPE, text=True) for _ in range(replicas)]
    outs = [json.loads(p.communicate()[0].strip().splitlines()[-1]) for p in procs]
    wall = time.time() - t0
    sec = max(o["sec_per_vcycle_median"] for o in outs)
    return {"cells_per_replica": outs[0]["cells"], "replicas": replicas, "sec_per_vcycle": sec,
            "dof_per_s": replicas * outs[0]["cells"] / sec, "wall_s": wall, "desc": desc}


def run_reference_arm(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    if not os.path.exists(REF_BIN):
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/ref_gmg not built (run `make -C oracle ref` where /root/reference exists)"}))
        return
    cores = os.cpu_count() or 1
    sample_cfg = cpu_sample_for(args.config)
    steps, warm = max(1, args.steps), max(1, args.warmup)
    res = cpu_reference_run(sample_cfg, steps, warm, cores)
    sample = ("bounded sample of the workload: %d concurrent single-rank replicas (one per host core, standing in for the MPI ranks of the "
              "reference; no communication cost, an optimistic bound) of the reference's own Cycle::apply (oracle/_ref/ref_gmg = unmodified "
              "reference sources on single-rank shims), each on %s - same mesh family, patch size and cycle as the workload, which itself "
              "(8.6 GB per vector x ~12 vectors) does not fit the host; median of %d cycles after %d warm-ups; %s"
              % (cores, res["desc"], steps, warm, DFT_CAVEAT))
    line = {"impl": "reference", "metric": "fp64 GMG V-cycle DOF/s", "value": res["dof_per_s"], "unit": "DOF/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["sec_per_vcycle"] * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_block(args.config, args.gpus),
            "cpu_baseline": {"value": res["dof_per_s"], "unit": "DOF/s", "cores": cores, "kind": "reference", "sample": sample},
            "e2e": {"value": res["dof_per_s"], "unit": "DOF/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": res["wall_s"]}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------------
class Env:
    """process-wide plumbing: context, torch.distributed (gloo) for id broadcast / barriers / max-over-ranks"""

    def __init__(self):
        import pressurepoissonsolver_b200 as pps
        self.pps = pps
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.dist = None
        self.ctx = pps.Context(self.local_rank)
        if self.world > 1:
            # torch.distributed (gloo) is plumbing only: NCCL id broadcast, barrier, max-over-ranks of the device time.
            # The data path (halo faces, coarse right-hand side, norms) goes through the library's own communicator.
            import torch.distributed as dist
            self.dist = dist
            dist.init_process_group("gloo")
            ids = [pps.comm_unique_id() if self.rank == 0 else None]
            dist.broadcast_object_list(ids, src=0)
            self.ctx.comm_init(ids[0], self.rank, self.world)

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()

    def reduce_max(self, *vals):
        if self.dist is None:
            return list(vals)
        import torch
        t = torch.tensor(list(vals), dtype=torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t]

    def reduce_sum(self, *vals):
        if self.dist is None:
            return list(vals)
        import torch
        t = torch.tensor(list(vals), dtype=torch.float64)
        self.dist.all_reduce(t)
        return [float(x) for x in t]


def build_hierarchy(env, cfg, box_frac=None, distributed=True):
    """mesh ingest + partition + device tables; returns (hierarchy, mesh, partition or None, set-up seconds)"""
    pps = env.pps
    D, mesh_file, divide, n, _, _ = CONFIGS[cfg]
    t0 = time.perf_counter()
    mesh = pps.Mesh.load(os.path.join(MESHES, mesh_file), D).refine_leaves(divide)
    if cfg in NEUMANN:
        mesh.set_neumann(True)
    if box_frac is not None:
        mesh.refine_box((0.0, 0.0, 0.0), (box_frac, 1.0, 1.0))
    part = None
    if env.world > 1 and distributed:
        # levels with fewer than ~256 patches in total (32 per rank at 8 GPUs) are cheaper to replicate than to exchange
        # halos for (measured at 8 GPUs on D16: 1.82 ms per cycle with this threshold, 1.96 ms with 2048); the threshold
        # is in cells: a 32^3 patch counts for eight 16^3 patches
        mpr = int(os.environ.get("BENCH_MIN_PATCHES_PER_RANK", max(32, 256 // env.world)))
        if n > 16:
            mpr = max(4, mpr * 16 ** D // n ** D)
        part = pps.Partition(mesh, n, env.rank, env.world, min_patches_per_rank=mpr)
        h = pps.Hierarchy.from_partition(env.ctx, part)
    else:
        h = pps.Hierarchy.from_mesh(env.ctx, mesh, n)
    env.ctx.sync()
    return h, mesh, part, time.perf_counter() - t0


def time_cycles(env, h, f, u, opts, steps, warmup):
    """W untimed cycles, then K cycles between CUDA events on the library's stream, barrier + sync on both sides, max over ranks"""
    ctx = env.ctx
    for _ in range(warmup):
        h.vcycle(f, u, opts)
    ctx.sync()
    env.barrier()
    l0 = ctx.kernel_launches()
    ctx.timer_start()
    for _ in range(steps):
        h.vcycle(f, u, opts)
    ms = ctx.timer_stop()
    launches = ctx.kernel_launches() - l0
    env.barrier()
    return env.reduce_max(ms)[0] / steps, launches, ms / steps


def dump_outputs(out_dir, u):
    """u of the last timed step -> out_dir/u.npy (see the module docstring)"""
    import numpy as np
    a = u.download()
    if a.size > DUMP_MAX_VALUES:
        a = a[np.sort(np.random.default_rng(DUMP_SEED).choice(a.size, DUMP_MAX_VALUES, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "u.npy"), a)


def kernel_profile(env, h, f, u, opts, steps):
    """the same steps again with CUDA events around every launch (graph replay bypassed)"""
    env.ctx.profile_begin()
    for _ in range(steps):
        h.vcycle(f, u, opts)
    agg = {}
    for name, lvl, kms in env.ctx.profile_end():
        a = agg.setdefault((name, lvl), [0, 0.0])
        a[0] += 1
        a[1] += kms
    return agg


def smoother_kernel_name(D, n):
    if D == 3 and n == 16:
        return "smooth3d16_kernel"
    if D == 3 and n == 32:
        return "smooth3d32c_kernel (one 2-CTA cluster per patch)"
    if D == 2 and n == 32:
        return "smooth2d32_kernel (one warp per patch)"
    return "smooth_kernel<%d, %d>" % (D, n)


def roofline_block(cfg, D, n, cells, level_cells, agg, ms_per_step, steps):
    """dominant kernel = the block-Jacobi patch-solve smoother on the finest level.  Its two instantiations are credited
    with their own compulsory bytes: the sweep from a zero guess that only emits faces reads f (8 B/cell) and writes the
    2D boundary slices (8 * 2D / n B/cell); the post-smoothing sweep reads f and writes u (16 B/cell; the face and coarse
    values it gathers are not counted)."""
    peak, peak_src = measured_peaks()
    per = {}
    pre_b = (8.0 + 8.0 * 2 * D / n) * cells
    post_b = 16.0 * cells
    for (name, lvl), (cnt, tot) in agg.items():
        if lvl != 0 or not name.startswith("smooth"):
            continue
        b = pre_b if name == "smooth_zero_guess_faces" else post_b
        per[name] = {"launches_per_step": cnt / steps, "ms_per_launch": tot / cnt, "algorithmic_bytes_per_launch": b,
                     "achieved_gbs": b / (tot / cnt * 1e-3) / 1e9, "frac": b / (tot / cnt * 1e-3) / 1e9 / peak}
    tot_ms = sum(v["ms_per_launch"] * v["launches_per_step"] for v in per.values())
    tot_b = sum(v["algorithmic_bytes_per_launch"] * v["launches_per_step"] for v in per.values())
    nl = sum(v["launches_per_step"] for v in per.values())
    achieved = tot_b / (tot_ms * 1e-3) / 1e9 if tot_ms else None
    prof_total = sum(v[1] for v in agg.values())
    share = sum(v[1] for (name, lvl), v in agg.items() if name.startswith("smooth")) / prof_total if prof_total else None
    cycle_bytes = ALGO_BYTES_PER_CELL_VISIT * sum(level_cells)
    cycle_gbs = cycle_bytes / (ms_per_step * 1e-3) / 1e9
    traffic, traffic_src = ncu_traffic(cfg)
    return {"bound": "hbm", "kernel": smoother_kernel_name(D, n) + ": block-Jacobi patch-solve smoother, all its launches on the finest level of one step (rank 0)",
            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None,
            "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
            "ms_per_launch": tot_ms / nl if nl else None, "algorithmic_bytes_per_launch": tot_b / nl if nl else None,
            "per_instantiation": per, "share_of_step": share,
            "vcycle_algorithmic_gbs": cycle_gbs, "vcycle_frac": cycle_gbs / peak, "vcycle_bytes_per_dof": cycle_bytes / cells,
            # SURVEY 8(d): also against B200's nominal 8 TB/s, and the traffic of the unfused call-by-call sequence the
            # reference executes (104 B per cell per level visit instead of the compulsory 48) moved in the same time
            "vcycle_frac_of_nominal_8000_gbs": cycle_gbs / 8000.0,
            "vcycle_gbs_if_unfused_104_bytes_per_cell_visit": cycle_gbs * 104.0 / ALGO_BYTES_PER_CELL_VISIT}


def time_to_solution(env, h, f, opts, total_cells):
    """time to 1e-10 relative residual (north star): BiCGStab with the V-cycle as right preconditioner
    (apps/3d/steady.cpp:522, BiCGStab.h:45-106) and the stationary iteration u += V(f - A u), both from u = 0"""
    ctx = env.ctx
    x = h.new_vec(0)
    h.bicgstab(f, x, opts, tol=1e-10, max_it=100)  # warm-up (graph capture for the Krylov work vectors)
    x.set(0.0)
    ctx.sync()
    env.barrier()
    t0 = time.perf_counter()
    its, rel = h.bicgstab(f, x, opts, tol=1e-10, max_it=100)
    ctx.sync()
    bicg_ms = (time.perf_counter() - t0) * 1e3
    h.trim()  # the Krylov work vectors (8 x the size of f) go back to the device before the next phase
    r, e = h.new_vec(0), h.new_vec(0)
    fnorm = f.two_norm()
    x.set(0.0)
    ctx.sync()
    env.barrier()
    t0 = time.perf_counter()
    ncyc, srel = 0, 1.0
    while srel > 1e-10 and ncyc < 100:
        h.residual(0, f, x, r)
        srel = r.two_norm() / fnorm
        if srel <= 1e-10:
            break
        h.vcycle(r, e, opts)
        x.add(e)
        ncyc += 1
    ctx.sync()
    stat_ms = (time.perf_counter() - t0) * 1e3
    for v in (x, r, e):
        v.close()
    h.trim()
    bicg_ms, stat_ms = env.reduce_max(bicg_ms, stat_ms)
    return {"tolerance": 1e-10, "bicgstab_ms": bicg_ms, "bicgstab_iterations": its, "bicgstab_rel_residual": rel,
            "stationary_ms": stat_ms, "stationary_cycles": ncyc, "stationary_rel_residual": srel,
            "note": "wall clock around the C-ABI calls, u = 0 start, includes the norm/dot host round trips"}


def e2e_block(env, h, f, u, opts, steps, cells, total_cells):
    """host buffers through the C-ABI.  Every step copies its own right-hand side from pinned host memory to the device and
    its result back (both inside the timed region).  The steps are independent right-hand sides, so the library's pipelined
    entry point is used: upload of step k + 1, cycle k and download of step k - 1 overlap (PCIe is full duplex); the serial,
    one-call-at-a-time form (tgpu_vcycle_host) is reported next to it, and so is the box's copy ceiling: the same bytes moved
    both ways with no cycle in between."""
    import numpy as np
    pps, ctx = env.pps, env.ctx
    big = cells * 8 > (1 << 30)
    # one input buffer serves both slots when a vector exceeds 1 GB per rank (the right-hand sides are equal anyway)
    fps = [pps.PinnedBuffer(cells)]
    fps.append(fps[0] if big else pps.PinnedBuffer(cells))
    ups = [pps.PinnedBuffer(cells) for _ in range(2)]
    fh = f.download()
    for b_ in (fps[:1] if big else fps):
        b_.array[:] = fh
    del fh
    n_e2e = max(3, min(steps, 10)) if not big else 3
    for k in range(2):
        h.vcycle_host(fps[k], ups[k], opts)
    env.barrier()
    t0 = time.perf_counter()
    for k in range(n_e2e):
        h.vcycle_host(fps[k & 1], ups[k & 1], opts)
    serial_ms = (time.perf_counter() - t0) * 1e3 / n_e2e
    h.trim()
    for k in range(4):
        h.vcycle_host_async(fps[k & 1], ups[k & 1], opts)
    h.vcycle_host_wait()
    env.barrier()
    n_pipe = 2 * n_e2e
    t0 = time.perf_counter()
    for k in range(n_pipe):
        h.vcycle_host_async(fps[k & 1], ups[k & 1], opts)
    h.vcycle_host_wait()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / n_pipe
    u_ref = u.download()
    same = bool(np.array_equal(ups[0].array, u_ref) and np.array_equal(ups[1].array, u_ref))  # same f, same cycle, bit for bit
    del u_ref
    # copy ceiling: H2D of f and D2H of u concurrently on two streams, nothing else (all ranks at once)
    tin, tout = h.new_vec(0), h.new_vec(0)
    ctx.sync()
    env.barrier()
    t0 = time.perf_counter()
    for k in range(n_e2e):
        h.copy_pair(tin, fps[0], tout, ups[0])
    copy_ms = (time.perf_counter() - t0) * 1e3 / n_e2e
    tin.close()
    tout.close()
    h.trim()
    for b_ in set(fps) | set(ups):
        b_.close()
    e2e_ms, serial_ms, copy_ms = env.reduce_max(e2e_ms, serial_ms, copy_ms)
    assert same, "e2e result differs from the device-resident cycle"
    # bytes of the whole job per step, like `value` (every rank copies its own patches' share: cells * 8 each way)
    return {"value": total_cells / (e2e_ms * 1e-3), "unit": "DOF/s", "h2d_bytes_per_step": total_cells * 8, "d2h_bytes_per_step": total_cells * 8,
            "h2d_bytes_per_step_rank0": cells * 8, "d2h_bytes_per_step_rank0": cells * 8,
            "ms_per_step": e2e_ms, "steps": n_pipe,
            "api": "tgpu_vcycle_host_async + tgpu_vcycle_host_wait (per step: pinned host f -> device, V-cycle, u -> pinned host; consecutive steps pipelined over copy-in / compute / copy-out streams)",
            "serial_ms_per_step": serial_ms, "serial_value": total_cells / (serial_ms * 1e-3), "serial_api": "tgpu_vcycle_host (one blocking call per step)",
            "copy_only_ms_per_step": copy_ms,
            "copy_only_note": "the step's host->device and device->host copies alone, both directions concurrently, all ranks at once: the PCIe ceiling of this box for the e2e figure (%.1f GB/s per direction per GPU)" % (cells * 8 / (copy_ms * 1e-3) / 1e9),
            "bit_identical_to_device_resident_cycle": same}


def nvlink_block(env, part, D, n, ms_per_step):
    """bytes every rank stores into its peers' face buffers per V(1,1) cycle (two hand-overs per distributed level: the
    faces of the pre-smoothed u, then faces + prolonged correction), max over ranks, against NVLink 5's nominal 900 GB/s
    per direction per GPU (north star: fraction of the NVLink roofline where sharded)"""
    M = n ** (D - 1)
    faces = [sum(len(p["send_patch"]) for p in part.level(l)["peers"]) for l in range(part.ndist)]
    sent = float(sum(faces) * M * 8 * 2)
    sent_max, = env.reduce_max(sent)
    gbs = sent_max / (ms_per_step * 1e-3) / 1e9
    return {"bytes_sent_per_rank_per_cycle": sent_max, "faces_sent_per_level_rank0": faces, "achieved_gbs_per_rank": gbs, "peak_gbs": 900.0,
            "frac": gbs / 900.0, "note": "halo faces only; the exchange is latency-bound (two hand-overs per level visit), not bandwidth-bound"}


def multi_gpu_parity(env):
    """driver-run numerical evidence for the N > 1 path, outside every timed region: distributed V-cycles against the
    reference's golden vectors (tests/golden/*.npz, produced by the reference's own code) and, for the specialised 16^3 /
    32^3 kernels, against the single-GPU path of the same library (itself pinned to the oracle by tests/ -m gpu)."""
    import numpy as np
    pps = env.pps
    out = {}

    def rel(u_loc, ref_loc):
        e2, r2 = env.reduce_sum(float(np.sum((u_loc - ref_loc) ** 2)), float(np.sum(ref_loc ** 2)))
        return (e2 / r2) ** 0.5

    for name in ("3d_2refine_n8", "3d_2refine_d1_n4", "2d_multi_refine_8_n4"):
        g = np.load(os.path.join(GOLDEN, name + ".npz"))
        D, n = int(g["D"]), int(g["n"])
        mesh = pps.Mesh.load(os.path.join(MESHES, str(g["mesh"])), D).refine_leaves(int(g["divide"]))
        part = pps.Partition(mesh, n, env.rank, env.world, min_patches_per_rank=1)
        h = pps.Hierarchy.from_partition(env.ctx, part)
        own = part.level(0)["owned_global"]
        fg, ug = g["rhs_f"].reshape(-1, n ** D), g["vcycle"].reshape(-1, n ** D)
        f, u = h.new_vec(0, fg[own]), h.new_vec(0)
        h.vcycle(f, u, pps.CycleOpts.default(use_graph=2))
        h.vcycle(f, u, pps.CycleOpts.default(use_graph=2))  # replayed graph incl. the exchanges
        out["golden_" + name] = {"rel_l2": rel(u.download().reshape(-1, n ** D), ug[own]), "distributed_levels": part.ndist}
        h.close()
        part.close()
        mesh.close()
    for D, n, mesh_file, divide in ((3, 16, "2refine.bin", 1), (3, 32, "2refine.bin", 1), (2, 32, "2d_multi_refine_8.bin", 1)):
        mesh = pps.Mesh.load(os.path.join(MESHES, mesh_file), D).refine_leaves(divide)
        h1 = pps.Hierarchy.from_mesh(env.ctx, mesh, n)  # the whole mesh on this GPU
        f1, u1 = h1.new_vec(0), h1.new_vec(0)
        h1.init_trig_rhs(f1)
        h1.vcycle(f1, u1)
        ref = u1.download().reshape(-1, n ** D)
        fg = f1.download().reshape(-1, n ** D)
        h1.close()
        part = pps.Partition(mesh, n, env.rank, env.world, min_patches_per_rank=2)
        h = pps.Hierarchy.from_partition(env.ctx, part)
        own = part.level(0)["owned_global"]
        f, u = h.new_vec(0, fg[own]), h.new_vec(0)
        h.vcycle(f, u, pps.CycleOpts.default(use_graph=2))
        h.vcycle(f, u, pps.CycleOpts.default(use_graph=2))  # replayed graph
        out["vs_single_gpu_%dd_n%d" % (D, n)] = {"rel_l2": rel(u.download().reshape(-1, n ** D), ref[own]), "distributed_levels": part.ndist}
        h.close()
        part.close()
        mesh.close()
    out["max_rel_l2"] = max(v["rel_l2"] for v in out.values())
    out["tolerance"] = 1e-12
    out["ok"] = bool(out["max_rel_l2"] < 1e-12)
    return out


def measure_config(env, cfg, steps, warmup, box_frac=None, profile=True, dump_dir=None):
    """device-resident cycle timing of one workload -> dict (value, ms_per_step, roofline, ...); with dump_dir, the timed
    steps' result is written there before anything else runs on u"""
    pps = env.pps
    D, mesh_file, divide, n, _, desc = CONFIGS[cfg]
    h, mesh, part, setup_s = build_hierarchy(env, cfg, box_frac)
    cells = h.ncells(0)
    level_cells = [h.ncells(l) for l in range(h.nlevels)]
    f, u = h.new_vec(0), h.new_vec(0)
    if cfg in NEUMANN:  # Init::initNeumann + the mean removal of apps/3d/steady.cpp:330-334
        h.init_neumann_rhs(f, None, NEUMANN[cfg])
        integral, volume = h.integrate(f)
        f.shift(-integral / volume)
    else:
        h.init_trig_rhs(f)
    opts = pps.CycleOpts.default()
    if env.world > 1:
        opts.use_graph = 2  # capture the halo exchanges into the CUDA graph as well
    ms_per_step, launches, my_ms = time_cycles(env, h, f, u, opts, steps, warmup)
    if dump_dir is not None:
        dump_outputs(dump_dir, u)
    total_cells = int(env.reduce_sum(cells)[0])
    res = {"workload": desc if box_frac is None else desc + "; leaves with centre x < %.2f refined once more" % box_frac,
           "n_gpus": env.world, "value": total_cells / (ms_per_step * 1e-3), "unit": "DOF/s", "ms_per_step": ms_per_step,
           "steps": steps, "cells": total_cells, "cells_rank0": cells, "setup_s": setup_s, "gpu_launches": launches}
    if profile:
        agg = kernel_profile(env, h, f, u, opts, steps)
        # roofline of the whole cycle from rank 0's share: rank-0 level cells over the max-over-ranks step time
        res["roofline"] = roofline_block(cfg, D, n, cells, level_cells, agg, ms_per_step, steps)
        res["kernel_profile_ms_per_step"] = {"%s@L%d" % k: round(v[1] / steps, 5) for k, v in sorted(agg.items(), key=lambda kv: -kv[1][1])}
    res["level_cells_rank0"] = level_cells
    return res, (h, mesh, part, f, u, opts, cells, total_cells, level_cells)


def close_all(state):
    h, mesh, part, f, u = state[:5]
    f.close()
    u.close()
    h.close()
    if part is not None:
        part.close()
    mesh.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--config", default=os.environ.get("BENCH_CONFIG", HEADLINE))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cycle-only", action="store_true", help="only the device-resident V-cycle timing and its roofline")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the other BASELINE configs")
    ap.add_argument("--with-solve", action="store_true", help="with --cycle-only: also the time to 1e-10 residual")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's result to DIR/u.npy (one GPU, not with --impl reference)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs works on one GPU and not with --impl reference")
    if args.impl == "reference":
        return run_reference_arm(args)

    t_start = time.time()
    env = Env()
    cfg = args.config
    D, mesh_file, divide, n, _, desc = CONFIGS[cfg]
    W = max(args.warmup, 3)
    sampler = ClockSampler(env.local_rank)
    sampler.start()
    res, state = measure_config(env, cfg, args.steps, W, dump_dir=args.dump_outputs)
    sampler.stop_flag = True
    sampler.join()
    h, mesh, part, f, u, opts, cells, total_cells, level_cells = state

    line = {
        "metric": "fp64 GMG V-cycle DOF/s", "value": res["value"], "unit": "DOF/s", "n_gpus": env.world, "steps": args.steps, "warmup": W,
        "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": config_block(cfg, env.world),
        "roofline": res["roofline"], "gpu_launches": res["gpu_launches"], "clocks": sampler.summary(),
        "setup_s": res["setup_s"], "cells_rank0": cells, "level_cells_rank0": level_cells,
        "kernel_profile_ms_per_step": res["kernel_profile_ms_per_step"],
    }
    if env.world > 1 and part is not None:
        line["nvlink"] = nvlink_block(env, part, D, n, res["ms_per_step"])
    if not args.cycle_only:
        line["time_to_solution"] = time_to_solution(env, h, f, opts, total_cells)
        line["e2e"] = e2e_block(env, h, f, u, opts, args.steps, cells, total_cells)
    else:
        line["e2e"] = None
        if args.with_solve:
            line["time_to_solution"] = time_to_solution(env, h, f, opts, total_cells)
    close_all(state)

    if env.world > 1 and not args.cycle_only:
        line["multi_gpu_parity"] = multi_gpu_parity(env)
    if env.world > 1 and not args.cycle_only and not args.no_other_configs:
        # BASELINE configs whose stated GPU count is > 1, in process on the same communicator
        others = {}
        extra = [("D16", None)]
        if env.world == 8:
            extra.append(("C4", None))
        ecfg, efrac = E_WEAK.get(env.world, (None, None))
        if ecfg:
            extra.append((ecfg, efrac))
        for name, frac in extra:
            try:
                r, st = measure_config(env, name, max(5, args.steps // 2), 3, box_frac=frac)
                close_all(st)
                key = name if frac is None and not name.startswith("E") else "E_weak"
                others[key] = {k: r[k] for k in ("workload", "n_gpus", "value", "unit", "ms_per_step", "steps", "cells", "setup_s")}
                others[key]["vcycle_frac_of_hbm_roofline_rank0"] = r["roofline"]["vcycle_frac"]
                if key == "E_weak":
                    others[key]["cells_per_gpu"] = r["cells"] / env.world
                    others[key]["dof_per_s_per_gpu"] = r["value"] / env.world
            except Exception as ex:  # never let an extra line break the contract line
                others[name] = {"error": str(ex)[:300]}
        line["other_configs"] = others

    if env.rank == 0 and env.world == 1 and not args.no_cpu_baseline and os.path.exists(REF_BIN):
        sample_cfg = cpu_sample_for(cfg)
        r = cpu_reference_run(sample_cfg, 5, 1, 1)
        line["cpu_baseline"] = {"value": r["dof_per_s"], "unit": "DOF/s", "cores": 1, "kind": "reference",
                                "sample": "the reference's own Cycle::apply (oracle/_ref/ref_gmg, 1 rank = 1 core) on a bounded sample of the workload: "
                                          + r["desc"] + "; median of 5 cycles after 1 warm-up; " + DFT_CAVEAT}
    if env.rank == 0 and env.world == 1 and not args.cycle_only and not args.no_other_configs:
        # the other BASELINE configs (and config D's mesh with 16^3 patches), each in a child process with the same kernels
        others = {}
        for name in ("B", "A", "C", "E", "D16", "D2", "GMGEX"):
            try:
                out = subprocess.run([sys.executable, os.path.abspath(__file__), "--config", name, "--cycle-only", "--steps", "10", "--warmup", "3",
                                      "--no-cpu-baseline"] + (["--with-solve"] if name in ("B", "GMGEX") else []), capture_output=True, text=True, timeout=900).stdout
                o = json.loads([l for l in out.splitlines() if l.startswith("{")][-1])
                others[name] = {"workload": o["config"]["workload"], "n_gpus": 1, "value": o["value"], "unit": "DOF/s", "ms_per_step": o["ms_per_step"],
                                "steps": o["steps"], "cells": o["config"]["cells"], "setup_s": o["setup_s"],
                                "vcycle_frac_of_hbm_roofline": o["roofline"]["vcycle_frac"], "smoother_frac": o["roofline"]["frac"],
                                "smoother_per_instantiation": {k: round(v["frac"], 4) for k, v in o["roofline"]["per_instantiation"].items()}}
                if "time_to_solution" in o:
                    others[name]["time_to_solution"] = {k: o["time_to_solution"][k] for k in ("bicgstab_ms", "bicgstab_iterations", "stationary_ms", "stationary_cycles")}
            except Exception as ex:
                others[name] = {"error": str(ex)[:300]}
        line["other_configs"] = others
    line["wall_s"] = time.time() - t_start
    if env.rank == 0:
        print(json.dumps(line))
    if env.dist is not None:
        env.dist.barrier()
        env.dist.destroy_process_group()


if __name__ == "__main__":
    main()
