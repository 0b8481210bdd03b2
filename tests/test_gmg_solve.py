"""Stationary multigrid from an initial guess: tgpu_vcycle_update (u <- u + Cycle(f - A u), one fused cycle that starts
the finest level's pre-sweep from u's boundary slices) and tgpu_gmg_solve (cycles until ||f - A u|| <= tol ||f||, on
the residual norm evaluated from the boundary slices), against the oracle, the reference's own stationary iteration
(golden vhist) and the hand-written loop residual -> vcycle -> add."""
import os
import re
import subprocess
import sys
import tempfile

import numpy as np
import pytest

import gmg_oracle as go
from conftest import GOLDEN_CASES, MESHES, ROOT, load_golden, rel_l2

TOL = 1e-12


def cycle_from_guess(levels, f, u0, cycle_type="V", pre=1, post=1, mid=1, coarse_sweeps=1):
    """the oracle's go.cycle with the finest level started from u0 instead of zero (coarser levels from zero): the
    schedule the library runs when tgpu_vcycle_update starts from a guess"""
    def visit(l, fl, u):
        L = levels[l]
        if l == len(levels) - 1:
            for _ in range(coarse_sweeps):
                u = go.smooth(L, fl, u)
            return u

        def coarse_correction(u):
            fc = go.restrict(L, levels[l + 1], -1 * go.apply_op(L, u) + fl)
            return go.interpolate(L, levels[l + 1], visit(l + 1, fc, np.zeros(levels[l + 1].shape)), u)

        for _ in range(pre):
            u = go.smooth(L, fl, u)
        u = coarse_correction(u)
        if cycle_type == "W":
            for _ in range(mid):
                u = go.smooth(L, fl, u)
            u = coarse_correction(u)
        for _ in range(post):
            u = go.smooth(L, fl, u)
        return u

    return visit(0, f, np.array(u0, dtype=np.float64).reshape(levels[0].shape))


# ---- CPU ----
@pytest.mark.parametrize("mesh_file,D,n,divide", [("2d2ref.bin", 2, 8, 1), ("2refine.bin", 3, 4, 1)])
def test_cycle_from_a_guess_is_the_correction_of_the_residual(mesh_file, D, n, divide):
    """the smoother is linear, stationary and consistent, so one cycle from u0 is u0 + Cycle(f - A u0)"""
    levels = go.build_hierarchy(os.path.join(MESHES, mesh_file), D, n, divide)
    rng = np.random.default_rng(5)
    f, u0 = rng.standard_normal(levels[0].shape), rng.standard_normal(levels[0].shape)
    for kw in ({}, dict(pre=2, post=2), dict(cycle_type="W")):
        a = cycle_from_guess(levels, f, u0, **kw)
        b = u0 + go.cycle(levels, f - go.apply_op(levels[0], u0), **kw)
        assert rel_l2(a, b) < 1e-13, kw
    assert np.array_equal(cycle_from_guess(levels, f, np.zeros(levels[0].shape)), go.cycle(levels, f))


def test_app_builds_with_the_gmg_solver():
    import build_native
    build_native.build()
    app = build_native.build_app()
    assert os.path.exists(app)
    src = open(os.path.join(ROOT, "apps", "steady.cpp")).read()
    assert '"--solver"' in src and "GMGSolve<D>::solve" in src


# ---- GPU ----
def _pps():
    import pressurepoissonsolver_b200 as pps
    return pps


@pytest.fixture(scope="module")
def ctx():
    c = _pps().Context(0)
    yield c
    c.close()


def _build(ctx, mesh_file, D, n, divide=0, neumann=False):
    pps = _pps()
    mesh = pps.Mesh.load(os.path.join(MESHES, mesh_file), D)
    if neumann:
        mesh.set_neumann(True)
    mesh.refine_leaves(divide)
    return pps.Hierarchy.from_mesh(ctx, mesh, n), mesh


def _loop_update(h, f, u, opts=None):
    """the hand-written step u += V(f - A u): residual -> vcycle -> add"""
    r, e = h.new_vec(0), h.new_vec(0)
    h.residual(0, f, u, r)
    h.vcycle(r, e, opts)
    u.add(e)
    r.close()
    e.close()


def _smooth_field(h, seed):
    """a seeded smooth level-0 field: one cycle applied to white noise"""
    g, z = h.new_vec(0, np.random.default_rng(seed).standard_normal(h.ncells(0))), h.new_vec(0)
    h.vcycle(g, z)
    return z.download()


GUESS_OPTS = [dict(), dict(pre_sweeps=2, post_sweeps=2), dict(cycle_type=1), dict(max_levels=2), dict(fused=0), dict(fused=2),
              dict(use_graph=0), dict(pre_sweeps=2, post_sweeps=2, coarse_sweeps=2, use_graph=0), dict(interpolator=1),
              dict(post_sweeps=0, pre_sweeps=2)]
UPDATE_CASES = [("2d_multi_refine_8.bin", 2, 16, 0, False), ("2d2ref.bin", 2, 32, 1, False), ("2refine.bin", 3, 8, 1, False),
                ("multi_refine.bin", 3, 8, 0, False), ("2refine.bin", 3, 16, 0, False), ("2refine.bin", 3, 32, 0, False),
                ("2refine.bin", 3, 8, 0, True), ("2d2ref.bin", 2, 8, 1, True), ("2uni.bin", 3, 16, 0, True),  # NEUMANN_CASES
                ("3uni.bin", 3, 32, 0, True)]


def _oracle_kw(o):
    return dict(cycle_type="W" if o.get("cycle_type", 0) == 1 else "V", pre=o.get("pre_sweeps", 1), post=o.get("post_sweeps", 1),
                coarse_sweeps=o.get("coarse_sweeps", 1), max_levels=o.get("max_levels", 0),
                interp=go.interpolate_trilinear if o.get("interpolator", 0) == 1 else None)


def _check_update(h, levels, f, fn, u0, o, lam=0.0, replays=1, tol_oracle=TOL):
    pps = _pps()
    opts = pps.CycleOpts.default(**o)
    ref = u0 + go.cycle(levels, fn - go.apply_op(levels[0], u0), lam=lam, **_oracle_kw(o))
    u = h.new_vec(0, u0)
    own = h.new_vec(0, u0)
    _loop_update(h, f, own, opts)
    for _ in range(replays):
        u.upload(u0)
        h.vcycle_update(f, u, opts)
        assert rel_l2(u.download(), ref.ravel()) < tol_oracle, o
        assert rel_l2(u.download(), own.download()) < TOL, o


@pytest.mark.gpu
@pytest.mark.parametrize("mesh_file,D,n,divide,neumann", UPDATE_CASES)
def test_update_from_a_guess_vs_oracle(ctx, mesh_file, D, n, divide, neumann):
    h, mesh = _build(ctx, mesh_file, D, n, divide, neumann)
    levels = go.build_hierarchy(os.path.join(MESHES, mesh_file), D, n, divide, neumann=neumann)
    rng = np.random.default_rng(2024)
    fn, u0 = rng.standard_normal(levels[0].shape), rng.standard_normal(levels[0].shape)
    f = h.new_vec(0, fn)
    for o in GUESS_OPTS:
        _check_update(h, levels, f, fn, u0, o, replays=3 if o.get("use_graph", 1) else 1)
    h.close()
    mesh.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mesh_file,D,n,divide", [("2refine.bin", 3, 16, 0), ("2d2ref.bin", 2, 32, 1), ("2refine.bin", 3, 32, 0)])
def test_update_with_a_shifted_patch_solve_vs_oracle(ctx, mesh_file, D, n, divide):
    h, mesh = _build(ctx, mesh_file, D, n, divide)
    h.set_lambda(-0.75)
    levels = go.build_hierarchy(os.path.join(MESHES, mesh_file), D, n, divide)
    rng = np.random.default_rng(31)
    fn, u0 = rng.standard_normal(levels[0].shape), rng.standard_normal(levels[0].shape)
    f = h.new_vec(0, fn)
    for o in (dict(), dict(fused=2, use_graph=0), dict(pre_sweeps=2, post_sweeps=2)):
        _check_update(h, levels, f, fn, u0, o, lam=-0.75, replays=2, tol_oracle=1e-11)  # as the other shifted-solve tests
    h.close()
    mesh.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_solve_history_vs_reference(ctx, name):
    """the reference's own stationary iteration u += V(f - A u) (golden vhist / vhist_u, 6 cycles from zero)"""
    g = load_golden(name)
    h, mesh = _build(ctx, str(g["mesh"]), int(g["D"]), int(g["n"]), int(g["divide"]))
    f, u = h.new_vec(0, g["rhs_f"]), h.new_vec(0)
    its, rel, hist = h.gmg_solve(f, u, tol=0.0, max_it=6, history=True)
    assert its == 6 and len(hist) == 7 and rel == hist[-1]
    assert np.max(np.abs(np.array(hist) / g["vhist"] - 1)) < 1e-8
    assert rel_l2(u.download(), g["vhist_u"]) < 1e-10
    h.close()
    mesh.close()


FACE_NORM_CASES = [("2refine.bin", 3, 16, 0, False, 1), ("2refine.bin", 3, 16, 0, False, 2), ("2refine.bin", 3, 8, 1, False, 1),
                   ("2d2ref.bin", 2, 32, 1, False, 1), ("2d_multi_refine_8.bin", 2, 16, 0, False, 2), ("2refine.bin", 3, 32, 0, False, 1),
                   ("2refine.bin", 3, 32, 0, False, 2), ("2refine.bin", 3, 8, 1, True, 1), ("3uni.bin", 3, 32, 0, True, 1),
                   ("multi_refine.bin", 3, 4, 0, False, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("mesh_file,D,n,divide,neumann,post", FACE_NORM_CASES)
def test_face_residual_norm_vs_full_residual(ctx, mesh_file, D, n, divide, neumann, post):
    pps = _pps()
    h, mesh = _build(ctx, mesh_file, D, n, divide, neumann)
    rng = np.random.default_rng(8)
    fn = rng.standard_normal(h.ncells(0))
    if neumann:
        fn -= fn.mean()  # (mean-free only up to the cell volumes of refined meshes: the check does not need convergence)
    f, u, r = h.new_vec(0, fn), h.new_vec(0, rng.standard_normal(h.ncells(0))), h.new_vec(0)
    fnorm = f.two_norm()
    opts = pps.CycleOpts.default(post_sweeps=post, pre_sweeps=post)
    checked = 0
    for k in range(8):
        rel = h.vcycle_update(f, u, opts)
        h.residual(0, f, u, r)
        full = r.two_norm() / fnorm
        if full > 1e-12:
            assert abs(rel / full - 1) < 1e-10, (k, rel, full)
            checked += 1
    assert checked >= 4
    h.close()
    mesh.close()


# Neumann: the stationary iteration on the refined Neumann goldens stalls above 1e-10 (the singular system is compatible only
# up to rounding), the loop's as much as the library's; the uniform one converges
SOLVE_CASES = [("3d_2refine_n8", False), ("2d_2d2ref_d1_n8", False), ("3d_multi_refine_n4", False), ("3d_2uni_n16_neumann", True)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,neumann", SOLVE_CASES)
def test_solve_to_tolerance_and_warm_start(ctx, name, neumann):
    pps = _pps()
    g = load_golden(name)
    h, mesh = _build(ctx, str(g["mesh"]), int(g["D"]), int(g["n"]), int(g["divide"]), neumann)
    f = h.new_vec(0, g["rhs_f"])
    # the hand-written loop, with its own convergence test
    u_loop, r = h.new_vec(0), h.new_vec(0)
    fn = f.two_norm()
    loop_its = 0
    while True:
        h.residual(0, f, u_loop, r)
        if r.two_norm() / fn <= 1e-10 or loop_its == 100:
            break
        e = h.new_vec(0)
        h.vcycle(r, e)
        u_loop.add(e)
        e.close()
        loop_its += 1
    assert loop_its < 100
    u = h.new_vec(0)
    its, rel = h.gmg_solve(f, u, tol=1e-10, max_it=100)
    assert its == loop_its and rel <= 1e-10
    assert rel_l2(u.download(), u_loop.download()) < 1e-10
    h.residual(0, f, u, r)
    assert r.two_norm() / fn <= 1e-10
    # warm start: f' = f + 1e-3 g, from the previous solution and from zero
    gfield = _smooth_field(h, 17)
    gfield *= np.linalg.norm(g["rhs_f"]) / np.linalg.norm(gfield)
    fp = h.new_vec(0, g["rhs_f"] + 1e-3 * gfield)
    if neumann:  # keep f' compatible: remove the mean the perturbation added
        integral, volume = h.integrate(fp)
        fp.shift(-integral / volume)
    its_warm, rel_warm = h.gmg_solve(fp, u, tol=1e-10, max_it=100)
    z = h.new_vec(0)
    its_cold, rel_cold = h.gmg_solve(fp, z, tol=1e-10, max_it=100)
    assert rel_warm <= 1e-10 and rel_cold <= 1e-10
    assert its_warm < its_cold, (its_warm, its_cold)
    # the fallback schedule takes the same number of cycles to the same solution
    z.set(0.0)
    its_f, _ = h.gmg_solve(fp, z, pps.CycleOpts.default(fused=0), tol=1e-10, max_it=100)
    assert its_f == its_cold
    h.close()
    mesh.close()


@pytest.mark.gpu
def test_fused_update_does_no_full_passes(ctx):
    h, mesh = _build(ctx, "2refine.bin", 3, 16, 0)
    rng = np.random.default_rng(3)
    f, u = h.new_vec(0, rng.standard_normal(h.ncells(0))), h.new_vec(0, rng.standard_normal(h.ncells(0)))
    full = {"apply", "residual", "apply_dots", "blas1"}
    ctx.profile_begin()
    h.vcycle_update(f, u)
    prof = ctx.profile_end()
    names = [(k, l) for k, l, _ in prof]
    assert not [k for k, l in names if l == 0 and k in full], names
    assert ("face_residual_norm", 0) in names and ("extract_faces", 0) in names
    ctx.profile_begin()
    its, rel = h.gmg_solve(f, u, tol=1e-10, max_it=50)
    prof = ctx.profile_end()
    names = [(k, l) for k, l, _ in prof]
    # one full residual before the first cycle (the starting point's residual, history[0]) and one confirmation
    assert sum(1 for k, l in names if l == 0 and k == "residual") == 2, names
    assert not [k for k, l in names if l == 0 and k in full - {"residual"}], names
    assert sum(1 for k, l in names if k == "face_residual_norm") == 2 * its  # the norm kernel and its device-side reduction
    assert rel <= 1e-10
    h.close()
    mesh.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mesh_file,D,n,divide", [("4uni.bin", 3, 16, 1), ("4uni.bin", 3, 32, 0)])
def test_update_at_size(ctx, mesh_file, D, n, divide):
    """config B (4096 patches of 16^3) and 512 patches of 32^3: one update from a random guess against the library's own
    residual -> vcycle -> add, and the face norm against the full residual"""
    pps = _pps()
    h, mesh = _build(ctx, mesh_file, D, n, divide)
    assert h.npatch(0) == (4096 if n == 16 else 512)
    rng = np.random.default_rng(44)
    fn, u0 = rng.standard_normal(h.ncells(0)), rng.standard_normal(h.ncells(0))
    f, r = h.new_vec(0, fn), h.new_vec(0)
    for o in (dict(), dict(pre_sweeps=2, post_sweeps=2)):
        opts = pps.CycleOpts.default(**o)
        u, own = h.new_vec(0, u0), h.new_vec(0, u0)
        _loop_update(h, f, own, opts)
        rel = h.vcycle_update(f, u, opts)
        assert rel_l2(u.download(), own.download()) < TOL, o
        h.residual(0, f, u, r)
        assert abs(rel / (r.two_norm() / f.two_norm()) - 1) < 1e-10
        u.close()
        own.close()
    h.close()
    mesh.close()


@pytest.mark.gpu
def test_bad_arguments_leave_u_untouched(ctx):
    pps = _pps()
    h, mesh = _build(ctx, "2refine.bin", 3, 8, 0)
    h2, mesh2 = _build(ctx, "2refine.bin", 3, 8, 0)
    rng = np.random.default_rng(9)
    u0 = rng.standard_normal(h.ncells(0))
    f, u = h.new_vec(0, rng.standard_normal(h.ncells(0))), h.new_vec(0, u0)
    coarse, other = h.new_vec(1), h2.new_vec(0)
    calls = [lambda: h.vcycle_update(u, u), lambda: h.gmg_solve(u, u),
             lambda: h.vcycle_update(coarse, u), lambda: h.gmg_solve(f, coarse),
             lambda: h.vcycle_update(other, u), lambda: h.gmg_solve(f, other),
             lambda: h.gmg_solve(f, u, tol=-1.0), lambda: h.gmg_solve(f, u, max_it=-1),
             lambda: h.gmg_solve(f, u, tol=float("nan")),
             lambda: h.vcycle_update(f, u, pps.CycleOpts.default(pre_sweeps=-1))]
    for call in calls:
        with pytest.raises(pps.TgpuError):
            call()
        assert np.array_equal(u.download(), u0)
    h.close()
    h2.close()
    mesh.close()
    mesh2.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["3d_2refine_n8", "2d_2d2ref_d1_n8"])
def test_app_gmg_solver(name):
    """apps/steady --solver gmg: stationary solve to 1e-10 relative to f.  Both it and the BiCGStab solve approximate the
    same discrete solution x: ||u - x|| <= ||A^-1|| ||f - A u||, so ||u_gmg - u_bicg|| / ||u|| is bounded by
    cond(A) (rel_gmg + rel_bicg) ||f|| / (||A|| ||u||) <= cond(A) (rel_gmg + rel_bicg); the refined 8^3 / 8^2 meshes have
    cond(A) < 1e4 (h = 1/64), so with rel_gmg <= 1e-10 the two solutions agree to 1e-10 * 1e4 = 1e-6."""
    import build_native
    build_native.build()
    app = build_native.build_app()
    g = load_golden(name)
    with tempfile.TemporaryDirectory() as tmp:
        out = os.path.join(tmp, "u.bin")
        res = subprocess.run([app, str(int(g["D"])), os.path.join(MESHES, str(g["mesh"])), str(int(g["divide"])), str(int(g["n"])),
                              "--solver", "gmg", "--out", out], capture_output=True, text=True, check=True)
        resid = float(re.search(r"Residual: (\S+)", res.stdout).group(1))
        assert resid <= 1e-10
        assert int(re.search(r"Iterations: (\d+)", res.stdout).group(1)) > 0
        assert rel_l2(np.fromfile(out), g["bicgstab_u"]) < 1e-6


# ---- several GPUs (launcher pattern of test_multi_gpu.py) ----
def _ngpu():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


def _worker(rank, world, idfile, mesh_file, D, n, divide, f_global, ret, neumann):
    sys.path.insert(0, ROOT)
    import time
    import pressurepoissonsolver_b200 as pps
    ctx = pps.Context(rank)
    if rank == 0:
        uid = pps.comm_unique_id()
        with open(idfile + ".tmp", "wb") as fh:
            fh.write(uid)
        os.rename(idfile + ".tmp", idfile)
    else:
        while not os.path.exists(idfile):
            time.sleep(0.05)
        uid = open(idfile, "rb").read()
    ctx.comm_init(uid, rank, world)
    mesh = pps.Mesh.load(os.path.join(MESHES, mesh_file), D)
    if neumann:
        mesh.set_neumann(True)
    mesh.refine_leaves(divide)
    part = pps.Partition(mesh, n, rank, world, min_patches_per_rank=2)
    h = pps.Hierarchy.from_partition(ctx, part)
    pl = part.level(0)
    nc = n ** D
    fg = np.asarray(f_global).reshape(-1, nc)
    f, u = h.new_vec(0, fg[pl["owned_global"]]), h.new_vec(0)
    its, rel = h.gmg_solve(f, u, tol=1e-10, max_it=100)
    ret[rank] = {"owned": pl["owned_global"], "ndist": part.ndist, "its": its, "rel": rel, "u": u.download().reshape(-1, nc)}
    h.close()
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mesh_file,D,n,divide,neumann", [("2refine.bin", 3, 16, 1, False), ("3uni.bin", 3, 16, 1, True)])
def test_distributed_solve_matches_single_gpu(ctx, mesh_file, D, n, divide, neumann):
    world = min(_ngpu(), 2)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    h, mesh = _build(ctx, mesh_file, D, n, divide, neumann)
    fn = _smooth_field(h, 23)
    if neumann:
        fn -= fn.mean()
    f, u = h.new_vec(0, fn), h.new_vec(0)
    its, rel = h.gmg_solve(f, u, tol=1e-10, max_it=100)
    single = u.download().reshape(-1, n ** D)
    h.close()
    mesh.close()
    mpc = mp.get_context("spawn")
    ret = mpc.Manager().dict()
    with tempfile.TemporaryDirectory() as tmp:
        idfile = os.path.join(tmp, "nccl_id")
        procs = [mpc.Process(target=_worker, args=(r, world, idfile, mesh_file, D, n, divide, fn, ret, neumann)) for r in range(world)]
        for p in procs:
            p.start()
        for p in procs:
            p.join(300)
            assert p.exitcode == 0
    owned = np.concatenate([ret[r]["owned"] for r in range(world)])
    gathered = np.concatenate([ret[r]["u"] for r in range(world)])[np.argsort(owned)]
    assert ret[0]["ndist"] >= 1
    assert all(ret[r]["its"] == its for r in range(world))
    assert rel_l2(gathered, single) < 1e-12
