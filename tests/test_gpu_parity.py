"""GPU parity tests: every call goes through the C-ABI (libtgpu.so) and is compared with
 (a) golden vectors produced by the reference's own code (tests/golden/*.npz),
 (b) the numpy oracle (oracle/gmg_oracle.py) on seeded inputs at other sizes,
 (c) size-independent properties at BASELINE.json's full single-GPU size.
Tolerance: north_star asks for 1e-10 relative L2; fp re-association is all that differs, so the
tests hold the kernels to 1e-12 (1e-10 only for Krylov trajectories)."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

import gmg_oracle as go
import pressurepoissonsolver_b200 as pps
from conftest import GOLDEN_CASES, MESHES, NEUMANN_CASES, ROOT, load_golden, rel_l2

pytestmark = pytest.mark.gpu
TOL = 1e-12


@pytest.fixture(scope="module")
def ctx():
    c = pps.Context(0)
    yield c
    c.close()


def build(ctx, mesh_file, D, n, divide=0):
    mesh = pps.Mesh.load(os.path.join(MESHES, mesh_file), D)
    mesh.refine_leaves(divide)
    return pps.Hierarchy.from_mesh(ctx, mesh, n), mesh


@pytest.fixture(scope="module", params=GOLDEN_CASES)
def gcase(request, ctx):
    g = load_golden(request.param)
    h, mesh = build(ctx, str(g["mesh"]), int(g["D"]), int(g["n"]), int(g["divide"]))
    yield g, h
    h.close()
    mesh.close()


def test_level_operators_vs_reference(gcase):
    g, h = gcase
    for l in range(h.nlevels):
        u = h.new_vec(l, g["L%d_in_u" % l])
        f = h.new_vec(l, g["L%d_in_f" % l])
        out = h.new_vec(l)
        h.apply(l, u, out)
        assert rel_l2(out.download(), g["L%d_apply" % l]) < TOL
        h.residual(l, f, u, out)
        assert rel_l2(out.download(), g["L%d_in_f" % l] - g["L%d_apply" % l]) < TOL
        if l + 1 < h.nlevels:
            c = h.new_vec(l + 1)
            h.restrict(l, u, c)
            assert np.array_equal(c.download(), g["L%d_restrict" % l])  # bit exact
            uc = h.new_vec(l + 1, g["L%d_in_uc" % l])
            fine = h.new_vec(l, g["L%d_in_u" % l])
            h.prolong_add(l, uc, fine)
            assert np.array_equal(fine.download(), g["L%d_interp" % l])  # bit exact
            h.residual_restrict(l, f, u, c)
            # fused residual+restrict == restrict(f - A u) of the separate kernels up to the order of
            # the 2^D-term average (warp-shuffle tree instead of the reference's left fold)
            h.residual(l, f, u, out)
            c2 = h.new_vec(l + 1)
            h.restrict(l, out, c2)
            assert rel_l2(c.download(), c2.download()) < 1e-15
        h.smooth(l, f, u)
        assert rel_l2(u.download(), g["L%d_smooth" % l]) < TOL


@pytest.mark.parametrize("fused,graph", [(1, 1), (1, 0), (2, 1), (2, 0), (0, 1), (0, 0)])
def test_vcycle_vs_reference(gcase, fused, graph):
    g, h = gcase
    f = h.new_vec(0, g["rhs_f"])
    u = h.new_vec(0)
    opts = pps.CycleOpts.default(fused=fused, use_graph=graph)
    h.vcycle(f, u, opts)
    assert rel_l2(u.download(), g["vcycle"]) < TOL
    h.vcycle(f, u, opts)  # graph replay path
    assert rel_l2(u.download(), g["vcycle"]) < TOL


def test_rhs_init_vs_reference(gcase):
    g, h = gcase
    f, e = h.new_vec(0), h.new_vec(0)
    h.init_trig_rhs(f, e)
    assert rel_l2(f.download(), g["rhs_f"]) < 1e-13
    assert rel_l2(e.download(), g["rhs_exact"]) < 1e-13


def test_residual_history_and_bicgstab_vs_reference(gcase):
    g, h = gcase
    f = h.new_vec(0, g["rhs_f"])
    u, r, e = h.new_vec(0), h.new_vec(0), h.new_vec(0)
    fn = f.two_norm()
    hist = []
    for k in range(7):
        h.residual(0, f, u, r)
        hist.append(r.two_norm() / fn)
        if k == 6:
            break
        h.vcycle(r, e)
        u.add(e)
    # per-cycle residual reduction and the solution at the same cycle count (north_star's criterion)
    assert np.max(np.abs(np.array(hist) / g["vhist"] - 1)) < 1e-8
    assert rel_l2(u.download(), g["vhist_u"]) < 1e-10
    x = h.new_vec(0)
    its, rel = h.bicgstab(f, x, tol=1e-12, max_it=100)
    assert its == int(g["bicgstab_info"][0])
    assert rel_l2(x.download(), g["bicgstab_u"]) < 1e-10


ORACLE_CASES = [("3uni.bin", 3, 16, 0), ("2refine.bin", 3, 16, 0), ("2refine.bin", 3, 8, 1), ("2d2ref.bin", 2, 32, 1),
                ("2d_multi_refine_8.bin", 2, 16, 0), ("2d2uni.bin", 2, 32, 2), ("multi_refine.bin", 3, 8, 0),
                ("2uni.bin", 3, 32, 0), ("2refine.bin", 3, 32, 0)]  # 32^3 patches (BASELINE config D) have their own kernels


@pytest.mark.parametrize("mesh_file,D,n,divide", ORACLE_CASES)
def test_vs_oracle_seeded(ctx, mesh_file, D, n, divide):
    h, mesh = build(ctx, mesh_file, D, n, divide)
    levels = go.build_hierarchy(os.path.join(MESHES, mesh_file), D, n, divide)
    assert [L.P for L in levels] == [h.npatch(l) for l in range(h.nlevels)]
    rng = np.random.default_rng(1234)
    for l, L in enumerate(levels):
        un = rng.standard_normal(L.shape)
        fn = rng.standard_normal(L.shape)
        u, f, out = h.new_vec(l, un), h.new_vec(l, fn), h.new_vec(l)
        h.apply(l, u, out)
        assert rel_l2(out.download(), go.apply_op(L, un)) < TOL
        h.smooth(l, f, u)
        assert rel_l2(u.download(), go.smooth(L, fn, un)) < TOL
        if l + 1 < len(levels):
            c = h.new_vec(l + 1)
            h.restrict(l, f, c)
            assert np.array_equal(c.download(), go.restrict(L, levels[l + 1], fn).ravel())
    fn = rng.standard_normal(levels[0].shape)
    f, u = h.new_vec(0, fn), h.new_vec(0)
    h.vcycle(f, u)
    assert rel_l2(u.download(), go.vcycle(levels, fn)) < TOL
    for opts in (dict(pre_sweeps=2, post_sweeps=2, coarse_sweeps=2), dict(pre_sweeps=2, post_sweeps=1, fused=0),
                 dict(pre_sweeps=3, post_sweeps=2, coarse_sweeps=3, fused=2), dict(pre_sweeps=3, post_sweeps=3),
                 dict(cycle_type=1), dict(pre_sweeps=0, post_sweeps=2)):
        h.vcycle(f, u, pps.CycleOpts.default(**opts))
        ref = go.cycle(levels, fn, cycle_type="W" if opts.get("cycle_type", 0) == 1 else "V", pre=opts.get("pre_sweeps", 1),
                       post=opts.get("post_sweeps", 1), coarse_sweeps=opts.get("coarse_sweeps", 1))
        assert rel_l2(u.download(), ref) < TOL, opts
    h.close()
    mesh.close()


@pytest.mark.parametrize("mesh_file,divide", [("3uni.bin", 0), ("2refine.bin", 1), ("multi_refine.bin", 0)])
def test_specialised_3d16_kernels_vs_generic(ctx, mesh_file, divide):
    """D = 3, n = 16 has its own smoother kernel (smooth3d16.cuh); every variant of it must agree with
    the size-generic kernel, and both with the oracle."""
    h, mesh = build(ctx, mesh_file, 3, 16, divide)
    levels = go.build_hierarchy(os.path.join(MESHES, mesh_file), 3, 16, divide)
    rng = np.random.default_rng(99)
    fn = rng.standard_normal(levels[0].shape)
    un = rng.standard_normal(levels[0].shape)
    f = h.new_vec(0, fn)
    res = {}
    for generic in (False, True):
        h.force_generic_kernels(generic)
        u = h.new_vec(0, un)
        h.smooth(0, f, u)
        res[generic, "smooth"] = u.download()
        for name, opts in (("v11", {}), ("v22", dict(pre_sweeps=2, post_sweeps=2, coarse_sweeps=2)),
                           ("v11_u", dict(fused=2)), ("v32_u", dict(pre_sweeps=3, post_sweeps=2, fused=2)),
                           ("plain", dict(fused=0))):
            h.vcycle(f, u, pps.CycleOpts.default(**opts))
            res[generic, name] = u.download()
    h.force_generic_kernels(False)
    for key in ("smooth", "v11", "v22", "v11_u", "v32_u", "plain"):
        assert rel_l2(res[False, key], res[True, key]) < 1e-13, key
    assert rel_l2(res[False, "smooth"], go.smooth(levels[0], fn, un)) < TOL
    assert rel_l2(res[False, "v11"], go.vcycle(levels, fn)) < TOL
    assert rel_l2(res[False, "v11_u"], go.vcycle(levels, fn)) < TOL
    assert rel_l2(res[False, "plain"], go.vcycle(levels, fn)) < TOL
    assert rel_l2(res[False, "v22"], go.vcycle(levels, fn, pre=2, post=2, coarse_sweeps=2)) < TOL
    assert rel_l2(res[False, "v32_u"], go.vcycle(levels, fn, pre=3, post=2)) < TOL
    h.close()
    mesh.close()


def test_apply_vs_the_references_assembled_matrix(ctx):
    """the operator kernels against the reference's second, independent implementation of the operator: the assembled
    matrix of MatrixHelper::formCRSMatrix / StencilHelper.h (golden 3d_assembled_operator, see make_golden.py), on every
    level of the refined 3D goldens, Dirichlet and Neumann"""
    a = load_golden("3d_assembled_operator")
    seen = 0
    for name in list(GOLDEN_CASES) + list(NEUMANN_CASES):
        g = load_golden(name)
        if int(g["D"]) != 3:
            continue
        mesh = pps.Mesh.load(os.path.join(MESHES, str(g["mesh"])), 3)
        if name.endswith("_neumann"):
            mesh.set_neumann(True)
        mesh.refine_leaves(int(g["divide"]))
        h = pps.Hierarchy.from_mesh(ctx, mesh, int(g["n"]))
        for l in range(h.nlevels):
            u, out = h.new_vec(l, g["L%d_in_u" % l]), h.new_vec(l)
            h.apply(l, u, out)
            assert rel_l2(out.download(), a["%s_L%d_matapply" % (name, l)]) < TOL, (name, l)
            seen += 1
        h.close()
        mesh.close()
    assert seen == 19


@pytest.mark.parametrize("name", NEUMANN_CASES)
def test_neumann_vs_reference(ctx, name):
    """Neumann domain boundaries: per-level operator and smoother and the V-cycle against the reference's
    golden vectors; the residual-from-faces schedule against the API-granular one."""
    g = load_golden(name)
    D, n = int(g["D"]), int(g["n"])
    mesh = pps.Mesh.load(os.path.join(MESHES, str(g["mesh"])), D).set_neumann(True)
    mesh.refine_leaves(int(g["divide"]))
    h = pps.Hierarchy.from_mesh(ctx, mesh, n)
    assert h.nlevels == int(g["nlevels"])
    for l in range(h.nlevels):
        u, f, out = h.new_vec(l, g["L%d_in_u" % l]), h.new_vec(l, g["L%d_in_f" % l]), h.new_vec(l)
        h.apply(l, u, out)
        assert rel_l2(out.download(), g["L%d_apply" % l]) < TOL
        h.smooth(l, f, u)
        assert rel_l2(u.download(), g["L%d_smooth" % l]) < 1e-11
    f, u = h.new_vec(0, g["rhs_f"]), h.new_vec(0)
    for fused in (1, 2, 0):
        h.vcycle(f, u, pps.CycleOpts.default(fused=fused))
        assert rel_l2(u.download(), g["vcycle"]) < 1e-10, fused
    h.close()
    mesh.close()


def test_neumann_vs_oracle_seeded(ctx):
    """larger Neumann cases against the oracle, incl. the D = 3, n = 16 size (which must leave its
    specialised Dirichlet kernel for the general path) and multi-sweep cycles"""
    for mesh_file, D, n, divide in (("2refine.bin", 3, 16, 0), ("2d_multi_refine_8.bin", 2, 32, 0), ("3uni.bin", 3, 4, 0),
                                    ("2uni.bin", 3, 32, 0),   # 32^3: general path through a scratch block (smooth3d32n_kernel)
                                    ("3uni.bin", 3, 32, 0),   # 32^3, mixed level: 8 interior patches on the cluster kernel, 56 on the general path
                                    ("3uni.bin", 3, 16, 1)):  # 16^3, mixed level of 512 patches (smooth3d16_kernel skips, smooth_kernel sweeps the rest)
        mesh = pps.Mesh.load(os.path.join(MESHES, mesh_file), D).set_neumann(True)
        mesh.refine_leaves(divide)
        h = pps.Hierarchy.from_mesh(ctx, mesh, n)
        levels = go.build_hierarchy(os.path.join(MESHES, mesh_file), D, n, divide, neumann=True)
        rng = np.random.default_rng(77)
        for l, L in enumerate(levels):
            un, fn = rng.standard_normal(L.shape), rng.standard_normal(L.shape)
            u, f, out = h.new_vec(l, un), h.new_vec(l, fn), h.new_vec(l)
            h.apply(l, u, out)
            assert rel_l2(out.download(), go.apply_op(L, un)) < TOL
            h.smooth(l, f, u)
            assert rel_l2(u.download(), go.smooth(L, fn, un)) < 1e-11
        fn = rng.standard_normal(levels[0].shape)
        fn -= fn.mean()
        f, u = h.new_vec(0, fn), h.new_vec(0)
        h.vcycle(f, u)
        assert rel_l2(u.download(), go.vcycle(levels, fn)) < 1e-10
        h.vcycle(f, u, pps.CycleOpts.default(pre_sweeps=2, post_sweeps=2, coarse_sweeps=2))
        assert rel_l2(u.download(), go.vcycle(levels, fn, pre=2, post=2, coarse_sweeps=2)) < 1e-10
        h.close()
        mesh.close()


@pytest.mark.parametrize("mesh_file,D,n,divide,neumann", [("2refine.bin", 3, 16, 1, False), ("2uni.bin", 3, 32, 0, False), ("2d2ref.bin", 2, 32, 1, False),
                                                          ("2refine.bin", 3, 16, 1, True)])  # Neumann instantiation + plain one on mixed levels
def test_cycle_is_bitwise_reproducible(ctx, mesh_file, D, n, divide, neumann):
    """the specialised kernels hand data between warps, CTAs of a cluster and kernels through shared memory, distributed
    shared memory and face buffers: a missing barrier would show up as bits that change from run to run"""
    mesh = pps.Mesh.load(os.path.join(MESHES, mesh_file), D)
    if neumann:
        mesh.set_neumann(True)
    mesh.refine_leaves(divide)
    h = pps.Hierarchy.from_mesh(ctx, mesh, n)
    fn = np.random.default_rng(21).standard_normal(h.ncells(0))
    f, u = h.new_vec(0, fn), h.new_vec(0)
    ref_bits = None
    for rep in range(12):
        h.vcycle(f, u, pps.CycleOpts.default(use_graph=rep & 1))
        bits = u.download().tobytes()
        ref_bits = ref_bits or bits
        assert bits == ref_bits, rep
    h.close()
    mesh.close()


def test_neumann_rhs_initialiser_vs_reference(ctx):
    """tgpu_init_neumann_rhs / tgpu_vec_integrate against the reference's own Init::initNeumann and Domain::integrate
    (golden 3d_2refine_n8_neumann_init: trig and gauss problems of apps/3d/steady.cpp on the refined octree)"""
    g = load_golden("3d_2refine_n8_neumann_init")
    mesh = pps.Mesh.load(os.path.join(MESHES, str(g["mesh"])), 3).set_neumann(True)
    h = pps.Hierarchy.from_mesh(ctx, mesh, int(g["n"]))
    f, e = h.new_vec(0), h.new_vec(0)
    for prob in ("trig", "gauss"):
        h.init_neumann_rhs(f, e, prob)
        assert rel_l2(f.download(), g["f_" + prob]) < 1e-13
        assert rel_l2(e.download(), g["exact_" + prob]) < 1e-14
        integral, volume = h.integrate(f)
        assert abs(volume - float(g["volume"])) < 1e-14
        assert abs(integral / volume - float(g["fdiff_" + prob])) < 1e-11 * max(1.0, abs(float(g["fdiff_" + prob])))
    h.close()
    mesh.close()
    # 2D: Init::initNeumann2d, trig problem
    g2 = load_golden("2d_2d2ref_d1_n8_neumann_init")
    mesh2 = pps.Mesh.load(os.path.join(MESHES, str(g2["mesh"])), 2).set_neumann(True)
    mesh2.refine_leaves(int(g2["divide"]))
    h2 = pps.Hierarchy.from_mesh(ctx, mesh2, int(g2["n"]))
    f2, e2 = h2.new_vec(0), h2.new_vec(0)
    h2.init_neumann_rhs(f2, e2, "trig")
    assert rel_l2(f2.download(), g2["f_trig"]) < 1e-13
    assert rel_l2(e2.download(), g2["exact_trig"]) < 1e-14
    integral, volume = h2.integrate(f2)
    assert abs(volume - 1.0) < 1e-14 and abs(integral / volume - float(g2["fdiff_trig"])) < 1e-11
    h2.close()
    mesh2.close()
    # the app's Neumann solve: remove the mean, BiCGStab + V-cycle, compare with the exact solution up to a constant
    mesh = pps.Mesh.load(os.path.join(MESHES, str(g["mesh"])), 3).set_neumann(True)
    h = pps.Hierarchy.from_mesh(ctx, mesh, int(g["n"]))
    f, e = h.new_vec(0), h.new_vec(0)
    h.init_neumann_rhs(f, e, "trig")
    integral, volume = h.integrate(f)
    f.shift(-integral / volume)
    u = h.new_vec(0)
    its, rel = h.bicgstab(f, u, tol=1e-10, max_it=100)
    assert rel < 1e-10
    d = u.download() - e.download()
    d -= d.mean()
    assert np.linalg.norm(d) / np.linalg.norm(e.download()) < 0.05  # second-order discretisation error on 8^3 patches
    h.close()
    mesh.close()


def test_neumann_generic_kernels_vs_oracle(ctx):
    """16^3 Neumann levels with the size-generic kernels forced: every patch of a level through smooth_kernel's general path
    instead of the split between the Neumann instantiation and the plain one of smooth3d16_kernel - gives the oracle's cycle too"""
    for mesh_file, divide in (("3uni.bin", 1), ("2refine.bin", 0)):
        path = os.path.join(MESHES, mesh_file)
        mesh = pps.Mesh.load(path, 3).set_neumann(True)
        mesh.refine_leaves(divide)
        h = pps.Hierarchy.from_mesh(ctx, mesh, 16)
        h.force_generic_kernels(True)
        levels = go.build_hierarchy(path, 3, 16, divide, neumann=True)
        fn = np.random.default_rng(5).standard_normal(levels[0].shape)
        fn -= fn.mean()
        f, u = h.new_vec(0, fn), h.new_vec(0)
        ref = go.vcycle(levels, fn, pre=2, post=2, coarse_sweeps=2)
        for graph in (0, 1):
            h.vcycle(f, u, pps.CycleOpts.default(use_graph=graph, pre_sweeps=2, post_sweeps=2, coarse_sweeps=2))
            err = np.linalg.norm(u.download() - ref.ravel()) / np.linalg.norm(ref)
            assert err < 1e-10, (mesh_file, graph, err)
        h.close()
        mesh.close()


def test_blas1_and_reductions(ctx):
    h, mesh = build(ctx, "2refine.bin", 3, 8, 1)
    rng = np.random.default_rng(7)
    n = h.ncells(0)
    a, b, c = (rng.standard_normal(n) for _ in range(3))
    va, vb, vc = h.new_vec(0, a), h.new_vec(0, b), h.new_vec(0, c)
    assert abs(va.dot(vb) / np.dot(a, b) - 1) < 1e-12
    assert abs(va.two_norm() / np.linalg.norm(a) - 1) < 1e-13
    assert va.inf_norm() == np.max(np.abs(a))
    va.add_scaled(0.3, vb); a = a + b * 0.3
    va.add_scaled2(-1.5, vb, 0.25, vc); a = a + (b * -1.5 + c * 0.25)
    va.scale_then_add(2.0, vc); a = 2.0 * a + c
    va.scale_then_add_scaled(0.5, -3.0, vb); a = 0.5 * a + -3.0 * b
    va.scale_then_add_scaled2(1.25, 2.0, vb, -0.5, vc); a = 1.25 * a + 2.0 * b + -0.5 * c
    va.scale(0.7); a = a * 0.7
    va.shift(1.5); a = a + 1.5
    va.add(vb); a = a + b
    assert rel_l2(va.download(), a) < 1e-15
    vb.copy(va)
    assert np.array_equal(vb.download(), va.download())
    vb.set(3.0)
    assert np.all(vb.download() == 3.0)
    assert np.all(h.new_vec(0).download() == 0.0)  # new vectors are zero like PETSc Vecs
    h.close()
    mesh.close()


def test_error_behaviour(ctx):
    h, mesh = build(ctx, "2refine.bin", 3, 8, 0)
    u0, u1 = h.new_vec(0), h.new_vec(1)
    with pytest.raises(pps.TgpuError):
        h.apply(0, u1, u0)  # vector from another level (reference: throw 3)
    with pytest.raises(pps.TgpuError):
        h.vcycle(u0, u0)
    with pytest.raises(pps.TgpuError):
        h.vcycle(u0, h.new_vec(0), pps.CycleOpts.default(cycle_type=7))
    with pytest.raises(pps.TgpuError):
        pps.Hierarchy.from_mesh(ctx, mesh, 6)  # unsupported patch size
    with pytest.raises(pps.TgpuError):
        pps.Hierarchy.from_mesh(ctx, mesh, 64)
    h.close()
    mesh.close()


CYCLE_GOLDENS = ["3d_2refine_n8", "2d_2d2ref_d1_n8", "3d_multi_refine_n4"]
CYCLE_VARIANT_OPTS = {
    "W": dict(cycle_type=1), "W_p2m2c2": dict(cycle_type=1, pre_sweeps=2, mid_sweeps=2, post_sweeps=1, coarse_sweeps=2),
    "V_max_levels2": dict(max_levels=2), "V_ppp2": dict(patches_per_proc=2.0), "W_max_levels2": dict(cycle_type=1, max_levels=2),
}


@pytest.mark.parametrize("name", CYCLE_GOLDENS)
def test_cycle_variants_vs_reference(ctx, name):
    """W cycles (GMG/WCycle.h:45-68), the level truncation of the factory (CycleOpts max_levels / patches_per_proc,
    GMG/CycleFactory3d.cpp:99-104) and the patch solver's lambda (FftwPatchSolver.h:66,170) against golden vectors the
    reference itself produced (tests/golden/*_cycles.npz), on every schedule and with / without graph replay."""
    g, c = load_golden(name), load_golden(name + "_cycles")
    h, mesh = build(ctx, str(g["mesh"]), int(g["D"]), int(g["n"]), int(g["divide"]))
    f, u = h.new_vec(0, g["rhs_f"]), h.new_vec(0)
    for key, kw in CYCLE_VARIANT_OPTS.items():
        for fused in (1, 0):
            for graph in (1, 0):
                h.vcycle(f, u, pps.CycleOpts.default(fused=fused, use_graph=graph, **kw))
                assert rel_l2(u.download(), c["cycle_" + key]) < TOL, (key, fused, graph)
    # the plain cycle still comes out after truncated ones (the level limit is per call, not sticky)
    h.vcycle(f, u)
    assert rel_l2(u.download(), g["vcycle"]) < TOL
    # BiCGStab preconditioned with a W cycle converges in no more iterations than with the V cycle
    x = h.new_vec(0)
    its_w, rel = h.bicgstab(f, x, pps.CycleOpts.default(cycle_type=1), tol=1e-12, max_it=100)
    assert rel <= 1e-12 and its_w <= int(g["bicgstab_info"][0])
    lam = float(c["lambda"])
    h.set_lambda(lam)
    for l in range(h.nlevels):
        ul, fl = h.new_vec(l, c["L%d_in_u" % l]), h.new_vec(l, c["L%d_in_f" % l])
        h.smooth(l, fl, ul)
        assert rel_l2(ul.download(), c["L%d_smooth_lambda" % l]) < TOL, l
    for fused in (1, 2, 0):
        h.vcycle(f, u, pps.CycleOpts.default(fused=fused))
        assert rel_l2(u.download(), c["cycle_V_lambda"]) < 1e-11, fused
    h.set_lambda(0.0)
    h.vcycle(f, u)
    assert rel_l2(u.download(), g["vcycle"]) < TOL
    h.close()
    mesh.close()


@pytest.mark.parametrize("mesh_file,D,n,divide", [("2refine.bin", 3, 16, 0), ("2uni.bin", 3, 32, 0), ("2d2ref.bin", 2, 32, 1)])
def test_lambda_on_specialised_sizes_vs_oracle(ctx, mesh_file, D, n, divide):
    """a non-zero lambda must leave the specialised Dirichlet kernels (16^3, 32^3, 2D 32^2) for the general patch solve"""
    h, mesh = build(ctx, mesh_file, D, n, divide)
    levels = go.build_hierarchy(os.path.join(MESHES, mesh_file), D, n, divide)
    rng = np.random.default_rng(5)
    h.set_lambda(-7.25)
    for l, L in enumerate(levels):
        un, fn = rng.standard_normal(L.shape), rng.standard_normal(L.shape)
        u, f = h.new_vec(l, un), h.new_vec(l, fn)
        h.smooth(l, f, u)
        assert rel_l2(u.download(), go.smooth(L, fn, un, -7.25)) < 1e-11
    fn = rng.standard_normal(levels[0].shape)
    f, u = h.new_vec(0, fn), h.new_vec(0)
    h.vcycle(f, u)
    assert rel_l2(u.download(), go.cycle(levels, fn, lam=-7.25)) < 1e-11
    h.close()
    mesh.close()


def test_config_e_kernel_path_vs_oracle(ctx):
    """BASELINE config E's kernel path: the deeply refined quadtree multi_refine_8 with 32 x 32 patches and Dirichlet
    boundaries runs smooth2d32_kernel with coarse/fine faces on every level; per-level operators, the cycle (all
    schedules) and the Krylov solve against the oracle."""
    h, mesh = build(ctx, "2d_multi_refine_8.bin", 2, 32, 0)
    levels = go.build_hierarchy(os.path.join(MESHES, "2d_multi_refine_8.bin"), 2, 32, 0)
    assert [L.P for L in levels] == [h.npatch(l) for l in range(h.nlevels)] and levels[0].P == 160
    rng = np.random.default_rng(2718)
    for l, L in enumerate(levels):
        un, fn = rng.standard_normal(L.shape), rng.standard_normal(L.shape)
        u, f, out = h.new_vec(l, un), h.new_vec(l, fn), h.new_vec(l)
        h.apply(l, u, out)
        assert rel_l2(out.download(), go.apply_op(L, un)) < TOL
        h.smooth(l, f, u)
        assert rel_l2(u.download(), go.smooth(L, fn, un)) < TOL
        if l + 1 < len(levels):
            c = h.new_vec(l + 1)
            h.residual_restrict(l, f, u, c)
            r = -1 * go.apply_op(L, u.download().reshape(L.shape)) + fn
            assert rel_l2(c.download(), go.restrict(L, levels[l + 1], r)) < 1e-11
    fn = rng.standard_normal(levels[0].shape)
    f, u = h.new_vec(0, fn), h.new_vec(0)
    ref = go.vcycle(levels, fn)
    for fused in (1, 2, 0):
        for graph in (1, 0):
            h.vcycle(f, u, pps.CycleOpts.default(fused=fused, use_graph=graph))
            assert rel_l2(u.download(), ref) < TOL, (fused, graph)
    h.vcycle(f, u, pps.CycleOpts.default(pre_sweeps=2, post_sweeps=2, coarse_sweeps=2))
    assert rel_l2(u.download(), go.vcycle(levels, fn, pre=2, post=2, coarse_sweeps=2)) < TOL
    ft, et = go.trig_rhs(levels[0])
    f.upload(ft)
    x = h.new_vec(0)
    its, rel = h.bicgstab(f, x, tol=1e-12, max_it=100)
    xo, its_o = go.bicgstab(levels, ft)
    assert its == its_o and rel_l2(x.download(), xo) < 1e-10
    h.close()
    mesh.close()


@pytest.mark.parametrize("mesh_file,D,n,divide,neumann", [("2refine.bin", 3, 8, 0, False), ("2refine.bin", 3, 16, 0, False),
                                                          ("2d_multi_refine_8.bin", 2, 16, 0, False), ("2d2ref.bin", 2, 32, 1, True),
                                                          ("2uni.bin", 3, 32, 0, False), ("multi_refine.bin", 3, 4, 0, True)])
def test_weighted_jacobi_vs_oracle(ctx, mesh_file, D, n, divide, neumann):
    """the weighted-Jacobi option of the north star against oracle/gmg_oracle.jacobi (whose diagonal is pinned to the
    reference's operator by tests/test_oracle_vs_reference.py), three sweeps on every level"""
    mesh = pps.Mesh.load(os.path.join(MESHES, mesh_file), D).set_neumann(neumann)
    mesh.refine_leaves(divide)
    h = pps.Hierarchy.from_mesh(ctx, mesh, n)
    levels = go.build_hierarchy(os.path.join(MESHES, mesh_file), D, n, divide, neumann=neumann)
    rng = np.random.default_rng(31)
    for l, L in enumerate(levels):
        un, fn = rng.standard_normal(L.shape), rng.standard_normal(L.shape)
        u, f = h.new_vec(l, un), h.new_vec(l, fn)
        for omega in (0.8, 2.0 / 3.0, 1.0):
            h.smooth_jacobi(l, f, u, omega)
            un = go.jacobi(L, fn, un, omega)
        assert rel_l2(u.download(), un) < TOL, l
    h.close()
    mesh.close()


@pytest.mark.parametrize("mesh_file,D,n,divide", [("2refine.bin", 3, 8, 0), ("3uni.bin", 3, 16, 0), ("2d2ref.bin", 2, 32, 1),
                                                  ("2uni.bin", 3, 32, 0), ("multi_refine.bin", 3, 4, 0)])
def test_linear_interpolator(ctx, mesh_file, D, n, divide):
    """the piecewise (tri)linear interpolator: known answer of test/GMG.cpp:465-600 (linear fields are reproduced),
    agreement with the oracle's restatement of the TriLinIntp.cpp coefficient tables, and cycles that use it"""
    h, mesh = build(ctx, mesh_file, D, n, divide)
    levels = go.build_hierarchy(os.path.join(MESHES, mesh_file), D, n, divide)
    rng = np.random.default_rng(8)

    def field(L):
        out = np.zeros(L.shape)
        for p in range(L.P):
            c = [L.starts[p, a] + L.spacings[p, a] * (np.arange(n) + 0.5) for a in range(D)]
            out[p] = (c[0][None, None, :] + 0.5 * c[1][None, :, None] - c[2][:, None, None]) if D == 3 else (c[0][None, :] + 0.5 * c[1][:, None])
        return out

    for l in range(len(levels) - 1):
        fine, coarse = levels[l], levels[l + 1]
        uc, uf = h.new_vec(l + 1, field(coarse)), h.new_vec(l)
        h.prolong_add_linear(l, uc, uf)
        assert rel_l2(uf.download(), field(fine)) < 1e-14
        ucn, ufn = rng.standard_normal(coarse.shape), rng.standard_normal(fine.shape)
        uc.upload(ucn)
        uf.upload(ufn)
        h.prolong_add_linear(l, uc, uf)
        assert rel_l2(uf.download(), go.interpolate_trilinear(fine, coarse, ucn, ufn)) < 1e-14
    fn = rng.standard_normal(levels[0].shape)
    f, u = h.new_vec(0, fn), h.new_vec(0)
    for kw, okw in ((dict(), dict()), (dict(cycle_type=1, pre_sweeps=2), dict(cycle_type="W", pre=2))):
        h.vcycle(f, u, pps.CycleOpts.default(interpolator=1, **kw))
        assert rel_l2(u.download(), go.cycle(levels, fn, interp=go.interpolate_trilinear, **okw)) < TOL
    with pytest.raises(pps.TgpuError):
        h.vcycle(f, u, pps.CycleOpts.default(interpolator=5))
    h.close()
    mesh.close()


def test_vector_temporaries_keep_cached_graphs(ctx):
    """creating and destroying temporaries (what the API-granular plugin classes do every cycle, GMG/Cycle.h:59-64) neither
    invalidates the cycle graphs of other vectors nor changes results; tgpu_hierarchy_trim releases lazily allocated
    work space and everything still works afterwards"""
    h, mesh = build(ctx, "2refine.bin", 3, 16, 0)
    fn = np.random.default_rng(4).standard_normal(h.ncells(0))
    f, u = h.new_vec(0, fn), h.new_vec(0)
    h.vcycle(f, u)
    ref = u.download()
    n0 = ctx.kernel_launches()
    for _ in range(5):
        tmp = [h.new_vec(l) for l in range(h.nlevels)]
        for t in tmp:
            t.close()
        h.vcycle(f, u)
        assert np.array_equal(u.download(), ref)
    x = h.new_vec(0)
    its, _ = h.bicgstab(f, x, tol=1e-10, max_it=50)
    h.trim()
    x2 = h.new_vec(0)
    its2, _ = h.bicgstab(f, x2, tol=1e-10, max_it=50)
    assert its == its2 and np.array_equal(x.download(), x2.download())
    h.vcycle(f, u)
    assert np.array_equal(u.download(), ref) and ctx.kernel_launches() > n0
    h.close()
    mesh.close()


def test_weighted_jacobi_reduces_residual(ctx):
    h, mesh = build(ctx, "3uni.bin", 3, 8, 0)
    f, u, r = h.new_vec(0), h.new_vec(0), h.new_vec(0)
    h.init_trig_rhs(f)
    h.residual(0, f, u, r)
    r0 = r.two_norm()
    for _ in range(20):
        h.smooth_jacobi(0, f, u, 0.8)
    h.residual(0, f, u, r)
    assert r.two_norm() < 0.9 * r0
    h.close()
    mesh.close()


# ---- full-size (BASELINE config B: 4uni.bin --divide 1, n = 16, 16.8 M cells) properties ----
@pytest.fixture(scope="module")
def config_b(ctx):
    h, mesh = build(ctx, "4uni.bin", 3, 16, 1)
    yield h
    h.close()
    mesh.close()


def test_full_size_properties(config_b):
    h = config_b
    assert h.ncells(0) == 16777216 and h.nlevels == 5
    f, e, u, u2, r = (h.new_vec(0) for _ in range(5))
    h.init_trig_rhs(f, e)
    # linearity of the cycle: V(2 f) == 2 V(f) exactly (powers of two commute with every op)
    h.vcycle(f, u)
    f2 = h.new_vec(0)
    f2.copy(f)
    f2.scale(2.0)
    h.vcycle(f2, u2)
    u2.scale(0.5)
    assert np.array_equal(u.download(), u2.download())
    # fused schedules == API-granular schedule
    for fused in (0, 2):
        h.vcycle(f, u2, pps.CycleOpts.default(fused=fused, use_graph=0))
        u2.add_scaled(-1.0, u)
        assert u2.two_norm() / u.two_norm() < 1e-13, fused
    # stationary iteration contracts like the reference does on uniform meshes (~0.1-0.2 per cycle)
    u.set(0.0)
    hist = []
    fn = f.two_norm()
    for k in range(6):
        h.residual(0, f, u, r)
        hist.append(r.two_norm() / fn)
        h.vcycle(r, u2)
        u.add(u2)
    fac = [hist[i + 1] / hist[i] for i in range(5)]
    assert max(fac) < 0.35, fac
    # converged solution is second-order accurate w.r.t. the manufactured solution
    x = h.new_vec(0)
    its, rel = h.bicgstab(f, x, tol=1e-12, max_it=50)
    assert its <= 12 and rel <= 1e-12
    x.add_scaled(-1.0, e)
    assert x.inf_norm() < 2e-4
    # patch-constant vectors restrict/prolong to themselves
    c = h.new_vec(1)
    u.set(3.0)
    h.restrict(0, u, c)
    assert np.all(c.download() == 3.0)


def test_full_size_config_d_properties(ctx):
    """BASELINE config D itself (4uni.bin --divide 2, n = 32: 32,768 patches, 1,073,741,824 cells, the workload bench.py
    reports): size-independent properties evaluated on the device (no 8.6 GB host round trips): V(2 f) = 2 V(f) bit for bit,
    additivity V(f1 + f2) = V(f1) + V(f2) to rounding, the face-residual schedule against the one that forms the residual
    from u and f, the stationary iteration's contraction, and second-order accuracy of the converged solution."""
    import torch
    if torch.cuda.get_device_properties(0).total_memory < 120e9:
        pytest.skip("needs a 180 GB B200")
    mesh = pps.Mesh.load(os.path.join(MESHES, "4uni.bin"), 3).refine_leaves(2)
    h = pps.Hierarchy.from_mesh(ctx, mesh, 32)
    assert h.ncells(0) == 1073741824 and h.nlevels == 6
    f, e, u, u2, w = (h.new_vec(0) for _ in range(5))
    h.init_trig_rhs(f, e)
    h.vcycle(f, u)
    w.copy(f)
    w.scale(2.0)
    h.vcycle(w, u2)
    u2.scale(0.5)
    u2.add_scaled(-1.0, u)
    assert u2.inf_norm() == 0.0                      # powers of two commute with every operation of the cycle
    # additivity with a second, unrelated right-hand side (the first cycle's result)
    w.copy(f)
    w.add(u)                                         # w = f + u
    h.vcycle(u, u2)                                  # V(u)
    u2.add(u)                                        # ... + V(f)   (u still holds V(f): the cycle does not touch its input)
    r = h.new_vec(0)
    h.vcycle(w, r)                                   # V(f + u)
    r.add_scaled(-1.0, u2)
    assert r.two_norm() / u2.two_norm() < 1e-13
    h.vcycle(f, u2, pps.CycleOpts.default(fused=2, use_graph=0))
    u2.add_scaled(-1.0, u)
    assert u2.two_norm() / u.two_norm() < 1e-13
    u.set(0.0)
    hist = []
    fn = f.two_norm()
    for k in range(5):
        h.residual(0, f, u, r)
        hist.append(r.two_norm() / fn)
        h.vcycle(r, u2)
        u.add(u2)
    fac = [hist[i + 1] / hist[i] for i in range(4)]
    assert max(fac) < 0.35, fac
    for v in (u2, w, r):
        v.close()
    h.trim()
    x = h.new_vec(0)
    its, rel = h.bicgstab(f, x, tol=1e-10, max_it=30)
    assert its <= 10 and rel <= 1e-10
    x.add_scaled(-1.0, e)
    assert x.inf_norm() < 2e-5                       # h = 1/1024: second-order discretisation error (config B, h = 1/256: < 2e-4)
    for v in (x, f, e, u):
        v.close()
    h.close()
    mesh.close()


@pytest.mark.parametrize("mesh_file,D,n,divide,cells", [("2refine.bin", 3, 16, 3, 31457280), ("2d_multi_refine_8.bin", 2, 32, 4, 41943040)])
def test_full_size_adaptive_config_properties(ctx, mesh_file, D, n, divide, cells):
    """BASELINE configs C (2refine --divide 3, 16^3 patches) and E (2D multi_refine_8 --divide 4, 32^2 patches, 13 levels) at
    the sizes bench.py reports: exact homogeneity, additivity, the three schedules against each other, a contracting
    stationary iteration and a converging BiCGStab, all evaluated on the device"""
    mesh = pps.Mesh.load(os.path.join(MESHES, mesh_file), D).refine_leaves(divide)
    h = pps.Hierarchy.from_mesh(ctx, mesh, n)
    assert h.ncells(0) == cells
    f, e, u, u2, w, r = (h.new_vec(0) for _ in range(6))
    h.init_trig_rhs(f, e)
    h.vcycle(f, u)
    w.copy(f)
    w.scale(4.0)
    h.vcycle(w, u2)
    u2.scale(0.25)
    u2.add_scaled(-1.0, u)
    assert u2.inf_norm() == 0.0
    w.copy(f)
    w.add(u)
    h.vcycle(u, u2)
    u2.add(u)
    h.vcycle(w, r)
    r.add_scaled(-1.0, u2)
    assert r.two_norm() / u2.two_norm() < 1e-13
    for fused in (0, 2):
        h.vcycle(f, u2, pps.CycleOpts.default(fused=fused, use_graph=0))
        u2.add_scaled(-1.0, u)
        assert u2.two_norm() / u.two_norm() < 1e-13, fused
    u.set(0.0)
    hist = []
    fn = f.two_norm()
    for k in range(6):
        h.residual(0, f, u, r)
        hist.append(r.two_norm() / fn)
        h.vcycle(r, u2)
        u.add(u2)
    fac = [hist[i + 1] / hist[i] for i in range(5)]
    assert max(fac) < 0.8 and hist[-1] < 0.05 * hist[0], (fac, hist)
    x = h.new_vec(0)
    its, rel = h.bicgstab(f, x, tol=1e-10, max_it=60)
    assert rel <= 1e-10 and its <= 40, (its, rel)
    h.residual(0, f, x, r)
    assert r.two_norm() / fn < 2e-10                 # the recurrence residual BiCGStab reports is the true one
    h.close()
    mesh.close()


def test_medium_size_vs_reference_binary(ctx):
    """If the reference-built oracle binary travelled with the repo, compare a 2.1 M-cell V-cycle
    and its per-cycle residual reduction against the reference run on the same inputs."""
    ref = os.path.join(ROOT, "oracle", "_ref", "ref_gmg")
    if not os.path.exists(ref):
        pytest.skip("oracle/_ref/ref_gmg not built")
    h, mesh = build(ctx, "3uni.bin", 3, 16, 1)
    f, u, r, e = (h.new_vec(0) for _ in range(4))
    h.init_trig_rhs(f)
    with tempfile.TemporaryDirectory() as tmp:
        fp, vp, up, hp = (os.path.join(tmp, x) for x in ("f", "v", "u", "h"))
        f.download().tofile(fp)
        subprocess.check_call([ref, "3", os.path.join(MESHES, "3uni.bin"), "1", "16", "dft", "vcycle:%s:%s" % (fp, vp),
                               "vhist:%s:3:%s:%s" % (fp, up, hp)])
        h.vcycle(f, u)
        assert rel_l2(u.download(), np.fromfile(vp)) < 1e-11
        u.set(0.0)
        fn = f.two_norm()
        hist = []
        for k in range(4):
            h.residual(0, f, u, r)
            hist.append(r.two_norm() / fn)
            if k == 3:
                break
            h.vcycle(r, e)
            u.add(e)
        assert np.max(np.abs(np.array(hist) / np.fromfile(hp) - 1)) < 1e-8
        assert rel_l2(u.download(), np.fromfile(up)) < 1e-10
    h.close()
    mesh.close()
