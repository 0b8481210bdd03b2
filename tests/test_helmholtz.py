"""Helmholtz problems (tgpu_hierarchy_set_helmholtz): the operator A_l + lambda I on every level with the same patch solver
shift, so that every sweep solves its shifted patch problems exactly and the face identity of DESIGN 3 holds again.

The shifted reference is composed here from the oracle's pinned functions (oracle/ stays as it is): the operator
go.apply_op(L, u) + lambda u, the sweep go.smooth(L, f, u, lam=lambda), the weighted Jacobi sweep on the diagonal of
go.jacobi plus lambda, restriction and interpolation, and a cycle and FMG built on them.  go.smooth drops the joint zero
mode of an all-Neumann patch (the reference's FftwPatchSolver.h:197); the shifted problem keeps it, so the composed sweep
adds it back: on such a patch (no neighbours) the constant mode of the solution is mean(f_p) / lambda."""
import os

import numpy as np
import pytest

import gmg_oracle as go
from conftest import MESHES, rel_l2
from test_fmg import TRIG2, TRIG3, _mixed_hierarchy, boundary_values, fold_boundary, problem_data, restrict_rhs
from test_past_resident_grid import loop_thresholds

TOL = 1e-12
# sweeps and cycles from a random guess through the dense transforms of the Neumann patches (see test_boundary_closures)
TOL_GUESS = 1e-11
TGPU_ERR_ARG = 1


# ---- the composed shifted reference ----
def A(L, u, lam):
    return go.apply_op(L, u) + lam * u


def smooth(L, f, u, lam, mu=None):
    """one sweep; mu: a patch solver shift the operator does not carry (tgpu_hierarchy_set_lambda alone: the reference's
    patch solve, zero mode dropped)"""
    if mu is not None:
        return go.smooth(L, f, u, mu)
    out = go.smooth(L, f, u, lam)
    if lam != 0.0:
        for k in np.nonzero(L.neumann == (1 << (2 * L.D)) - 1)[0]:
            out[k] += f[k].mean() / lam
    return out


def jacobi(L, f, u, omega, lam):
    """u + omega (f - (A + lam) u) / (diag(A) + lam), diag(A) read off go.jacobi"""
    diag = 1.0 / go.jacobi(L, np.ones(L.shape), np.zeros(L.shape), 1.0)
    return u + omega * (f - A(L, u, lam)) / (diag + lam)


def cycle(levels, f, lam, mu=None, cycle_type="V", pre=1, post=1, mid=1, coarse_sweeps=1, max_levels=0, interp=None):
    """go.cycle with the shifted operator and sweep"""
    lv = go.active_levels(levels, max_levels)
    interp = interp or go.interpolate

    def visit(l, fl, u):
        L = lv[l]
        if l == len(lv) - 1:
            for _ in range(coarse_sweeps):
                u = smooth(L, fl, u, lam, mu)
            return u

        def coarse_correction(u):
            fc = go.restrict(L, lv[l + 1], fl - A(L, u, lam))
            return interp(L, lv[l + 1], visit(l + 1, fc, np.zeros(lv[l + 1].shape)), u)

        for _ in range(pre):
            u = smooth(L, fl, u, lam, mu)
        u = coarse_correction(u)
        if cycle_type == "W":
            for _ in range(mid):
                u = smooth(L, fl, u, lam, mu)
            u = coarse_correction(u)
        for _ in range(post):
            u = smooth(L, fl, u, lam, mu)
        return u

    return visit(0, f, np.zeros(lv[0].shape))


def fmg(levels, f, b, cycles, lam):
    """test_fmg.fmg with the shifted operator, sweep and cycle (V(1,1), linear interpolation of the coarser result)"""
    fs, bs = [np.asarray(f).reshape(levels[0].shape)], [b]
    for l in range(len(levels) - 1):
        fc, bc = restrict_rhs(levels[l], levels[l + 1], fs[l], bs[l])
        fs.append(fc)
        bs.append(bc)
    u = smooth(levels[-1], fs[-1], np.zeros(levels[-1].shape), lam)
    for l in range(len(levels) - 2, -1, -1):
        u = go.interpolate_trilinear(levels[l], levels[l + 1], u, np.zeros(levels[l].shape))
        for _ in range(cycles):
            u = u + cycle(levels[l:], fs[l] - A(levels[l], u, lam), lam)
    return u


def lam_for(L, c):
    """lambda with lambda h^2 = c on the finest cells of L"""
    return c / float(L.spacings[:, 0].min()) ** 2


# ---- CPU ----
@pytest.mark.parametrize("mesh_file,D,n,divide", [("2refine.bin", 3, 8, 0), ("2d2ref.bin", 2, 8, 1), ("2refine.bin", 3, 4, 1)])
@pytest.mark.parametrize("c", [-1e-3, -1.0, -100.0])
def test_face_identity_after_a_sweep(mesh_file, D, n, divide, c):
    """f - (A + lambda) u_new = (2/h^2) E^T (gamma(u_old) - gamma(u_new)): zero off the patch boundary cells"""
    L = go.build_hierarchy(os.path.join(MESHES, mesh_file), D, n, divide)[0]
    lam = lam_for(L, c)
    rng = np.random.default_rng(7)
    f, u0 = rng.standard_normal(L.shape), rng.standard_normal(L.shape)
    u1 = smooth(L, f, u0, lam)
    g0, g1 = go.interface_values(L, u0), go.interface_values(L, u1)
    want = np.zeros(L.shape)
    for s in range(2 * D):
        has = L.nbr_type[:, s] != go.NBR_NONE
        h2 = (L.spacings[:, s // 2] ** 2).reshape((-1,) + (1,) * (D - 1))
        go.face(want, D, s)[has] += (2.0 / h2 * (g0[:, s] - g1[:, s]))[has]
    r = f - A(L, u1, lam)
    assert rel_l2(r, want) < 1e-13


@pytest.mark.parametrize("mesh_file,D,n,divide,neumann", [("2d2ref.bin", 2, 8, 1, False), ("2refine.bin", 3, 4, 0, False),
                                                          ("2d2ref.bin", 2, 8, 1, True)])
def test_stationary_iteration_converges(mesh_file, D, n, divide, neumann):
    """u += Cycle(f - (A + lambda) u) reaches 1e-10 for lambda h^2 = -1e-3, -1, -100, and needs fewer cycles the larger
    |lambda| h^2 is"""
    levels = go.build_hierarchy(os.path.join(MESHES, mesh_file), D, n, divide, neumann=neumann)
    f = np.random.default_rng(9).standard_normal(levels[0].shape)
    counts = []
    for c in (-1e-3, -1.0, -100.0):
        lam = lam_for(levels[0], c)
        u = np.zeros(levels[0].shape)
        for k in range(60):
            r = f - A(levels[0], u, lam)
            if np.linalg.norm(r) <= 1e-10 * np.linalg.norm(f):
                break
            u = u + cycle(levels, r, lam)
        else:
            pytest.fail("no convergence at lambda h^2 = %g" % c)
        counts.append(k)
    assert counts[0] >= counts[1] >= counts[2], counts


def test_set_helmholtz_rejects_bad_lambda_without_a_device():
    import pressurepoissonsolver_b200 as pps
    for bad in (float("nan"), float("inf"), float("-inf"), 1e-300, 2.0):
        assert pps.lib.tgpu_hierarchy_set_helmholtz(None, bad) == TGPU_ERR_ARG, bad
        assert b"finite and <= 0" in pps.lib.tgpu_last_error()
    assert pps.lib.tgpu_hierarchy_set_helmholtz(None, -1.0) == TGPU_ERR_ARG  # (the null hierarchy)
    assert b"null" in pps.lib.tgpu_last_error()


# ---- GPU ----
def _pps():
    import pressurepoissonsolver_b200 as pps
    return pps


@pytest.fixture(scope="module")
def ctx():
    c = _pps().Context(0)
    yield c
    c.close()


# mesh, D, n, divide, Neumann side mask (0: Dirichlet; all ones: every domain side Neumann)
CASES = [("2refine.bin", 3, 4, 1, 0), ("2refine.bin", 3, 8, 0, 0), ("2refine.bin", 3, 16, 0, 0), ("2refine.bin", 3, 32, 0, 0),
         ("2d2ref.bin", 2, 8, 1, 0), ("2d2ref.bin", 2, 16, 1, 0), ("2d2ref.bin", 2, 32, 1, 0),
         ("2refine.bin", 3, 8, 0, 0b111111), ("2refine.bin", 3, 16, 0, 0b111111), ("2refine.bin", 3, 32, 0, 0b111111),
         ("2d2ref.bin", 2, 32, 1, 0b1111),
         ("3uni.bin", 3, 16, 1, 0b001100), ("2refine.bin", 3, 32, 0, 0b000010), ("2d2ref.bin", 2, 32, 1, 0b1100)]


def _id(c):
    return "%s_d%d_n%d_D%d_%s" % (c[0][:-4], c[3], c[2], c[1], format(c[4], "b"))


@pytest.fixture(scope="module")
def case(request, ctx):
    mesh_file, D, n, divide, mask = request.param
    h, mesh, levels = _mixed_hierarchy(ctx, mesh_file, D, n, divide, mask)
    lam = lam_for(levels[0], -1.0)
    h.set_helmholtz(lam)
    yield h, levels, lam
    h.close()
    mesh.close()


def _opts(**kw):
    o = _pps().CycleOpts.default()
    for k, v in kw.items():
        setattr(o, k, v)
    return o


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, indirect=True, ids=[_id(c) for c in CASES])
def test_level_operators(case):
    """apply, residual, the Jacobi sweep and the block-Jacobi sweep (from zero and from a guess) on every level"""
    h, levels, lam = case
    rng = np.random.default_rng(11)
    for l, L in enumerate(levels):
        un, fn = rng.standard_normal(L.shape), rng.standard_normal(L.shape)
        u, f, out = h.new_vec(l, un), h.new_vec(l, fn), h.new_vec(l)
        h.apply(l, u, out)
        assert rel_l2(out.download(), A(L, un, lam)) < TOL, ("apply", l)
        h.residual(l, f, u, out)
        assert rel_l2(out.download(), fn - A(L, un, lam)) < TOL, ("residual", l)
        out.copy(u)
        h.smooth_jacobi(l, f, out, 0.8)
        assert rel_l2(out.download(), jacobi(L, fn, un, 0.8, lam)) < TOL, ("jacobi", l)
        out.set(0.0)
        h.smooth(l, f, out)
        assert rel_l2(out.download(), smooth(L, fn, np.zeros(L.shape), lam)) < TOL, ("sweep from zero", l)
        out.copy(u)
        h.smooth(l, f, out)
        assert rel_l2(out.download(), smooth(L, fn, un, lam)) < TOL_GUESS, ("sweep from a guess", l)
        for v in (u, f, out):
            v.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, indirect=True, ids=[_id(c) for c in CASES])
def test_cycles(case):
    """V(1,1) on the three schedules, direct and as a graph, V(2,2) and W against the composed cycle; graph replays are
    bit-identical to direct runs"""
    h, levels, lam = case
    fn = np.random.default_rng(13).standard_normal(levels[0].shape)
    f, u = h.new_vec(0, fn), h.new_vec(0)
    want = cycle(levels, fn, lam)
    for fused in (0, 1, 2):
        got = []
        for graph in (0, 1, 1):
            h.vcycle(f, u, _opts(fused=fused, use_graph=graph))
            got.append(u.download())
            assert rel_l2(got[-1], want) < TOL, (fused, graph)
        assert np.array_equal(got[0], got[1]) and np.array_equal(got[1], got[2]), fused
    h.vcycle(f, u, _opts(pre_sweeps=2, post_sweeps=2))
    assert rel_l2(u.download(), cycle(levels, fn, lam, pre=2, post=2)) < TOL
    h.vcycle(f, u, _opts(cycle_type=1))
    assert rel_l2(u.download(), cycle(levels, fn, lam, cycle_type="W")) < TOL
    f.close(), u.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, indirect=True, ids=[_id(c) for c in CASES])
def test_update_solve_and_krylov(case):
    """vcycle_update from a guess; gmg_solve against the hand-written loop (same cycles, same solution) with its face-only
    residual norm against the full residual; BiCGStab converges on the shifted operator"""
    h, levels, lam = case
    L0 = levels[0]
    rng = np.random.default_rng(17)
    fn, u0 = rng.standard_normal(L0.shape), rng.standard_normal(L0.shape)
    f, u, r, c = h.new_vec(0, fn), h.new_vec(0, u0), h.new_vec(0), h.new_vec(0)
    rel = h.vcycle_update(f, u)
    want = u0 + cycle(levels, fn - A(L0, u0, lam), lam)
    assert rel_l2(u.download(), want) < TOL_GUESS
    full = np.linalg.norm(fn - A(L0, want, lam)) / np.linalg.norm(fn)
    assert abs(rel - full) <= 1e-9 * full + 1e-15
    # gmg_solve vs residual -> cycle -> add
    u.set(0.0)
    its, rel = h.gmg_solve(f, u, tol=1e-10, max_it=60)
    assert rel <= 1e-10
    loop = h.new_vec(0)
    for k in range(61):
        h.residual(0, f, loop, r)
        if r.two_norm() <= 1e-10 * f.two_norm():
            break
        h.vcycle(r, c)
        loop.add(c)
    assert k == its, (k, its)
    assert rel_l2(u.download(), loop.download()) < 1e-9
    u.set(0.0)
    its, rel = h.bicgstab(f, u, tol=1e-10, max_it=200)
    assert rel <= 1e-10, (its, rel)
    assert np.linalg.norm(fn - A(L0, u.download().reshape(L0.shape), lam)) / np.linalg.norm(fn) < 1e-9
    for v in (f, u, r, c, loop):
        v.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", [c for c in CASES if c[4] in (0, 0b111111, 0b1111)], indirect=True,
                         ids=[_id(c) for c in CASES if c[4] in (0, 0b111111, 0b1111)])
def test_fmg(case):
    """FMG with two V(1,1) per level against the composed FMG, with Dirichlet or Neumann boundary data"""
    h, levels, lam = case
    L0 = levels[0]
    neumann = bool(L0.neumann.any())
    src, bdata, _ = problem_data(L0, TRIG3 if L0.D == 3 else TRIG2, neumann)
    fn = src + fold_boundary(L0, bdata)
    f, u, b = h.new_vec(0, fn), h.new_vec(0), h.new_boundary_vec(bdata)
    h.fmg(f, u, b, cycles=2)
    assert rel_l2(u.download(), fmg(levels, fn, bdata, 2, lam)) < TOL
    f.close(), u.close(), b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("D,n", [(3, 16), (2, 32), (3, 32)])
def test_specialised_smoothers_against_the_generic_ones_and_the_smoother_only_state(ctx, D, n):
    """the specialised 16^3 / 2-D 32^2 sweeps equal the size-generic ones; set_lambda(mu != lambda) after set_helmholtz
    runs the general path with (operator lambda, smoother mu); set_helmholtz(0) gives a fresh hierarchy's bytes"""
    mesh_file, divide = ("2refine.bin", 0) if D == 3 else ("2d2ref.bin", 1)
    h, mesh, levels = _mixed_hierarchy(ctx, mesh_file, D, n, divide, 0)
    L0 = levels[0]
    rng = np.random.default_rng(19)
    fn, un = rng.standard_normal(L0.shape), rng.standard_normal(L0.shape)
    f, u = h.new_vec(0, fn), h.new_vec(0)
    h.vcycle(f, u)
    fresh = u.download()
    lam = lam_for(L0, -1.0)
    h.set_helmholtz(lam)
    if n != 32 or D == 2:
        u.upload(un)
        h.smooth(0, f, u)
        spec = u.download()
        h.force_generic_kernels(True)
        u.upload(un)
        h.smooth(0, f, u)
        assert rel_l2(u.download(), spec) < 1e-13
        h.force_generic_kernels(False)
    mu = 0.5 * lam
    h.set_lambda(mu)
    h.vcycle(f, u)
    assert rel_l2(u.download(), cycle(levels, fn, lam, mu=mu)) < TOL_GUESS
    h.set_lambda(lam)
    h.vcycle(f, u)
    assert rel_l2(u.download(), cycle(levels, fn, lam)) < TOL
    h.set_helmholtz(-7.0)
    h.set_helmholtz(0.0)
    h.vcycle(f, u)
    assert np.array_equal(u.download(), fresh)
    for bad in (float("nan"), float("inf"), 1.0):
        with pytest.raises(_pps().TgpuError):
            h.set_helmholtz(bad)
    h.vcycle(f, u)
    assert np.array_equal(u.download(), fresh)  # (unchanged by the rejected calls)
    f.close(), u.close(), h.close(), mesh.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mesh_file,D,n,divide", [("multi_refine.bin", 3, 32, 0), ("multi_refine.bin", 3, 16, 2),
                                                  ("2d_multi_refine_8.bin", 2, 32, 2)])
def test_past_the_resident_grid(ctx, mesh_file, D, n, divide):
    """meshes on which the persistent 32^3 / 16^3 / 2-D 32^2 kernels loop more than once and whose level 0 mixes several
    cell sizes: per-level sweeps and one cycle of each schedule against the composed reference"""
    h, mesh, levels = _mixed_hierarchy(ctx, mesh_file, D, n, divide, 0)
    L0 = levels[0]
    assert np.unique(L0.spacings[:, 0]).size >= 2
    import torch
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    thr = loop_thresholds(D, n, sm)
    key = {32: "smooth3d32c", 16: "smooth3d16"}[n] if D == 3 else "smooth2d32"
    assert L0.P > thr[key][1], (L0.P, thr[key])
    lam = lam_for(L0, -1.0)
    h.set_helmholtz(lam)
    rng = np.random.default_rng(23)
    fn, un = rng.standard_normal(L0.shape), rng.standard_normal(L0.shape)
    f, u = h.new_vec(0, fn), h.new_vec(0, un)
    h.smooth(0, f, u)
    assert rel_l2(u.download(), smooth(L0, fn, un, lam)) < TOL_GUESS
    want = cycle(levels, fn, lam)
    for fused in (0, 1, 2):
        h.vcycle(f, u, _opts(fused=fused))
        assert rel_l2(u.download(), want) < TOL, fused
    f.close(), u.close(), h.close(), mesh.close()


def _profile(ctx, fn):
    ctx.profile_begin()
    fn()
    return [(name, lvl) for name, lvl, _ in ctx.profile_end()]


@pytest.mark.gpu
@pytest.mark.parametrize("mesh_file,D,n,divide", [("2refine.bin", 3, 16, 0), ("2refine.bin", 3, 32, 0), ("2d2ref.bin", 2, 32, 1)])
def test_launch_profile_is_the_poisson_one(ctx, mesh_file, D, n, divide):
    """vcycle_update launches the same kernels at lambda != 0 as at 0: a start from the guess's slices, no full residual on
    level 0, the face-only norm; the smoother-only state shows the fallback it replaces"""
    h, mesh, levels = _mixed_hierarchy(ctx, mesh_file, D, n, divide, 0)
    f = h.new_vec(0, np.random.default_rng(29).standard_normal(levels[0].shape))
    u = h.new_vec(0)
    o = _opts(use_graph=0)
    runs = {}
    for state, lam in (("poisson", 0.0), ("helmholtz", lam_for(levels[0], -1.0)), ("smoother_only", None)):
        if lam is None:  # the same shift in the patch solves only
            h.set_helmholtz(0.0)
            h.set_lambda(runs["lam"])
        else:
            h.set_helmholtz(lam)
            runs["lam"] = lam
        u.set(1.0)
        h.vcycle_update(f, u, o)
        runs[state] = _profile(ctx, lambda: h.vcycle_update(f, u, o))
    assert runs["helmholtz"] == runs["poisson"]
    names = [nm for nm, _ in runs["helmholtz"]]
    assert "extract_faces" in names and "face_residual_norm" in names
    assert ("residual", 0) not in runs["helmholtz"]
    assert runs["smoother_only"] != runs["poisson"]
    f.close(), u.close(), h.close(), mesh.close()


@pytest.mark.gpu
@pytest.mark.parametrize("D", [2, 3])
def test_second_order_accuracy(ctx, D):
    """(Laplacian + lambda) g = f with the trig solution and its Dirichlet values as a boundary vector, h = 1/64 ... 1/512
    (3-D: up to 4096 patches of 32^3, 134 M cells): the discrete solution's error falls about 4x per halving of h, and FMG
    with two cycles per level ends within 1.5x of it.  f is the Poisson initialiser's plus lambda g."""
    pps = _pps()
    lam = -50.0
    mesh_file, prob = ("2d2uni.bin", TRIG2) if D == 2 else ("2uni.bin", TRIG3)
    errs = []
    for divide in (0, 1, 2, 3):
        mesh = pps.Mesh.load(os.path.join(MESHES, mesh_file), D).refine_leaves(divide)
        h = pps.Hierarchy.from_mesh(ctx, mesh, 32)
        h.set_helmholtz(lam)
        L = go.build_hierarchy(os.path.join(MESHES, mesh_file), D, 32, divide)[0]
        f, exact, e = h.new_vec(0), h.new_vec(0), h.new_vec(0)
        h.init_trig_rhs(f, exact)
        f.add_scaled(lam, exact)
        b = h.new_boundary_vec(boundary_values(L, prob, False))
        uh, u = h.new_vec(0), h.new_vec(0)
        its, rel = h.gmg_solve(f, uh, tol=1e-12, max_it=100)
        assert rel <= 1e-12, (its, rel)
        h.fmg(f, u, b, cycles=2)

        def err(v):
            e.copy(v)
            e.add_scaled(-1.0, exact)
            return e.two_norm() / exact.two_norm()

        errs.append((float(L.spacings[:, 0].min()), err(uh), err(u)))
        for v in (f, exact, e, b, uh, u, h, mesh):
            v.close()
    assert errs[-1][0] == 1.0 / 512, errs
    for (_, e0, _), (_, e1, _) in zip(errs, errs[1:]):
        assert 3.0 < e0 / e1 < 5.0, errs
    for _, eh, ef in errs:
        assert ef <= 1.5 * eh, errs


@pytest.mark.gpu
def test_cell_sizes_share_tables_and_past_256_only_poisson(ctx):
    """one multiplier table per cell size: spacings that differ in the last bits share one (the sweeps still match the
    reference); a hierarchy with more than 256 cell sizes is created as before, solves the Poisson problem, and refuses a
    shift with TGPU_ERR_UNSUPPORTED, unchanged"""
    pps = _pps()
    levels = go.build_hierarchy(os.path.join(MESHES, "3uni.bin"), 3, 4, 1)
    fn = np.random.default_rng(31).standard_normal(levels[0].shape)
    lam = lam_for(levels[0], -1.0)
    for rel_step, many in ((2e-16, False), (1e-9, True)):
        mesh = pps.Mesh.load(os.path.join(MESHES, "3uni.bin"), 3).refine_leaves(1)
        nl, descs = mesh.extract_levels(4)
        assert descs[0].npatch > 256
        for p in range(descs[0].npatch):
            for a in range(3):
                descs[0].spacing[p * 3 + a] *= 1.0 + (p % 300 if many else p % 8) * rel_step
        h = pps.Hierarchy(ctx, 3, 4, nl, descs)
        f, u = h.new_vec(0, fn), h.new_vec(0)
        if not many:
            h.set_helmholtz(lam)
            h.vcycle(f, u)
            assert rel_l2(u.download(), cycle(levels, fn, lam)) < TOL
        else:
            h.vcycle(f, u)
            before = u.download()
            assert rel_l2(before, go.cycle(levels, fn)) < 1e-4  # (the spacings moved by up to 3e-7)
            with pytest.raises(pps.TgpuError, match="256"):
                h.set_helmholtz(lam)
            h.set_helmholtz(0.0)
            h.vcycle(f, u)
            assert np.array_equal(u.download(), before)
        f.close(), u.close(), h.close(), mesh.close()


# ---- several GPUs (skipped below two, like tests/test_multi_gpu.py) ----
def _distributed_worker(rank, world, idfile, mesh_file, D, n, divide, f_global, lam, ret):
    """one rank: the distributed hierarchy with set_helmholtz(lam), a V(1,1) direct and as a graph, V(2,2), gmg_solve"""
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
    mesh = pps.Mesh.load(os.path.join(MESHES, mesh_file), D).refine_leaves(divide)
    part = pps.Partition(mesh, n, rank, world, min_patches_per_rank=2)
    h = pps.Hierarchy.from_partition(ctx, part)
    h.set_helmholtz(lam)
    pl = part.level(0)
    nc = n ** D
    f = h.new_vec(0, np.asarray(f_global).reshape(-1, nc)[pl["owned_global"]])
    u, ug, x = h.new_vec(0), h.new_vec(0), h.new_vec(0)
    out = {"owned": pl["owned_global"], "ndist": part.ndist}
    h.vcycle(f, u)
    out["vcycle"] = u.download().reshape(-1, nc)
    g = pps.CycleOpts.default(use_graph=2)  # the exchanges captured in the graph
    h.vcycle(f, ug, g)
    h.vcycle(f, ug, g)
    out["vcycle_graph"] = ug.download().reshape(-1, nc)
    h.vcycle(f, ug, pps.CycleOpts.default(use_graph=2, pre_sweeps=2, post_sweeps=2, coarse_sweeps=2))
    out["vcycle22"] = ug.download().reshape(-1, nc)
    out["its"], out["rel"] = h.gmg_solve(f, x, tol=1e-10, max_it=100)
    out["x"] = x.download().reshape(-1, nc)
    ret[rank] = out
    for v in (f, u, ug, x, h):
        v.close()
    ctx.close()


def run_distributed(world, mesh_file, D, n, divide, f_global, lam):
    """-> (per-rank results, gather(key): the ranks' rows in global patch order)"""
    import tempfile
    import torch.multiprocessing as mp
    mpc = mp.get_context("spawn")
    ret = mpc.Manager().dict()
    with tempfile.TemporaryDirectory() as tmp:
        idfile = os.path.join(tmp, "nccl_id")
        procs = [mpc.Process(target=_distributed_worker, args=(r, world, idfile, mesh_file, D, n, divide, f_global, lam, ret))
                 for r in range(world)]
        for p in procs:
            p.start()
        for p in procs:
            p.join(300)
            assert p.exitcode == 0
    owned = np.concatenate([ret[r]["owned"] for r in range(world)])
    return ret, lambda key: np.concatenate([ret[r][key] for r in range(world)])[np.argsort(owned)]


def check_distributed(ctx, world, mesh_file, D, n, divide):
    levels = go.build_hierarchy(os.path.join(MESHES, mesh_file), D, n, divide)
    lam = lam_for(levels[0], -1.0)
    fn = np.random.default_rng(37).standard_normal(levels[0].shape)
    ret, gather = run_distributed(world, mesh_file, D, n, divide, fn, lam)
    nc = n ** D
    assert rel_l2(gather("vcycle"), cycle(levels, fn, lam).reshape(-1, nc)) < TOL
    assert np.array_equal(gather("vcycle_graph"), gather("vcycle"))
    assert rel_l2(gather("vcycle22"), cycle(levels, fn, lam, pre=2, post=2, coarse_sweeps=2).reshape(-1, nc)) < TOL
    h, mesh, _ = _mixed_hierarchy(ctx, mesh_file, D, n, divide, 0)
    h.set_helmholtz(lam)
    f, x = h.new_vec(0, fn), h.new_vec(0)
    its, rel = h.gmg_solve(f, x, tol=1e-10, max_it=100)
    assert all(ret[r]["its"] == ret[0]["its"] for r in range(world))
    assert abs(ret[0]["its"] - its) <= 1 and ret[0]["rel"] <= 1e-10, (ret[0]["its"], its, ret[0]["rel"])  # (summation order)
    assert rel_l2(gather("x"), x.download().reshape(-1, nc)) < 1e-9
    for v in (f, x, h, mesh):
        v.close()
    return ret


@pytest.mark.gpu
@pytest.mark.parametrize("mesh_file,D,n,divide", [("2refine.bin", 3, 16, 1), ("2refine.bin", 3, 32, 0), ("2d_multi_refine_8.bin", 2, 32, 0)])
def test_distributed_cycle_and_solve(ctx, mesh_file, D, n, divide):
    """the specialised 16^3, 32^3 and 2-D 32^2 sweeps with the in-kernel halo hand-over and the fused schedule on two GPUs
    at lambda != 0: cycles against the composed reference, gmg_solve against the single-GPU solve"""
    import torch
    world = min(torch.cuda.device_count(), 2)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    assert check_distributed(ctx, world, mesh_file, D, n, divide)[0]["ndist"] >= 1
