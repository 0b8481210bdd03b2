"""Full multigrid (tgpu_fmg) and caller-supplied boundary data (tgpu_boundary_sides, tgpu_boundary_vec_create,
tgpu_fold_boundary).

The FMG reference below is composed from the oracle's pinned pieces (restrict, interpolate_trilinear, smooth, apply_op,
cycle): boundary data lives in the library's layout, one row of n^(D-1) face values per domain-boundary side of level 0
in ascending (patch, side) order, and the coarse right-hand sides re-pose the Dirichlet folds for the coarse spacing."""
import os
import sys
import tempfile

import numpy as np
import pytest

import gmg_oracle as go
from conftest import GOLDEN_CASES, MESHES, ROOT, load_golden, rel_l2

TOL = 1e-12


# ---- reference: boundary data and FMG on the oracle's levels ----
def boundary_sides(L):
    """the domain-boundary sides of L, ascending (patch, side): tgpu_boundary_sides"""
    p, s = np.nonzero(L.nbr_type == go.NBR_NONE)
    return p.astype(np.int32), s.astype(np.int8)


def _centres(L):
    """cell-centre coordinates, one array of L.shape per axis"""
    k = np.arange(L.n)
    out = []
    for a in range(L.D):
        c = L.starts[:, a, None] + L.spacings[:, a, None] / 2.0 + L.spacings[:, a, None] * k[None, :]
        shp = [L.P] + [1] * L.D
        shp[L.D - a] = L.n
        out.append(np.broadcast_to(c.reshape(shp), L.shape))
    return out


def face_coords(L):
    """coordinates of the face centres of every boundary side: D arrays [count, n^(D-1)] in face order"""
    patch, side = boundary_sides(L)
    cen = _centres(L)
    out = [np.empty((patch.size, L.n ** (L.D - 1))) for _ in range(L.D)]
    for s in range(2 * L.D):
        k = np.nonzero(side == s)[0]
        if not k.size:
            continue
        p, a = patch[k], s // 2
        for b in range(L.D):
            if b == a:
                edge = L.starts[p, a] + (L.spacings[p, a] * L.n if s % 2 else 0.0)
                out[b][k] = edge[:, None]
            else:
                out[b][k] = go.face(cen[b], L.D, s)[p].reshape(k.size, -1)
    return out


def fold_boundary(L, b, dirichlet_only=False):
    """the boundary terms of b as an addition to f: -2 b / h^2 on Dirichlet sides, -b / h on Neumann sides
    (dirichlet_only: Neumann sides contribute nothing)"""
    patch, side = boundary_sides(L)
    out = np.zeros(L.shape)
    b = np.asarray(b).reshape(patch.size, -1)
    for s in range(2 * L.D):
        k = np.nonzero(side == s)[0]
        if not k.size:
            continue
        p = patch[k]
        h = L.spacings[p, s // 2][:, None]
        neu = ((L.neumann[p] >> s) & 1 == 1)[:, None]
        term = np.where(neu, 0.0 if dirichlet_only else -b[k] / h, -2 * b[k] / (h * h))
        fv = go.face(out, L.D, s)
        fv[p] += term.reshape(fv[p].shape)
    return out


def restrict_boundary(fine, coarse, b):
    """the coarse level's boundary data: the mean of the 2^(D-1) fine face values over each coarse face cell (a patch on
    both levels copies)"""
    D, n = fine.D, fine.n
    fp, fs = boundary_sides(fine)
    cp, cs = boundary_sides(coarse)
    fshape = (n,) * (D - 1)
    B = np.full((fine.P, 2 * D) + fshape, np.nan)
    B[fp, fs] = np.asarray(b).reshape((fp.size,) + fshape)
    C = np.full((coarse.P, 2 * D) + fshape, np.nan)
    for p, s in zip(fp, fs):
        pc, orth = fine.parent_idx[p], fine.orth_on_parent[p]
        if orth < 0:
            C[pc, s] = B[p, s]
            continue
        F = B[p, s]
        rem = [a for a in reversed(range(D)) if a != s // 2]  # cartesian axis of each face dimension
        if D == 2:
            blk = (F[0::2] + F[1::2]) / 2
        else:
            blk = (F[0::2, 0::2] + F[0::2, 1::2] + F[1::2, 0::2] + F[1::2, 1::2]) / 4
        sl = tuple(slice(((orth >> a) & 1) * (n // 2), ((orth >> a) & 1) * (n // 2) + n // 2) for a in rem)
        C[pc, s][sl] = blk
    out = C[cp, cs].reshape(cp.size, -1)
    assert not np.isnan(out).any()
    return out


def restrict_rhs(fine, coarse, f, b):
    """(f_c, b_c): R f with the Dirichlet folds re-posed for the coarse spacing, R f + fold_c(b_c) - R fold_f(b)"""
    fc = go.restrict(fine, coarse, f)
    if b is None:
        return fc, None
    bc = restrict_boundary(fine, coarse, b)
    return fc + fold_boundary(coarse, bc, True) - go.restrict(fine, coarse, fold_boundary(fine, b, True)), bc


def fmg(levels, f, b, cycles, cycle_type="V", pre=1, post=1, mid=1, coarse_sweeps=1, max_levels=0, patches_per_proc=0.0,
        lam=0.0, interp=None):
    """full multigrid over go.active_levels: right-hand sides restricted down, coarse_sweeps sweeps from zero on the
    coarsest level, then per level the linear interpolation of the coarser result and `cycles` cycles from it"""
    lv = go.active_levels(levels, max_levels, patches_per_proc)
    fs, bs = [np.asarray(f).reshape(lv[0].shape)], [b]
    for l in range(len(lv) - 1):
        fc, bc = restrict_rhs(lv[l], lv[l + 1], fs[l], bs[l])
        fs.append(fc)
        bs.append(bc)
    u = np.zeros(lv[-1].shape)
    for _ in range(coarse_sweeps):
        u = go.smooth(lv[-1], fs[-1], u, lam)
    for l in range(len(lv) - 2, -1, -1):
        u = go.interpolate_trilinear(lv[l], lv[l + 1], u, np.zeros(lv[l].shape))
        for _ in range(cycles):
            u = u + go.cycle(lv[l:], fs[l] - go.apply_op(lv[l], u), cycle_type, pre, post, mid, coarse_sweeps, lam=lam, interp=interp)
    return u


# manufactured problems (apps/3d/steady.cpp, apps/2d/steady.cpp): exact solution, source, gradient
def _x3(x, y, z):
    return x + .3, y + .3, z + .3


TRIG3 = dict(g=go._g3, f=go._f3, dg=[
    lambda x, y, z: (lambda X, Y, Z: np.pi * np.cos(np.pi * X) * np.cos(2.0 / 3 * np.pi * Y) * np.sin(5.0 / 6 * np.pi * Z))(*_x3(x, y, z)),
    lambda x, y, z: (lambda X, Y, Z: -2.0 / 3 * np.pi * np.sin(np.pi * X) * np.sin(2.0 / 3 * np.pi * Y) * np.sin(5.0 / 6 * np.pi * Z))(*_x3(x, y, z)),
    lambda x, y, z: (lambda X, Y, Z: 5.0 / 6 * np.pi * np.sin(np.pi * X) * np.cos(2.0 / 3 * np.pi * Y) * np.cos(5.0 / 6 * np.pi * Z))(*_x3(x, y, z))])
GAUSS3 = dict(
    g=lambda x, y, z: np.exp(np.cos(10 * np.pi * x)) - np.exp(np.cos(11 * np.pi * y)) + np.exp(np.cos(12 * np.pi * z)),
    f=lambda x, y, z: -np.pi * np.pi * (100 * np.exp(np.cos(10 * np.pi * x)) * np.cos(10 * np.pi * x) - 100 * np.exp(np.cos(10 * np.pi * x)) * np.sin(10 * np.pi * x) ** 2
                                        - 121 * np.exp(np.cos(11 * np.pi * y)) * np.cos(11 * np.pi * y) + 121 * np.exp(np.cos(11 * np.pi * y)) * np.sin(11 * np.pi * y) ** 2
                                        + 144 * np.exp(np.cos(12 * np.pi * z)) * np.cos(12 * np.pi * z) - 144 * np.exp(np.cos(12 * np.pi * z)) * np.sin(12 * np.pi * z) ** 2),
    dg=[lambda x, y, z: -10 * np.pi * np.sin(10 * np.pi * x) * np.exp(np.cos(10 * np.pi * x)),
        lambda x, y, z: 11 * np.pi * np.sin(11 * np.pi * y) * np.exp(np.cos(11 * np.pi * y)),
        lambda x, y, z: -12 * np.pi * np.sin(12 * np.pi * z) * np.exp(np.cos(12 * np.pi * z))])
TRIG2 = dict(g=go._g2, f=go._f2, dg=[lambda x, y: -2 * np.pi * np.sin(np.pi * y) * np.sin(2 * np.pi * x),
                                     lambda x, y: np.pi * np.cos(np.pi * y) * np.cos(2 * np.pi * x)])


def boundary_values(L, prob, neumann):
    """the boundary data of a problem: Dirichlet values or outward normal derivatives on the boundary face centres"""
    fc = face_coords(L)
    _, side = boundary_sides(L)
    if neumann:
        sign = np.where(side % 2 == 1, 1.0, -1.0)[:, None]
        b = np.empty_like(fc[0])
        for a in range(L.D):
            k = side // 2 == a
            b[k] = sign[k] * prob["dg"][a](*[c[k] for c in fc])
    else:
        b = prob["g"](*fc)
    return b


def problem_data(L, prob, neumann):
    """(source at the cell centres, boundary data, exact solution)"""
    cen = _centres(L)
    return prob["f"](*cen) * np.ones(L.shape), boundary_values(L, prob, neumann), prob["g"](*cen) * np.ones(L.shape)


# ---- CPU ----
@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_fold_reproduces_the_reference_dirichlet_init(name):
    """source + fold of the exact solution on the boundary face centres = Init::initDirichlet's right-hand side"""
    g = load_golden(name)
    D = int(g["D"])
    L = go.build_hierarchy(os.path.join(MESHES, str(g["mesh"])), D, int(g["n"]), int(g["divide"]))[0]
    src, b, exact = problem_data(L, TRIG3 if D == 3 else TRIG2, False)
    assert rel_l2(src + fold_boundary(L, b), g["rhs_f"]) < 1e-14
    assert rel_l2(exact, g["rhs_exact"]) < 1e-14


@pytest.mark.parametrize("name,prob", [("3d_2refine_n8_neumann_init", "trig"), ("3d_2refine_n8_neumann_init", "gauss"),
                                       ("2d_2d2ref_d1_n8_neumann_init", "trig")])
def test_fold_reproduces_the_reference_neumann_init(name, prob):
    """source + fold of the outward normal derivative = Init::initNeumann's right-hand side"""
    g = load_golden(name)
    D = int(g["D"])
    L = go.build_hierarchy(os.path.join(MESHES, str(g["mesh"])), D, int(g["n"]), int(g["divide"]), neumann=True)[0]
    src, b, _ = problem_data(L, {"trig": TRIG3 if D == 3 else TRIG2, "gauss": GAUSS3}[prob], True)
    assert rel_l2(src + fold_boundary(L, b), g["f_" + prob]) < 1e-14


@pytest.mark.parametrize("mesh_file,D,n,divide,neumann", [("2refine.bin", 3, 8, 0, False), ("multi_refine.bin", 3, 4, 0, False),
                                                          ("2d2ref.bin", 2, 8, 1, False), ("2refine.bin", 3, 8, 0, True),
                                                          ("2d2ref.bin", 2, 8, 1, True)])
def test_restricted_rhs_is_the_coarse_problem(mesh_file, D, n, divide, neumann):
    """restrict_rhs of the folded f = the unfolded source restricted, folded with the restricted boundary data (Neumann:
    R f itself, the Neumann folds restrict consistently)"""
    levels = go.build_hierarchy(os.path.join(MESHES, mesh_file), D, n, divide, neumann=neumann)
    rng = np.random.default_rng(12)
    fine, coarse = levels[0], levels[1]
    src = rng.standard_normal(fine.shape)
    b = rng.standard_normal((boundary_sides(fine)[0].size, n ** (D - 1)))
    fc, bc = restrict_rhs(fine, coarse, src + fold_boundary(fine, b), b)
    want = go.restrict(fine, coarse, src) + fold_boundary(coarse, restrict_boundary(fine, coarse, b))
    assert rel_l2(fc, want) < 1e-14
    if neumann:
        assert rel_l2(go.restrict(fine, coarse, src + fold_boundary(fine, b)), want) < 1e-14
    # two levels down: the restricted data restricts again
    fc2, _ = restrict_rhs(coarse, levels[2], fc, bc)
    src2 = go.restrict(coarse, levels[2], go.restrict(fine, coarse, src))
    want2 = src2 + fold_boundary(levels[2], restrict_boundary(coarse, levels[2], bc))
    assert rel_l2(fc2, want2) < 1e-14


def test_fmg_on_one_level_is_the_coarse_solve():
    levels = go.build_hierarchy(os.path.join(MESHES, "2refine.bin"), 3, 4, 0)
    f = np.random.default_rng(3).standard_normal(levels[0].shape)
    u = fmg(levels, f, None, 2, max_levels=1)
    assert np.array_equal(u, go.smooth(levels[0], f, np.zeros(levels[0].shape)))


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


@pytest.mark.gpu
@pytest.mark.parametrize("mesh_file,D,n,divide,neumann,prob", [
    ("2refine.bin", 3, 8, 0, False, "trig"), ("multi_refine.bin", 3, 4, 0, False, "trig"), ("2d2ref.bin", 2, 8, 1, False, "trig"),
    ("2refine.bin", 3, 32, 0, False, "trig"), ("2refine.bin", 3, 8, 0, True, "trig"), ("2refine.bin", 3, 8, 0, True, "gauss"),
    ("2d2ref.bin", 2, 8, 1, True, "trig")])
def test_fold_boundary_equals_the_manufactured_initialisers(ctx, mesh_file, D, n, divide, neumann, prob):
    h, mesh = _build(ctx, mesh_file, D, n, divide, neumann)
    L = go.build_hierarchy(os.path.join(MESHES, mesh_file), D, n, divide, neumann=neumann)[0]
    patch, side = h.boundary_sides()
    want_p, want_s = boundary_sides(L)
    assert np.array_equal(patch, want_p) and np.array_equal(side, want_s)
    src, b, _ = problem_data(L, {"trig": TRIG3 if D == 3 else TRIG2, "gauss": GAUSS3}[prob], neumann)
    bv, f, ref = h.new_boundary_vec(b), h.new_vec(0, src), h.new_vec(0)
    assert bv.ncells == b.size
    h.fold_boundary(bv, f)
    if neumann:
        h.init_neumann_rhs(ref, problem=prob)
    else:
        h.init_trig_rhs(ref)
    assert rel_l2(f.download(), ref.download()) < 1e-14
    assert rel_l2(bv.download(), b.ravel()) == 0.0
    h.close()
    mesh.close()


def _oracle_kw(o):
    return dict(cycle_type="W" if o.get("cycle_type", 0) == 1 else "V", pre=o.get("pre_sweeps", 1), post=o.get("post_sweeps", 1),
                coarse_sweeps=o.get("coarse_sweeps", 1), max_levels=o.get("max_levels", 0),
                interp=go.interpolate_trilinear if o.get("interpolator", 0) == 1 else None)


def _trig_problem(h, L, neumann):
    """the manufactured trig problem on the device: f with its boundary data folded in, and that data (None: Neumann)"""
    f = h.new_vec(0)
    if neumann:
        h.init_neumann_rhs(f)
        return f, None, None
    h.init_trig_rhs(f)
    b = boundary_values(L, TRIG3 if L.D == 3 else TRIG2, False)
    return f, h.new_boundary_vec(b), b


FMG_OPTS = [(dict(), 1), (dict(), 2), (dict(pre_sweeps=2, post_sweeps=2), 2), (dict(cycle_type=1), 2), (dict(max_levels=3), 2),
            (dict(fused=0), 2), (dict(fused=2), 2), (dict(interpolator=1), 2), (dict(coarse_sweeps=2), 1)]
FMG_CASES = [("2refine.bin", 3, 8, 0, False, FMG_OPTS), ("2d2ref.bin", 2, 8, 1, False, FMG_OPTS),
             ("multi_refine.bin", 3, 4, 0, False, FMG_OPTS), ("2refine.bin", 3, 32, 0, False, [(dict(), 2)]),
             ("2refine.bin", 3, 8, 0, True, [(dict(), 2), (dict(fused=0), 1)])]


@pytest.mark.gpu
@pytest.mark.parametrize("mesh_file,D,n,divide,neumann,opts", FMG_CASES)
def test_fmg_vs_oracle(ctx, mesh_file, D, n, divide, neumann, opts):
    """tgpu_fmg against the reference FMG, with CUDA-graph replays bit-identical to direct runs"""
    pps = _pps()
    h, mesh = _build(ctx, mesh_file, D, n, divide, neumann)
    levels = go.build_hierarchy(os.path.join(MESHES, mesh_file), D, n, divide, neumann=neumann)
    f, bv, b = _trig_problem(h, levels[0], neumann)
    fn = f.download()
    u = h.new_vec(0)
    for o, cycles in opts:
        ref = fmg(levels, fn, b, cycles, **_oracle_kw(o)).ravel()
        direct = None
        for use_graph in (0, 1, 1):
            u.set(1.0)  # overwritten
            h.fmg(f, u, bv, pps.CycleOpts.default(use_graph=use_graph, **o), cycles)
            got = u.download()
            assert rel_l2(got, ref) < TOL, (o, cycles, rel_l2(got, ref))
            if direct is None:
                direct = got
            assert np.array_equal(got, direct), (o, cycles)
    h.close()
    mesh.close()


@pytest.mark.gpu
def test_fmg_with_a_shifted_patch_solve_vs_oracle(ctx):
    pps = _pps()
    h, mesh = _build(ctx, "2refine.bin", 3, 8, 0)
    h.set_lambda(-0.75)
    levels = go.build_hierarchy(os.path.join(MESHES, "2refine.bin"), 3, 8, 0)
    f, bv, b = _trig_problem(h, levels[0], False)
    u = h.new_vec(0)
    for o in (dict(), dict(use_graph=0)):
        h.fmg(f, u, bv, pps.CycleOpts.default(**o), 2)
        ref = fmg(levels, f.download(), b, 2, lam=-0.75).ravel()
        err = rel_l2(u.download(), ref)
        print("lambda = -0.75, %s: rel-L2 against the reference FMG %.3e" % (o, err))
        assert err < TOL, o
    h.close()
    mesh.close()


def _mixed_hierarchy(ctx, mesh_file, D, n, divide, keep_bits):
    """a hierarchy whose domain sides are Neumann where keep_bits has the side's bit, Dirichlet elsewhere, and the oracle's
    levels with the same sides"""
    pps = _pps()
    mesh = pps.Mesh.load(os.path.join(MESHES, mesh_file), D).set_neumann(True).refine_leaves(divide)
    nl, descs = mesh.extract_levels(n)
    for l in range(nl):
        for p in range(descs[l].npatch):
            descs[l].neumann_bits[p] &= keep_bits
    h = pps.Hierarchy(ctx, D, n, nl, descs)
    levels = go.build_hierarchy(os.path.join(MESHES, mesh_file), D, n, divide, neumann=True)
    for L in levels:
        L.neumann &= keep_bits
    return h, mesh, levels


@pytest.mark.gpu
@pytest.mark.parametrize("mesh_file,D,n,divide,keep_bits", [("2refine.bin", 3, 8, 0, 0b000001), ("2refine.bin", 3, 8, 0, 0b101101),
                                                            ("2d2ref.bin", 2, 8, 1, 0b0110), ("2refine.bin", 3, 8, 0, 0b111111)])
def test_fmg_on_mixed_boundaries_reads_no_neumann_data(ctx, mesh_file, D, n, divide, keep_bits):
    """Dirichlet and Neumann domain sides on one mesh (all Neumann for keep_bits = all sides): f is the source with both
    kinds of data folded in by tgpu_fold_boundary, b carries NaN in every Neumann row, and the result equals the reference
    FMG on the true data (with no Dirichlet side, FMG with and without that b are bit-identical)"""
    pps = _pps()
    h, mesh, levels = _mixed_hierarchy(ctx, mesh_file, D, n, divide, keep_bits)
    L = levels[0]
    prob = TRIG3 if D == 3 else TRIG2
    patch, side = boundary_sides(L)
    neu = (L.neumann[patch] >> side) & 1 == 1
    src = prob["f"](*_centres(L)) * np.ones(L.shape)
    b = np.where(neu[:, None], boundary_values(L, prob, True), boundary_values(L, prob, False))
    want_f = src + fold_boundary(L, b)
    bv, f = h.new_boundary_vec(b), h.new_vec(0, src)
    h.fold_boundary(bv, f)
    assert rel_l2(f.download(), want_f) < 1e-14
    poisoned = b.copy()
    poisoned[neu] = np.nan
    bv.upload(poisoned)
    u = h.new_vec(0)
    for o, cycles in ((dict(), 2), (dict(fused=0), 1)):
        ref = fmg(levels, f.download(), b, cycles, **_oracle_kw(o)).ravel()
        h.fmg(f, u, bv, pps.CycleOpts.default(**o), cycles)
        got = u.download()
        assert np.isfinite(got).all() and rel_l2(got, ref) < TOL, (o, rel_l2(got, ref))
        if neu.all():
            h.fmg(f, u, None, pps.CycleOpts.default(**o), cycles)
            assert np.array_equal(u.download(), got), o
    h.close()
    mesh.close()


@pytest.mark.gpu
def test_fused_fmg_does_no_full_passes(ctx):
    h, mesh = _build(ctx, "2refine.bin", 3, 16, 0)
    L = go.build_hierarchy(os.path.join(MESHES, "2refine.bin"), 3, 16, 0)[0]
    f, bv, _ = _trig_problem(h, L, False)
    u = h.new_vec(0)
    for cycles in (1, 2, 3):  # (from the second cycle on a level, the previous cycle's last sweep emits the slices)
        ctx.profile_begin()
        h.fmg(f, u, bv, cycles=cycles)
        prof = ctx.profile_end()
        names = [k for k, _, _ in prof]
        assert not {"extract_faces", "apply", "residual", "residual_restrict", "blas1"} & set(names), (cycles, names)
        assert names.count("restrict_rhs") == h.nlevels - 1 and names.count("fmg_interp") == h.nlevels - 1, names
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
    b, b_other = h.new_boundary_vec(), h2.new_boundary_vec()
    calls = [lambda: h.fmg(u, u), lambda: h.fmg(coarse, u), lambda: h.fmg(f, coarse), lambda: h.fmg(other, u),
             lambda: h.fmg(f, other), lambda: h.fmg(f, u, b_other), lambda: h.fmg(f, u, f), lambda: h.fmg(b, u),
             lambda: h.fmg(f, u, cycles=0), lambda: h.fmg(f, u, opts=pps.CycleOpts.default(pre_sweeps=-1)),
             lambda: h.fold_boundary(f, u), lambda: h.fold_boundary(b_other, u)]
    for call in calls:
        with pytest.raises(pps.TgpuError):
            call()
        assert np.array_equal(u.download(), u0)
    # a boundary vector is no level vector
    for call in (lambda: h.apply(0, b, u), lambda: h.vcycle(b, u), lambda: u.copy(b), lambda: h.integrate(b)):
        with pytest.raises(pps.TgpuError):
            call()
    b.upload(np.arange(b.ncells, dtype=np.float64))
    b.scale(2.0)
    assert b.two_norm() == pytest.approx(2 * np.linalg.norm(np.arange(b.ncells)), rel=1e-14)
    for v in (h, h2, mesh, mesh2):
        v.close()


@pytest.mark.gpu
def test_fmg_reaches_discretisation_accuracy(ctx):
    """trig Dirichlet problem on uniform meshes of 16^3 patches, h = 1/128 ... 1/1024: with two V(1,1) per level the
    FMG error against the exact solution stays within a fixed factor of the discrete solution's, and both fall as h^2.
    Without the boundary data (b = None) the coarse problems carry the wrong boundary values and the bound fails.
    The cycles = 2 ratio is not h-independent over these resolutions (DESIGN 3.7: measured on a B200 it grows from 0.80
    at h = 1/128 to 1.07 at h = 1/1024), so what is asserted is that it stays below 1.5 and that the algebraic error
    ||u_FMG - u_h|| stays below the discretisation error ||u_h - u||.  cycles = 1 is reported, not asserted: one V(1,1)
    with a contraction of about 0.32 > 1/4 per level gives no h-independent bound."""
    rows = []
    for divide in (0, 1, 2, 3):
        h, mesh = _build(ctx, "4uni.bin", 3, 16, divide)
        f, exact, e = h.new_vec(0), h.new_vec(0), h.new_vec(0)
        h.init_trig_rhs(f, exact)
        L = go.build_hierarchy(os.path.join(MESHES, "4uni.bin"), 3, 16, divide)[0]
        bdata = boundary_values(L, TRIG3, False)
        b = h.new_boundary_vec(bdata)
        del bdata

        def err(u):
            e.copy(u)
            e.add_scaled(-1.0, exact)
            return e.two_norm() / exact.two_norm()

        uh = h.new_vec(0)
        its, rel = h.gmg_solve(f, uh, tol=1e-12, max_it=100)
        assert rel <= 1e-10, (its, rel)
        row = {"divide": divide, "err_h": err(uh)}
        for cycles in (1, 2):
            u = h.new_vec(0)
            h.fmg(f, u, b, cycles=cycles)
            row["err_fmg%d" % cycles] = err(u)
            e.copy(u)
            e.add_scaled(-1.0, uh)
            row["alg_fmg%d" % cycles] = e.two_norm() / exact.two_norm()  # ||u_FMG - u_h||: the algebraic error left
            h.fmg(f, u, None, cycles=cycles)
            row["err_fmg%d_no_b" % cycles] = err(u)
            u.close()
        rows.append(row)
        for v in (f, exact, e, uh, b, h, mesh):
            v.close()
    for r in rows:
        print("divide %d: ||u_h - u|| %.3e; FMG/u_h error ratio: cycles=1 %.3f, cycles=2 %.3f; without b: %.3f, %.3f; "
              "||u_FMG - u_h|| / ||u_h - u||: cycles=1 %.3f, cycles=2 %.3f"
              % (r["divide"], r["err_h"], r["err_fmg1"] / r["err_h"], r["err_fmg2"] / r["err_h"], r["err_fmg1_no_b"] / r["err_h"],
                 r["err_fmg2_no_b"] / r["err_h"], r["alg_fmg1"] / r["err_h"], r["alg_fmg2"] / r["err_h"]))
    ratio = [r["err_fmg2"] / r["err_h"] for r in rows]
    alg = [r["alg_fmg2"] / r["err_h"] for r in rows]
    assert max(ratio) < 1.5, ratio
    # FMG ends at discretisation accuracy: the algebraic error it leaves stays below the discretisation error
    assert max(alg) < 1.0, alg
    for a, c in zip(rows, rows[1:]):
        assert 3.5 <= a["err_fmg2"] / c["err_fmg2"] <= 4.5, (a, c)
    assert rows[-1]["err_fmg2_no_b"] / rows[-1]["err_h"] > 2.0, rows


# ---- several GPUs (worker pattern of test_gmg_solve.test_distributed_solve_matches_single_gpu) ----
def _ngpu():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


def _worker(rank, world, idfile, mesh_file, D, n, divide, f_global, b_global, ret):
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
    mesh.refine_leaves(divide)
    part = pps.Partition(mesh, n, rank, world, min_patches_per_rank=2)
    h = pps.Hierarchy.from_partition(ctx, part)
    pl = part.level(0)
    nc = n ** D
    owned = pl["owned_global"]
    f, u = h.new_vec(0, np.asarray(f_global).reshape(-1, nc)[owned]), h.new_vec(0)
    # this rank's boundary sides are those of its owned patches, in the same (patch, side) order as the global list
    patch, side = h.boundary_sides()
    bg = b_global
    rows = [bg[(int(owned[p]), int(s))] for p, s in zip(patch, side)]
    b = h.new_boundary_vec(np.array(rows))
    h.fmg(f, u, b)
    ret[rank] = {"owned": owned, "ndist": part.ndist, "u": u.download().reshape(-1, nc)}
    h.close()
    ctx.close()


@pytest.mark.gpu
def test_distributed_fmg_matches_single_gpu(ctx):
    world = min(_ngpu(), 2)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    mesh_file, D, n, divide = "2refine.bin", 3, 16, 1
    h, mesh = _build(ctx, mesh_file, D, n, divide)
    L = go.build_hierarchy(os.path.join(MESHES, mesh_file), D, n, divide)[0]
    f, bv, b = _trig_problem(h, L, False)
    u = h.new_vec(0)
    h.fmg(f, u, bv)
    single = u.download().reshape(-1, n ** D)
    fn = f.download()
    patch, side = boundary_sides(L)
    bmap = {(int(p), int(s)): b[k] for k, (p, s) in enumerate(zip(patch, side))}
    h.close()
    mesh.close()
    mpc = mp.get_context("spawn")
    ret = mpc.Manager().dict()
    with tempfile.TemporaryDirectory() as tmp:
        idfile = os.path.join(tmp, "nccl_id")
        procs = [mpc.Process(target=_worker, args=(r, world, idfile, mesh_file, D, n, divide, fn, bmap, ret)) for r in range(world)]
        for p in procs:
            p.start()
        for p in procs:
            p.join(300)
            assert p.exitcode == 0
    owned = np.concatenate([ret[r]["owned"] for r in range(world)])
    gathered = np.concatenate([ret[r]["u"] for r in range(world)])[np.argsort(owned)]
    assert ret[0]["ndist"] >= 1
    print("distributed FMG vs single GPU: rel-L2 %.3e, bit-identical: %s" % (rel_l2(gathered, single), np.array_equal(gathered, single)))
    assert rel_l2(gathered, single) < 1e-12
