"""Mixed Dirichlet / Neumann domain sides.

Every patch carries one Neumann bit per side (TgpuLevelDesc::neumann_bits) and the kernels read it side by side: the ghost
closures of the operator, the transform kind per axis of the patch solve, the choice of patches each smoother launch
sweeps, the 32^3 interface slots, and the boundary folds.  With every domain side Dirichlet or every one Neumann, a kernel
that tests "this patch has a Neumann bit" instead of "this side's bit" gives the same answers; the tests here set the
sides one by one.

1. One patch, every one of the 2^(2D) side patterns, every patch size: the operator against its sparse assembly and the
   patch solve against an exact separable solve built from the eigenvectors of the 1-D operators (no transform formulas).
2. Mixed levels of the specialised kernels (16^3, 32^3 and 2-D 32^2 patches) against the oracle: level operators, cycles,
   the update from a guess, the face-only residual norm, FMG with both kinds of boundary data, lambda != 0, and the
   size-generic kernels.
3. Neumann bits that name no domain side are rejected when the hierarchy is created."""
import ctypes as C
import os
from collections import namedtuple

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

import gmg_oracle as go
from conftest import MESHES, rel_l2
from test_fmg import TRIG2, TRIG3, _centres, _mixed_hierarchy, _oracle_kw, boundary_sides, boundary_values, fmg, fold_boundary

TOL = 1e-12
TOL_GENERIC = 1e-13  # the specialised kernels against the size-generic ones: the same arithmetic up to summation order
# A cycle from a random guess at lambda != 0: every patch solve goes through dense n x n transforms (2D of them per sweep)
# on both sides, each with a rounding error up to about sqrt(n) eps = 6e-16 of its input for n = 32.  The first sweep's
# right-hand side is dominated by the interface terms 2 gamma / h^2 of the guess, and the solve divides by eigenvalues down
# to 1 / kappa of the largest, kappa = 1 / sin^2(pi / 2n) = 415, so each side's result carries up to kappa 2D sqrt(n) eps
# = 1.0e-12 (2D) / 1.5e-12 (3D) relative error per sweep.  Two sweeps on the finest level, library and oracle: 6e-12.
# (Measured on a B200 on the 9-level 2-D 32^2 hierarchies: 1.3e-12; the single sweeps from a guess stay below TOL.)
TOL_SHIFTED_GUESS = 1e-11
LAM = -0.75
TGPU_ERR_ARG = 1


# ---- reference: one patch, exact separable solve ----
def axis_operator(n, h, neu_lo, neu_hi):
    """T_a = tridiag(1, -2, 1) / h^2 with end entries -3 (Dirichlet side: ghost = -u) or -1 (Neumann side: ghost = u)"""
    T = np.diag(np.full(n, -2.0)) + np.diag(np.ones(n - 1), 1) + np.diag(np.ones(n - 1), -1)
    T[0, 0] = -1.0 if neu_lo else -3.0
    T[-1, -1] = -1.0 if neu_hi else -3.0
    return T / (h * h)


def axis_sides(bits, a):
    """(Neumann bit of the lower side, of the upper side) of cartesian axis a"""
    return (bits >> (2 * a)) & 1, (bits >> (2 * a + 1)) & 1


def sparse_operator(D, n, h, bits):
    """A = sum_a I (x) T_a (x) I on one patch, in the library's layout (x fastest: numpy axis D - 1 - a is cartesian a)"""
    I = sp.identity(n, format="csr")
    A = None
    for a in range(D):
        mats = [I] * D
        mats[D - 1 - a] = sp.csr_matrix(axis_operator(n, h, *axis_sides(bits, a)))
        term = mats[0]
        for m in mats[1:]:
            term = sp.kron(term, m, format="csr")
        A = term if A is None else A + term
    return A.tocsr()


def separable_solve(D, n, h, bits, lam, f):
    """(A + lam I)^-1 f in fp64 through numpy.linalg.eigh of every T_a.  All sides Neumann: the joint zero mode is dropped,
    (A + lam I)^-1 (f - mean f) with the result's mean zero (the library's patch solve, DftPatchSolver.h:199-201)"""
    x = np.asarray(f, dtype=np.float64).reshape((n,) * D)
    singular = bits == (1 << (2 * D)) - 1
    if singular:
        x = x - x.mean()
    denom = np.full((n,) * D, lam)
    vecs, zero = [], []
    for a in range(D):
        w, V = np.linalg.eigh(axis_operator(n, h, *axis_sides(bits, a)))
        ax = D - 1 - a
        shp = [1] * D
        shp[ax] = n
        denom = denom + w.reshape(shp)
        x = np.moveaxis(np.tensordot(V.T, x, axes=([1], [ax])), 0, ax)
        vecs.append(V)
        zero.append(int(np.argmax(w)))  # (all Neumann: the constant vector, eigenvalue 0)
    if singular:
        idx = tuple(zero[D - 1 - k] for k in range(D))
        x[idx] = 0.0
        denom[idx] = 1.0
    x = x / denom
    for a in range(D):
        ax = D - 1 - a
        x = np.moveaxis(np.tensordot(vecs[a], x, axes=([1], [ax])), 0, ax)
    return x.ravel()


def one_patch_level(D, n, h, bits):
    """the oracle's level of one patch with spacing h and no neighbours"""
    L = go.Level(D, n, 1)
    L.spacings[:] = h
    L.neumann[:] = bits
    return L


PATCH_SIZES = [(D, n) for D in (2, 3) for n in (4, 8, 16, 32)]


# ---- CPU ----
@pytest.mark.parametrize("D,n", [(D, n) for D, n in PATCH_SIZES if n <= 8])
def test_separable_reference_is_the_sparse_solve(D, n):
    h = 1.0 / n
    f = np.random.default_rng(100 + 10 * D + n).standard_normal(n ** D)
    for bits in range(1 << (2 * D)):
        A = sparse_operator(D, n, h, bits)
        for lam in (0.0, LAM):
            u = separable_solve(D, n, h, bits, lam, f)
            if bits == (1 << (2 * D)) - 1:
                # A + lam I restricted to mean-free fields; lam = 0: A is singular, its null space the constants
                g = f - f.mean()
                assert abs(u.mean()) < 1e-12 * np.abs(u).max(), (bits, lam)
                assert rel_l2(A @ u + lam * u, g) < TOL, (bits, lam)
                if lam != 0.0:
                    assert rel_l2(u, spla.spsolve((A + lam * sp.identity(A.shape[0])).tocsc(), g)) < TOL, (bits, lam)
            else:
                assert rel_l2(u, spla.spsolve((A + lam * sp.identity(A.shape[0])).tocsc(), f)) < TOL, (bits, lam)


@pytest.mark.parametrize("D,n", [(D, n) for D, n in PATCH_SIZES if n <= 16])
def test_oracle_closures_match_the_separable_reference(D, n):
    """go.apply_op and go.smooth on one patch, every side pattern, against the sparse assembly and the separable solve"""
    h = 1.0 / n
    rng = np.random.default_rng(200 + 10 * D + n)
    f, u0 = rng.standard_normal(n ** D), rng.standard_normal(n ** D)
    shape = (1,) + (n,) * D
    bad = []
    for bits in range(1 << (2 * D)):
        L = one_patch_level(D, n, h, bits)
        err = rel_l2(go.apply_op(L, u0.reshape(shape)), sparse_operator(D, n, h, bits) @ u0)
        if err >= TOL:
            bad.append((bits, "apply", err))
        for lam in (0.0, LAM):
            err = rel_l2(go.smooth(L, f.reshape(shape), np.zeros(shape), lam), separable_solve(D, n, h, bits, lam, f))
            if err >= TOL:
                bad.append((bits, "smooth lam=%g" % lam, err))
    assert not bad, bad


def test_extracted_and_partitioned_levels_set_neumann_bits_on_domain_sides_only():
    """mesh extraction and the partition mark Neumann sides only where a patch has no neighbour, and no bit >= 2D: the
    hierarchies they describe pass tgpu_hierarchy_create's check"""
    import pressurepoissonsolver_b200 as pps
    for mesh_file, D in (("2refine.bin", 3), ("multi_refine.bin", 3), ("3uni.bin", 3), ("2d2ref.bin", 2), ("2d_multi_refine_8.bin", 2)):
        mesh = pps.Mesh.load(os.path.join(MESHES, mesh_file), D).set_neumann(True)
        levels = mesh.level_arrays(8)
        parts = [pps.Partition(mesh, 8, r, 2, min_patches_per_rank=2) for r in range(2)]
        tables = [(d["neumann"], d["nbr_type"]) for d in levels]
        for part in parts:
            for l in range(part.nlevels):
                pl = part.level(l)
                tables.append((pl["neumann"][:pl["n_owned"]], pl["nbr_type"][:pl["n_owned"]]))
        marked = 0
        for neu, ty in tables:
            assert not np.any(neu >> (2 * D)), mesh_file
            bit = (neu[:, None] >> np.arange(2 * D)) & 1 == 1
            assert not np.any(bit & (ty != go.NBR_NONE)), mesh_file
            assert np.array_equal(bit, ty == go.NBR_NONE), mesh_file  # set_neumann: every domain side
            marked += int(bit.sum())
        assert marked > 0
        for part in parts:
            part.close()
        mesh.close()


# ---- GPU ----
def _pps():
    import pressurepoissonsolver_b200 as pps
    return pps


@pytest.fixture(scope="module")
def ctx():
    c = _pps().Context(0)
    yield c
    c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("D,n", PATCH_SIZES)
def test_one_patch_every_side_pattern(ctx, D, n):
    """apply and residual against the sparse matvec, and a sweep from zero and from a random guess (on one patch the guess
    must not matter) against the separable solve at lambda = 0 and -0.75.  Pattern 0 runs the plain specialised kernels,
    every other the Neumann instantiation of the 16^3 smoother, smooth3d32n_kernel or smooth_kernel's general path"""
    pps = _pps()
    mesh = pps.Mesh.uniform(D, 1)
    nl, descs = mesh.extract_levels(n)
    assert nl == 1 and descs[0].npatch == 1
    h = descs[0].spacing[0]
    rng = np.random.default_rng(300 + 10 * D + n)
    fn, u0 = rng.standard_normal(n ** D), rng.standard_normal(n ** D)
    bad = []
    for bits in range(1 << (2 * D)):
        descs[0].neumann_bits[0] = bits
        hier = pps.Hierarchy(ctx, D, n, 1, descs)
        f, u, out = hier.new_vec(0, fn), hier.new_vec(0, u0), hier.new_vec(0)
        au = sparse_operator(D, n, h, bits) @ u0
        hier.apply(0, u, out)
        bad.append((bits, "apply", rel_l2(out.download(), au)))
        hier.residual(0, f, u, out)
        bad.append((bits, "residual", rel_l2(out.download(), fn - au)))
        for lam in (0.0, LAM):
            hier.set_lambda(lam)
            ref = separable_solve(D, n, h, bits, lam, fn)
            for start, guess in (("zero", np.zeros(n ** D)), ("guess", u0)):
                u.upload(guess)
                hier.smooth(0, f, u)
                bad.append((bits, "smooth from %s, lambda %g" % (start, lam), rel_l2(u.download(), ref)))
        for v in (f, u, out, hier):
            v.close()
    bad = [b for b in bad if not b[2] < TOL]  # (NaN fails)
    mesh.close()
    assert not bad, "%d failures, side patterns %s: %s" % (len(bad), sorted({b[0] for b in bad}), bad[:12])


# mixed levels: mesh, D, n, divide, Neumann side mask; replay: the case also runs the bit-identical replays
Mixed = namedtuple("Mixed", "mesh D n divide mask replay")
M3 = (0b000001, 0b000010, 0b000011, 0b001100, 0b101010, 0b111110)
M2 = (0b0001, 0b0110, 0b1100, 0b1110)
MIXED = [
    # 16^3: 512 uniform patches; coarse/fine faces
    Mixed("3uni.bin", 3, 16, 1, 0b000001, True), Mixed("3uni.bin", 3, 16, 1, 0b001100, False), Mixed("3uni.bin", 3, 16, 1, 0b111110, False),
    Mixed("2refine.bin", 3, 16, 0, 0b000010, False), Mixed("2refine.bin", 3, 16, 0, 0b000011, False), Mixed("2refine.bin", 3, 16, 0, 0b101010, False),
    # 32^3: 64 patches (8 interior); coarse/fine faces; 8 patches that all have a Neumann side under 0b000011
    Mixed("3uni.bin", 3, 32, 0, 0b000001, True), Mixed("3uni.bin", 3, 32, 0, 0b101010, False),
    Mixed("2refine.bin", 3, 32, 0, 0b000010, False), Mixed("2refine.bin", 3, 32, 0, 0b001100, False), Mixed("2refine.bin", 3, 32, 0, 0b111110, False),
    Mixed("2uni.bin", 3, 32, 0, 0b000011, False),
    # 2-D 32^2
    Mixed("2d2ref.bin", 2, 32, 1, 0b0001, True), Mixed("2d2ref.bin", 2, 32, 1, 0b1100, False),
    Mixed("2d_multi_refine_8.bin", 2, 32, 0, 0b0110, False), Mixed("2d_multi_refine_8.bin", 2, 32, 0, 0b1110, False),
]


def _mixed_id(c):
    return "%s_d%d_n%d_%s" % (c.mesh[:-4], c.divide, c.n, format(c.mask, "0%db" % (2 * c.D)))


def test_every_mask_at_every_size():
    for D, n, masks in ((3, 16, M3), (3, 32, M3), (2, 32, M2)):
        assert {c.mask for c in MIXED if (c.D, c.n) == (D, n)} == set(masks), (D, n)
        assert sum(c.replay for c in MIXED if (c.D, c.n) == (D, n)) == 1, (D, n)


@pytest.fixture(scope="module")
def mixed(request, ctx):
    """(case, hierarchy, oracle levels), built once per case"""
    c = request.param
    h, mesh, levels = _mixed_hierarchy(ctx, c.mesh, c.D, c.n, c.divide, c.mask)
    assert [L.P for L in levels] == [h.npatch(l) for l in range(h.nlevels)]
    L0 = levels[0]
    assert 0 < np.count_nonzero(L0.neumann) <= L0.P
    yield c, h, levels
    h.close()
    mesh.close()


def _check(what, got, ref, tol, L):
    """global relative L2 below tol; on failure, the patches that differ most and their Neumann bits"""
    got, ref = np.asarray(got).reshape(L.P, -1), np.asarray(ref).reshape(L.P, -1)
    err = rel_l2(got, ref)
    if err < tol:
        return
    per = np.linalg.norm(got - ref, axis=1) / np.maximum(np.linalg.norm(ref, axis=1), 1e-300)
    worst = np.argsort(per)[::-1][:6]
    pytest.fail("%s: rel L2 %.3e; worst patches: %s" % (
        what, err, "; ".join("%d (bits %s, rel %.3e)" % (p, format(int(L.neumann[p]), "b"), per[p]) for p in worst)))


def _with_lambda(h, lam, fn):
    h.set_lambda(lam)
    try:
        return fn()
    finally:
        h.set_lambda(0.0)


@pytest.mark.gpu
@pytest.mark.parametrize("mixed", MIXED, indirect=True, ids=[_mixed_id(c) for c in MIXED])
def test_mixed_level_operators_vs_oracle(mixed):
    """per level: apply, residual, a sweep from a random guess (also at lambda = -0.75 and with the size-generic kernels)
    and the restriction to the next level"""
    c, h, levels = mixed
    rng = np.random.default_rng(500)
    for l, L in enumerate(levels):
        un, fn = rng.standard_normal(L.shape), rng.standard_normal(L.shape)
        u, f, out = h.new_vec(l, un), h.new_vec(l, fn), h.new_vec(l)
        au = go.apply_op(L, un)
        h.apply(l, u, out)
        _check("apply L%d" % l, out.download(), au, TOL, L)
        spec_apply = out.download()
        h.residual(l, f, u, out)
        _check("residual L%d" % l, out.download(), fn - au, TOL, L)
        h.smooth(l, f, u)
        _check("smooth L%d" % l, u.download(), go.smooth(L, fn, un), TOL, L)
        spec_smooth = u.download()
        h.force_generic_kernels(True)
        try:
            u.upload(un)
            h.apply(l, u, out)
            _check("generic apply L%d" % l, out.download(), spec_apply, TOL_GENERIC, L)
            h.smooth(l, f, u)
            _check("generic smooth L%d" % l, u.download(), spec_smooth, TOL_GENERIC, L)
        finally:
            h.force_generic_kernels(False)
        u.upload(un)
        _with_lambda(h, LAM, lambda: h.smooth(l, f, u))
        _check("smooth L%d lambda %g" % (l, LAM), u.download(), go.smooth(L, fn, un, LAM), TOL, L)
        if l + 1 < len(levels):
            coarse = h.new_vec(l + 1)
            h.restrict(l, f, coarse)
            _check("restrict L%d" % l, coarse.download(), go.restrict(L, levels[l + 1], fn), TOL, levels[l + 1])
            coarse.close()
        for v in (u, f, out):
            v.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mixed", MIXED, indirect=True, ids=[_mixed_id(c) for c in MIXED])
def test_mixed_cycles_vs_oracle(mixed):
    """V(1,1) on the three schedules, direct and as a graph; V(2,2); W; the size-generic kernels; lambda = -0.75; and
    (one case per size) twelve replays alternating graph and direct runs, bit-identical"""
    pps = _pps()
    c, h, levels = mixed
    L0 = levels[0]
    fn = np.random.default_rng(600).standard_normal(L0.shape)
    f, u = h.new_vec(0, fn), h.new_vec(0)
    ref = go.cycle(levels, fn)
    for fused in (1, 2, 0):
        for use_graph in (0, 1):
            h.vcycle(f, u, pps.CycleOpts.default(fused=fused, use_graph=use_graph))
            _check("V(1,1) fused=%d use_graph=%d" % (fused, use_graph), u.download(), ref, TOL, L0)
    spec = u.download()
    h.force_generic_kernels(True)
    try:
        h.vcycle(f, u)
        _check("generic V(1,1)", u.download(), spec, TOL_GENERIC, L0)
    finally:
        h.force_generic_kernels(False)
    if c.replay:
        first = None
        for rep in range(12):
            h.vcycle(f, u, pps.CycleOpts.default(use_graph=rep & 1))
            bits = u.download().tobytes()
            first = first or bits
            assert bits == first, rep
    h.vcycle(f, u, pps.CycleOpts.default(pre_sweeps=2, post_sweeps=2))
    _check("V(2,2)", u.download(), go.cycle(levels, fn, pre=2, post=2), TOL, L0)
    h.vcycle(f, u, pps.CycleOpts.default(cycle_type=1))
    _check("W(1,1)", u.download(), go.cycle(levels, fn, cycle_type="W"), TOL, L0)
    _with_lambda(h, LAM, lambda: h.vcycle(f, u))
    _check("V(1,1) lambda %g" % LAM, u.download(), go.cycle(levels, fn, lam=LAM), TOL, L0)
    f.close()
    u.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mixed", MIXED, indirect=True, ids=[_mixed_id(c) for c in MIXED])
def test_mixed_update_and_face_residual_norm(mixed):
    """vcycle_update from a random guess (also at lambda = -0.75), and gmg_solve's face-only residual norm against the
    full residual of its result"""
    c, h, levels = mixed
    L0 = levels[0]
    rng = np.random.default_rng(700)
    fn, u0 = rng.standard_normal(L0.shape), rng.standard_normal(L0.shape)
    f, u, r = h.new_vec(0, fn), h.new_vec(0, u0), h.new_vec(0)
    h.vcycle_update(f, u)
    _check("vcycle_update", u.download(), u0 + go.cycle(levels, fn - go.apply_op(L0, u0)), TOL, L0)
    u.upload(u0)
    _with_lambda(h, LAM, lambda: h.vcycle_update(f, u))
    _check("vcycle_update lambda %g" % LAM, u.download(), u0 + go.cycle(levels, fn - go.apply_op(L0, u0), lam=LAM), TOL_SHIFTED_GUESS,
           L0)
    fnorm = f.two_norm()
    u.upload(u0)
    for k in (1, 2):
        its, rel = h.gmg_solve(f, u, tol=0.0, max_it=1)
        h.residual(0, f, u, r)
        full = r.two_norm() / fnorm
        assert its == 1 and abs(rel / full - 1) < 1e-10, (k, rel, full)
    for v in (f, u, r):
        v.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mixed", MIXED, indirect=True, ids=[_mixed_id(c) for c in MIXED])
def test_mixed_fmg_vs_oracle(mixed):
    """FMG on the source with Dirichlet values and normal derivatives folded in by fold_boundary, b carrying NaN in every
    Neumann row (FMG reads Dirichlet rows only), against the reference FMG on the true data"""
    pps = _pps()
    c, h, levels = mixed
    L = levels[0]
    prob = TRIG3 if c.D == 3 else TRIG2
    patch, side = boundary_sides(L)
    neu = (L.neumann[patch] >> side) & 1 == 1
    assert neu.any() and not neu.all()
    src = prob["f"](*_centres(L)) * np.ones(L.shape)
    b = np.where(neu[:, None], boundary_values(L, prob, True), boundary_values(L, prob, False))
    bv, f = h.new_boundary_vec(b), h.new_vec(0, src)
    h.fold_boundary(bv, f)
    _check("fold_boundary", f.download(), src + fold_boundary(L, b), 1e-14, L)
    poisoned = b.copy()
    poisoned[neu] = np.nan
    bv.upload(poisoned)
    u = h.new_vec(0)
    o = dict()
    h.fmg(f, u, bv, pps.CycleOpts.default(**o), 1)
    got = u.download()
    assert np.isfinite(got).all()
    _check("FMG", got, fmg(levels, f.download(), b, 1, **_oracle_kw(o)), TOL, L)
    for v in (bv, f, u):
        v.close()


@pytest.mark.gpu
def test_set_lambda_on_a_mixed_32_level_rebuilds_the_cycle(ctx):
    """graph cycles on a mixed 32^3 level, then set_lambda(-0.75), cycles, set_lambda(0), cycles: each result the oracle's
    (set_lambda rebuilds the interface-term buffer and drops the captured graphs)"""
    pps = _pps()
    h, mesh, levels = _mixed_hierarchy(ctx, "2refine.bin", 3, 32, 0, 0b001100)
    L0 = levels[0]
    fn = np.random.default_rng(800).standard_normal(L0.shape)
    f, u = h.new_vec(0, fn), h.new_vec(0)
    ref0, ref_lam = go.cycle(levels, fn), go.cycle(levels, fn, lam=LAM)
    for lam, ref in ((0.0, ref0), (LAM, ref_lam), (0.0, ref0)):
        h.set_lambda(lam)
        for rep in range(2):  # captured, then replayed
            u.set(1.0)  # overwritten
            h.vcycle(f, u, pps.CycleOpts.default(use_graph=1))
            _check("V(1,1) lambda %g, graph run %d" % (lam, rep), u.download(), ref, TOL, L0)
    for v in (f, u, h, mesh):
        v.close()


def _create(ctx, D, n, descs, nl):
    hp = C.c_void_p()
    rc = _pps().lib.tgpu_hierarchy_create(ctx._p, D, n, nl, descs, C.byref(hp))
    if rc == 0:
        _pps().lib.tgpu_hierarchy_destroy(hp)
    else:
        assert not hp.value
    return rc


@pytest.mark.gpu
@pytest.mark.parametrize("D", (2, 3))
def test_neumann_bits_off_the_domain_boundary_are_rejected(ctx, D):
    """a Neumann bit on a side with a neighbour, or a bit >= 2D, on any level: TGPU_ERR_ARG; every domain side is fine"""
    pps = _pps()
    mesh = pps.Mesh.load(os.path.join(MESHES, "2refine.bin" if D == 3 else "2d2ref.bin"), D)
    arrays = mesh.level_arrays(8)  # copies of the tables; the extraction below is the one whose descriptors are passed
    nl, descs = mesh.extract_levels(8)
    assert nl >= 2
    for l in range(nl):
        ty = arrays[l]["nbr_type"]
        for p in range(descs[l].npatch):
            descs[l].neumann_bits[p] = int(np.sum((ty[p] == go.NBR_NONE) << np.arange(2 * D)))
    assert _create(ctx, D, 8, descs, nl) == 0
    for l in (0, 1):
        ty = arrays[l]["nbr_type"]
        assert np.any(ty != go.NBR_NONE), l
        p, s = map(int, np.argwhere(ty != go.NBR_NONE)[0])
        keep = descs[l].neumann_bits[p]
        descs[l].neumann_bits[p] = keep | (1 << s)
        assert _create(ctx, D, 8, descs, nl) == TGPU_ERR_ARG, (l, p, s)
        assert b"side with a neighbour" in pps.lib.tgpu_last_error()
        descs[l].neumann_bits[p] = keep | (1 << (2 * D))
        assert _create(ctx, D, 8, descs, nl) == TGPU_ERR_ARG, (l, p)
        assert b"past side" in pps.lib.tgpu_last_error()
        descs[l].neumann_bits[p] = keep
    assert _create(ctx, D, 8, descs, nl) == 0
    mesh.close()


@pytest.mark.gpu
def test_rejected_neumann_bits_release_the_levels_already_uploaded(ctx):
    import torch
    pps = _pps()
    mesh = pps.Mesh.uniform(3, 5)
    nl, descs = mesh.extract_levels(32)
    assert descs[0].npatch >= 4096 and nl >= 2
    descs[1].neumann_bits[0] = 1 << 6  # found after level 0's 0.4 GB of face buffers are on the device

    def free_bytes():
        ctx.sync()
        return torch.cuda.mem_get_info(0)[0]

    before = free_bytes()
    for _ in range(8):
        assert _create(ctx, 3, 32, descs, nl) == TGPU_ERR_ARG
    assert before - free_bytes() < 1 << 30
    mesh.close()
