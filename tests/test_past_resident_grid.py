"""Persistent kernels past their resident grid, against the oracle.

Almost every hot kernel is persistent: the host clamps its grid to what the GPU holds at once, and each CTA (or 2-CTA
cluster) loops over patches, alternating between shared-memory buffers and prefetching the next patch while it works on
the current one.  A second or later pass of that loop can go wrong where the first cannot: a stale buffer half, a prefetch
of the wrong patch, a missing barrier between iterations, a slot or patch index that is wrong after the first wave.  The
other oracle tests run one pass at most.  Each case here is large enough to push the kernels it names past their clamp on
the GPU it runs on (loop_thresholds restates the host's grid formulas; every GPU test checks its case against the device's
SM count, and the CPU test checks the table for a 148-SM B200), and is compared with the oracle on every level, patch by
patch, so that a failure names the pass that went wrong."""
import os
from collections import namedtuple

import numpy as np
import pytest

import gmg_oracle as go
from conftest import MESHES, rel_l2
from test_gmg_solve import cycle_from_guess

TOL = 1e-12
TOL_NEU_SMOOTH, TOL_NEU_CYCLE = 1e-11, 1e-10  # the oracle's Neumann patch solve is a dense transform (as the other Neumann tests)
# A single wrong patch among thousands moves the global relative L2 by its share only, so each patch is held to the
# tolerance too, with room for rounding: one patch's relative error reaches a few times the global figure where the
# result is a small difference of large terms, as an update from a random guess is
PATCH_SLACK = 10


def loop_thresholds(D, n, sm_count):
    """{kernel: (unit, units per pass)} for the persistent kernels of patch size n^D: a level runs a second pass of a
    kernel's loop when it has more units than one pass of the clamped grid covers.  Units: "P" patches of the level,
    "slots" interface slots of a 32^3 level (iface_slots32), "neu" patches with Neumann sides (the Neumann instantiation of
    smooth3d16_kernel walks their list), "neu_end" one past the highest index of such a patch (smooth3d32n_kernel strides
    over the whole level and sweeps only those).  Restates the host's grid formulas, csrc/tgpu.cu (line numbers as of this
    writing): k_apply 1567 / 1581, launch_smooth3d16 1606 / 1610, k_smooth 1640 / 1652 / 1672 / 1681 / 1693,
    k_face_residual_restrict 1714 / 1720 / 1728, k_face_residual_norm 2520."""
    sm = sm_count
    out = {"face_residual_norm": ("P", min(8 * sm, 2048))}  # min(P, 8 sm, MAX_PARTIAL) CTAs, one patch each
    if (D, n) == (3, 32):
        out.update({
            "smooth3d32c": ("P", sm // 2),                  # 2 min(P, sm / 2) CTAs: a cluster of two per patch
            "apply3d32_tma": ("P", sm // 2),                # min(4 P, 2 sm) CTAs, one per 8-plane slab: four per patch
            "iface_rhs32": ("slots", 2 * sm * 6),           # min(ceil(slots / 6), 2 sm) CTAs of six warps, one warp per slot
            "face_residual_restrict_big": ("P", 4 * sm),    # min(P, 4 sm)
            "smooth3d32n": ("neu_end", 2 * sm),             # min(P, 2 sm), over every patch of the level
        })
        return out
    ppb = 256 // n ** (D - 1)  # Geo<D, N>::PPB: patches per CTA of the size-generic kernels (TGPU_THREADS = 256)
    out.update({
        "apply_tma<%d,%d>" % (D, n): ("P", 2 * sm * ppb),                      # min(ceil(P / PPB), 2 sm)
        "smooth<%d,%d>" % (D, n): ("P", (1 if n >= 32 else 3) * sm * ppb),     # min(ceil(P / PPB), sm smooth_min_blocks<N>)
        "face_residual_restrict<%d,%d>" % (D, n): ("P", 8 * sm * ppb),         # min(ceil(P / PPB), 8 sm)
    })
    if (D, n) == (3, 16):
        out.update({
            "smooth3d16": ("P", 3 * sm),                    # min(P, sm s16_ctas_per_sm(false))
            "smooth3d16_zero_guess": ("P", 4 * sm),         # min(P, sm s16_ctas_per_sm(true))
            "smooth3d16_neumann": ("neu", 2 * sm),          # min(P_neu, sm s16_ctas_per_sm(*, true))
            "face_residual_restrict16": ("P", 8 * sm),      # min(P, 8 sm)
        })
    if (D, n) == (2, 32):
        out["smooth2d32"] = ("P", 2 * sm * ppb)             # min(ceil(P / Q32_WARPS), 2 sm), one warp per patch
    return out


def iface_slots32(L):
    """the slot table of a 32^3 level (build_iface_slots32, csrc/patch3d32.cuh): -> (gslot [P, 6], number of slots).  A
    mutual same-level pair of sides of two patches without Neumann sides shares one slot (owned by the lower index); every
    other side with a neighbour has its own; domain-boundary sides and patches with Neumann sides have none."""
    gslot = np.full((L.P, 2 * L.D), -1, np.int64)
    k = 0

    def shared(p, s):
        q = L.nbr_idx[p, s, 0]
        if L.neumann[p] or L.nbr_type[p, s] != go.NBR_NORMAL or q == p or q < 0:
            return False
        return (not L.neumann[q] and L.nbr_type[q, s ^ 1] == go.NBR_NORMAL and L.nbr_idx[q, s ^ 1, 0] == p
                and np.array_equal(L.spacings[p], L.spacings[q]))

    for p in range(L.P):
        if L.neumann[p]:
            continue
        for s in range(2 * L.D):
            if L.nbr_type[p, s] == go.NBR_NONE:
                continue
            q = L.nbr_idx[p, s, 0]
            if shared(p, s):
                if q < p:
                    continue
                gslot[q, s ^ 1] = k
            gslot[p, s] = k
            k += 1
    return gslot, k


def level_units(L):
    neu = np.flatnonzero(L.neumann)
    return {"P": L.P, "slots": iface_slots32(L)[1] if (L.D, L.n) == (3, 32) else 0, "neu": len(neu),
            "neu_end": int(neu[-1]) + 1 if len(neu) else 0}


# mesh, D, n, divide, Neumann sides, kernels the finest level must push past their clamp; generic: also run the cases'
# operators and cycles with the size-generic kernels forced (force_generic_kernels)
Case = namedtuple("Case", "id mesh D n divide neumann pushes generic")
CASES = [
    # 960, 904, 456, 64, 8, 1 patches; 2988 slots on level 0
    Case("3d_n32", "multi_refine.bin", 3, 32, 1, False, ("smooth3d32c", "apply3d32_tma", "iface_rhs32", "face_residual_restrict_big"), False),
    # 354 of the 960 patches with Neumann sides: the cluster kernel skips them while it loops, smooth3d32n reuses its scratch
    Case("3d_n32_neumann", "multi_refine.bin", 3, 32, 1, True,
         ("smooth3d32c", "smooth3d32n", "apply3d32_tma", "iface_rhs32", "face_residual_restrict_big"), False),
    # 7680, 7232, 3648, 512, 64, 8, 1 patches
    Case("3d_n16", "multi_refine.bin", 3, 16, 2, False,
         ("smooth3d16", "smooth3d16_zero_guess", "face_residual_restrict16", "face_residual_norm", "apply_tma<3,16>", "smooth<3,16>",
          "face_residual_restrict<3,16>"), True),
    # 1588 of the 7680 patches with Neumann sides
    Case("3d_n16_neumann", "multi_refine.bin", 3, 16, 2, True,
         ("smooth3d16", "smooth3d16_zero_guess", "smooth3d16_neumann", "face_residual_restrict16", "face_residual_norm", "apply_tma<3,16>"), False),
    Case("3d_n8", "multi_refine.bin", 3, 8, 2, False, ("smooth<3,8>", "apply_tma<3,8>", "face_residual_restrict<3,8>", "face_residual_norm"), False),
    # 2560, 2224, 1936, ... patches
    Case("2d_n32", "2d_multi_refine_8.bin", 2, 32, 2, False, ("smooth2d32", "apply_tma<2,32>"), False),
]
REPRODUCIBLE = [c for c in CASES if c.id in ("3d_n32", "3d_n32_neumann", "3d_n16_neumann")]


def oracle_levels(c):
    return go.build_hierarchy(os.path.join(MESHES, c.mesh), c.D, c.n, c.divide, neumann=c.neumann)


def not_past_clamp(c, L0, sm_count):
    """the kernels of c.pushes whose loop the finest level L0 does not take past its first pass"""
    th, units = loop_thresholds(c.D, c.n, sm_count), level_units(L0)
    return [(k, th[k], units[th[k][0]]) for k in c.pushes if units[th[k][0]] <= th[k][1]]


# ---- CPU ----
def test_cases_run_past_the_resident_grid_of_a_b200():
    for c in CASES:
        L0 = oracle_levels(c)[0]
        assert not not_past_clamp(c, L0, 148), (c.id, not_past_clamp(c, L0, 148))
        if c.id == "3d_n32":
            assert iface_slots32(L0)[1] == 2988


# ---- GPU ----
def _pps():
    import pressurepoissonsolver_b200 as pps
    return pps


def _sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def ctx():
    c = _pps().Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def case(request, ctx):
    """(case, hierarchy, oracle levels), built once per case"""
    pps, c = _pps(), request.param
    mesh = pps.Mesh.load(os.path.join(MESHES, c.mesh), c.D).set_neumann(c.neumann)
    mesh.refine_leaves(c.divide)
    h = pps.Hierarchy.from_mesh(ctx, mesh, c.n)
    levels = oracle_levels(c)
    assert [L.P for L in levels] == [h.npatch(l) for l in range(h.nlevels)]
    yield c, h, levels
    h.close()
    mesh.close()


def _assert_past_clamp(c, levels):
    sm = _sm_count()
    assert not not_past_clamp(c, levels[0], sm), (c.id, sm, not_past_clamp(c, levels[0], sm))


def _passes(c, L, p, sm_count):
    """the loop pass in which each kernel of c.pushes handles patch p of level L (of the slots it reads, for iface_rhs32)"""
    out = []
    for k, (unit, per) in loop_thresholds(c.D, c.n, sm_count).items():
        if k not in c.pushes:
            continue
        if unit == "slots":
            ks = iface_slots32(L)[0][p]
            out.append("%s %s" % (k, sorted({int(s) // per for s in ks if s >= 0})))
        elif unit == "neu":
            if L.neumann[p]:
                out.append("%s %d" % (k, int(np.searchsorted(np.flatnonzero(L.neumann), p)) // per))
        elif unit == "neu_end":
            if L.neumann[p]:
                out.append("%s %d" % (k, p // per))
        else:
            out.append("%s %d" % (k, p // per))
    return ", ".join(out)


def check(what, got, ref, tol, c, L):
    """global relative L2 below tol and the relative error of every patch below PATCH_SLACK tol; on failure the worst
    patches with the loop pass each kernel handled them in"""
    got, ref = np.asarray(got).reshape(L.P, -1), np.asarray(ref).reshape(L.P, -1)
    per = np.linalg.norm(got - ref, axis=1) / np.maximum(np.linalg.norm(ref, axis=1), 1e-300)
    err = rel_l2(got, ref)
    if err < tol and per.max() < PATCH_SLACK * tol:
        return
    sm = _sm_count()
    worst = np.argsort(per)[::-1][:6]
    pytest.fail("%s [%s]: rel L2 %.3e, %d of %d patches above %.0e; worst: %s" % (
        what, c.id, err, int(np.sum(per >= tol)), L.P, tol,
        "; ".join("patch %d %.3e (pass: %s)" % (p, per[p], _passes(c, L, p, sm)) for p in worst)))


def _tols(c):
    return (TOL_NEU_SMOOTH, TOL_NEU_CYCLE) if c.neumann else (TOL, TOL)


def _rhs(rng, L, neumann):
    f = rng.standard_normal(L.shape)
    return f - f.mean() if neumann else f


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, indirect=True, ids=[c.id for c in CASES])
def test_level_operators_vs_oracle(case):
    """apply, residual and a sweep from a non-zero guess on every level (on 32^3 levels: iface_rhs32 + the cluster sweep)"""
    c, h, levels = case
    _assert_past_clamp(c, levels)
    tol_s, _ = _tols(c)
    rng = np.random.default_rng(4100)
    for l, L in enumerate(levels):
        un, fn = rng.standard_normal(L.shape), rng.standard_normal(L.shape)
        u, f, out = h.new_vec(l, un), h.new_vec(l, fn), h.new_vec(l)
        au = go.apply_op(L, un)
        h.apply(l, u, out)
        check("apply L%d" % l, out.download(), au, TOL, c, L)
        h.residual(l, f, u, out)
        check("residual L%d" % l, out.download(), fn - au, TOL, c, L)
        ref = go.smooth(L, fn, un)
        h.smooth(l, f, u)
        check("smooth L%d" % l, u.download(), ref, tol_s, c, L)
        if c.generic:
            h.force_generic_kernels(True)
            u.upload(un)
            h.smooth(l, f, u)
            h.force_generic_kernels(False)
            check("generic smooth L%d" % l, u.download(), ref, tol_s, c, L)
        for v in (u, f, out):
            v.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, indirect=True, ids=[c.id for c in CASES])
def test_cycles_vs_oracle(case):
    """V(1,1) on the three schedules (the zero-guess and faces-only sweeps and the fused residual + restriction run only
    inside cycles) and V(2,2) with two coarse sweeps"""
    pps = _pps()
    c, h, levels = case
    _assert_past_clamp(c, levels)
    _, tol_c = _tols(c)
    fn = _rhs(np.random.default_rng(4200), levels[0], c.neumann)
    f, u = h.new_vec(0, fn), h.new_vec(0)
    ref = go.vcycle(levels, fn)
    for fused in (1, 2, 0):
        h.vcycle(f, u, pps.CycleOpts.default(fused=fused))
        check("V(1,1) fused=%d" % fused, u.download(), ref, tol_c, c, levels[0])
    if c.generic:
        h.force_generic_kernels(True)
        h.vcycle(f, u)
        h.force_generic_kernels(False)
        check("generic V(1,1)", u.download(), ref, tol_c, c, levels[0])
    ref = go.vcycle(levels, fn, pre=2, post=2, coarse_sweeps=2)
    h.vcycle(f, u, pps.CycleOpts.default(pre_sweeps=2, post_sweeps=2, coarse_sweeps=2))
    check("V(2,2) coarse 2", u.download(), ref, tol_c, c, levels[0])
    f.close()
    u.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, indirect=True, ids=[c.id for c in CASES])
def test_update_from_a_guess_vs_oracle(case):
    """vcycle_update from a random guess (the finest pre-sweep starts from u's boundary slices) and, where
    face_residual_norm_kernel loops, the norm it returns against ||f - A u|| / ||f|| of the result formed on the host"""
    c, h, levels = case
    _assert_past_clamp(c, levels)
    _, tol_c = _tols(c)
    rng = np.random.default_rng(4300)
    L0 = levels[0]
    fn, u0 = _rhs(rng, L0, c.neumann), rng.standard_normal(L0.shape)
    f, u = h.new_vec(0, fn), h.new_vec(0, u0)
    rel = h.vcycle_update(f, u)
    got = u.download()
    check("vcycle_update", got, cycle_from_guess(levels, fn, u0), tol_c, c, L0)
    if "face_residual_norm" in c.pushes:
        full = np.linalg.norm(fn - go.apply_op(L0, got.reshape(L0.shape))) / np.linalg.norm(fn)
        assert abs(rel / full - 1) < 1e-10, (rel, full)
    f.close()
    u.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", REPRODUCIBLE, indirect=True, ids=[c.id for c in REPRODUCIBLE])
def test_cycle_is_bitwise_reproducible(case):
    """a missing barrier between two iterations of a persistent loop shows up as bits that change from run to run"""
    pps = _pps()
    c, h, levels = case
    _assert_past_clamp(c, levels)
    f, u = h.new_vec(0, _rhs(np.random.default_rng(4400), levels[0], c.neumann)), h.new_vec(0)
    first = None
    for rep in range(6):
        h.vcycle(f, u, pps.CycleOpts.default(use_graph=rep & 1))
        bits = u.download().tobytes()
        first = first or bits
        assert bits == first, rep
    f.close()
    u.close()
