"""32^3 sweeps that do not start from zero read their interface terms through a slot table: one term per same-level
interface between two owned patches (gathered for the lower patch index), one per other side with a neighbour, none on
domain-boundary sides and on patches with Neumann sides.  These tests cover each kind of side and the table being rebuilt."""
import os
import sys

import numpy as np
import pytest

import gmg_oracle as go
import pressurepoissonsolver_b200 as pps
from conftest import MESHES, ROOT, rel_l2

pytestmark = pytest.mark.gpu
TOL = 1e-12

# 3uni: shared interfaces and domain-boundary sides; 2refine: coarse / fine sides next to shared ones; 3uni with Neumann
# sides: a mixed level (interior patches on the cluster kernel, the others on the general path)
CASES = [("3uni.bin", False), ("2refine.bin", False), ("3uni.bin", True)]


@pytest.fixture(scope="module")
def ctx():
    c = pps.Context(0)
    yield c
    c.close()


def build(ctx, mesh_file, neumann):
    mesh = pps.Mesh.load(os.path.join(MESHES, mesh_file), 3).set_neumann(neumann)
    return pps.Hierarchy.from_mesh(ctx, mesh, 32), mesh, go.build_hierarchy(os.path.join(MESHES, mesh_file), 3, 32, 0, neumann=neumann)


@pytest.mark.parametrize("mesh_file,neumann", CASES)
def test_sweep_and_cycles_vs_oracle(ctx, mesh_file, neumann):
    h, mesh, levels = build(ctx, mesh_file, neumann)
    # the oracle's Neumann patch solve is a dense transform: the existing Neumann tests' tolerances
    tol_s, tol_c = (1e-11, 1e-10) if neumann else (TOL, TOL)
    rng = np.random.default_rng(505)
    un, fn = rng.standard_normal(levels[0].shape), rng.standard_normal(levels[0].shape)
    if neumann:
        fn -= fn.mean()
    u, f = h.new_vec(0, un), h.new_vec(0, fn)
    h.smooth(0, f, u)
    assert rel_l2(u.download(), go.smooth(levels[0], fn, un)) < tol_s
    h.vcycle(f, u)
    assert rel_l2(u.download(), go.vcycle(levels, fn)) < tol_c
    # V(2, 2): the second post-sweep runs without the prolongation
    h.vcycle(f, u, pps.CycleOpts.default(pre_sweeps=2, post_sweeps=2, coarse_sweeps=2))
    assert rel_l2(u.download(), go.vcycle(levels, fn, pre=2, post=2, coarse_sweeps=2)) < tol_c
    h.close()
    mesh.close()


@pytest.mark.parametrize("mesh_file,neumann", CASES)
def test_cycle_unchanged_after_lambda_round_trip(ctx, mesh_file, neumann):
    """set_lambda frees the interface terms and their slot table (lambda != 0) and builds them again (lambda = 0)"""
    h, mesh, levels = build(ctx, mesh_file, neumann)
    fn = np.random.default_rng(506).standard_normal(levels[0].shape)
    if neumann:
        fn -= fn.mean()
    f, u = h.new_vec(0, fn), h.new_vec(0)
    h.vcycle(f, u)
    before = u.download().tobytes()
    h.set_lambda(0.3)
    h.vcycle(f, u)
    h.set_lambda(0.0)
    h.vcycle(f, u)
    assert u.download().tobytes() == before
    h.close()
    mesh.close()


@pytest.mark.parametrize("env", [None, {"TGPU_HALO_IN_KERNEL": "0"}])
def test_distributed_32cubed_cycle_vs_oracle(env):
    """interior patches first: with the split schedule (TGPU_HALO_IN_KERNEL=0) the launch over the patches with halo
    neighbours reads slots that the launch over the interior patches wrote; with the in-kernel hand-over one launch waits
    per slot owner"""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_multi_gpu import _ngpu, run_distributed
    world = min(_ngpu(), 2)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    levels = go.build_hierarchy(os.path.join(MESHES, "2refine.bin"), 3, 32, 0)
    fn = np.random.default_rng(507).standard_normal(levels[0].shape)
    ret, gather, ncells = run_distributed(world, "2refine.bin", 3, 32, 0, fn, env)
    assert ret[0]["ndist"] >= 1 and ncells == fn.size
    assert rel_l2(gather("vcycle"), go.vcycle(levels, fn).reshape(-1, 32 ** 3)) < TOL
    ref22 = go.vcycle(levels, fn, pre=2, post=2, coarse_sweeps=2)
    assert rel_l2(gather("vcycle22"), ref22.reshape(-1, 32 ** 3)) < TOL
