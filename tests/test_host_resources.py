"""Every device allocation, stream, event and graph of a hierarchy has one owner: a create that rejects its input releases
what it had already uploaded, and destroying a hierarchy releases what its calls allocated lazily.  Device free memory is
read with torch.cuda.mem_get_info; the GPU may be shared, so the tolerance is well below the leaks these tests catch."""
import ctypes as C

import pytest

import pressurepoissonsolver_b200 as pps

pytestmark = pytest.mark.gpu
TOL = 1 << 30  # bytes
TGPU_ERR_ARG = 1


@pytest.fixture(scope="module")
def ctx():
    c = pps.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def probe(ctx):
    """a small hierarchy whose trim() returns the vector pool's free blocks to the device before each reading"""
    mesh = pps.Mesh.uniform(3, 2)
    h = pps.Hierarchy.from_mesh(ctx, mesh, 32)
    yield h
    h.close()
    mesh.close()


def free_bytes(probe):
    import torch
    probe.ctx.sync()
    probe.trim()
    return torch.cuda.mem_get_info(0)[0]


def test_rejected_descriptor_releases_the_levels_already_uploaded(ctx, probe):
    # 4096 patches of 32^3 on level 0: its two face buffers alone take 2 x 4096 x 6 x 1024 x 8 B = 0.4 GB
    mesh = pps.Mesh.uniform(3, 5)
    nl, descs = mesh.extract_levels(32)
    assert descs[0].npatch >= 4096 and nl >= 2
    descs[1].nbr_type[0] = 7  # a neighbour type out of range, found after level 0 is on the device
    before = free_bytes(probe)
    for _ in range(8):
        h = C.c_void_p()
        assert pps.lib.tgpu_hierarchy_create(ctx._p, 3, 32, nl, descs, C.byref(h)) == TGPU_ERR_ARG
        assert not h.value
    assert b"bad neighbour type" in pps.lib.tgpu_last_error()
    assert before - free_bytes(probe) < TOL
    mesh.close()


def lazy_round(ctx, mesh):
    """a hierarchy that allocates everything its calls create lazily, then is destroyed"""
    h = pps.Hierarchy.from_mesh(ctx, mesh, 32)
    f, u = h.new_vec(0), h.new_vec(0)
    h.init_trig_rhs(f)
    for _ in range(2):  # captured, then replayed
        h.vcycle(f, u)
    h.bicgstab(f, u, tol=1e-12, max_it=100)
    u.set(0.0)
    h.gmg_solve(f, u, tol=1e-10, max_it=50)
    fp, up = pps.PinnedBuffer(f.ncells), pps.PinnedBuffer(f.ncells)
    fp.array[:] = 1.0
    for _ in range(3):
        h.vcycle_host_async(fp, up)
    h.vcycle_host_wait()
    h.set_lambda(1.0)  # allocates the general patch solve's scratch and frees the interface terms
    h.set_lambda(0.0)  # builds them again
    ctx.profile_begin()
    h.vcycle(f, u)
    assert ctx.profile_end()
    for x in (f, u, fp, up):
        x.close()
    h.close()


def test_destroy_releases_what_the_hierarchy_allocated_lazily(ctx, probe):
    # 512 patches of 32^3: a vector is 134 MB; the Krylov and stationary work vectors, the pipeline slots, the per-level
    # cycle vectors and the scratch add up to about 2 GB per round
    mesh = pps.Mesh.uniform(3, 4)
    lazy_round(ctx, mesh)  # the first round also loads the kernels the rounds launch
    before = free_bytes(probe)
    for _ in range(3):
        lazy_round(ctx, mesh)
        assert before - free_bytes(probe) < TOL
    mesh.close()
