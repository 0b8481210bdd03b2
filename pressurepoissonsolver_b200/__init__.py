"""pressurepoissonsolver_b200 - B200-native GMG (FAC V-cycle) hot path of ThunderEgg.

This package is a thin ctypes binding over the C-ABI library ``libtgpu.so`` (include/tgpu.h); all
arithmetic runs in hand-written sm_100a CUDA kernels (csrc/kernels.cuh).  There is NO CPU fallback:
importing works without a GPU (so the ABI can be inspected), but creating a ``Context`` without a
CUDA device, or importing without the built library, raises.

The class names mirror the reference's plugin surface (src/Thunderegg/GMG/*.h, Vector.h):
``Hierarchy`` ~ the Level list built by GMG::CycleFactory, ``Vec`` ~ Vector<D>,
``Hierarchy.apply/smooth/restrict/prolong_add/vcycle`` ~ Operator/Smoother/Restrictor/
Interpolator/Cycle, ``Hierarchy.bicgstab`` ~ BiCGStab<D>::solve, ``Hierarchy.vcycle_update/gmg_solve`` ~ stationary
multigrid from an initial guess, ``Hierarchy.fmg`` ~ full multigrid (with ``new_boundary_vec/fold_boundary`` for the
caller's boundary data).
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libtgpu.so")


class TgpuError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "libtgpu.so is not built (%s). Run `python build_native.py` "
            "(needs nvcc); there is no CPU fallback." % LIB_PATH)
    return C.CDLL(LIB_PATH)


lib = _load()


class LevelDesc(C.Structure):
    _fields_ = [("npatch", C.c_int32), ("spacing", C.POINTER(C.c_double)), ("starts", C.POINTER(C.c_double)),
                ("neumann_bits", C.POINTER(C.c_uint8)), ("nbr_type", C.POINTER(C.c_int8)),
                ("nbr_idx", C.POINTER(C.c_int32)), ("orth_on_coarse", C.POINTER(C.c_int8)),
                ("parent_idx", C.POINTER(C.c_int32)), ("orth_on_parent", C.POINTER(C.c_int8))]


class ProfileEntry(C.Structure):
    _fields_ = [("kernel", C.c_char_p), ("level", C.c_int32), ("ms", C.c_float)]


class CycleOpts(C.Structure):
    _fields_ = [("pre_sweeps", C.c_int32), ("post_sweeps", C.c_int32), ("mid_sweeps", C.c_int32),
                ("coarse_sweeps", C.c_int32), ("cycle_type", C.c_int32), ("fused", C.c_int32),
                ("use_graph", C.c_int32), ("max_levels", C.c_int32), ("interpolator", C.c_int32),
                ("reserved_", C.c_int32), ("patches_per_proc", C.c_double)]

    @classmethod
    def default(cls, **kw):
        o = cls()
        lib.tgpu_cycle_opts_default(C.byref(o))
        for k, v in kw.items():
            if not hasattr(o, k):
                raise AttributeError(k)
            setattr(o, k, v)
        return o


# every symbol include/tgpu.h declares (tests check that the library exports all of them)
ABI_SYMBOLS = [
    "tgpu_last_error", "tgpu_version", "tgpu_init", "tgpu_finalize", "tgpu_set_stream", "tgpu_sync",
    "tgpu_kernel_launches", "tgpu_timer_start", "tgpu_timer_stop", "tgpu_profile_begin", "tgpu_profile_end", "tgpu_mesh_load", "tgpu_mesh_uniform",
    "tgpu_mesh_refine_leaves", "tgpu_mesh_refine_box", "tgpu_mesh_destroy", "tgpu_mesh_info", "tgpu_mesh_extract_levels",
    "tgpu_mesh_level_ids", "tgpu_hierarchy_create", "tgpu_hierarchy_destroy", "tgpu_hierarchy_info",
    "tgpu_level_npatch", "tgpu_vec_create", "tgpu_vec_destroy", "tgpu_vec_upload", "tgpu_vec_download",
    "tgpu_vec_upload_async", "tgpu_vec_download_async", "tgpu_vec_device_ptr", "tgpu_host_alloc", "tgpu_host_free",
    "tgpu_vec_set", "tgpu_vec_scale", "tgpu_vec_shift", "tgpu_vec_copy", "tgpu_vec_add", "tgpu_vec_add_scaled",
    "tgpu_vec_add_scaled2", "tgpu_vec_scale_then_add", "tgpu_vec_scale_then_add_scaled",
    "tgpu_vec_scale_then_add_scaled2", "tgpu_vec_two_norm", "tgpu_vec_inf_norm", "tgpu_vec_dot", "tgpu_apply",
    "tgpu_residual", "tgpu_smooth", "tgpu_smooth_jacobi", "tgpu_restrict", "tgpu_prolong_add",
    "tgpu_residual_restrict", "tgpu_cycle_opts_default", "tgpu_vcycle", "tgpu_bicgstab", "tgpu_vcycle_host",
    "tgpu_init_trig_rhs", "tgpu_init_neumann_rhs", "tgpu_vec_integrate", "tgpu_mesh_partition", "tgpu_part_destroy", "tgpu_part_info", "tgpu_part_level", "tgpu_part_peer", "tgpu_part_level_interior",
    "tgpu_comm_unique_id", "tgpu_comm_init", "tgpu_hierarchy_create_distributed",
    "tgpu_hierarchy_force_generic_kernels", "tgpu_mesh_set_neumann", "tgpu_vcycle_host_async", "tgpu_vcycle_host_wait",
    "tgpu_hierarchy_trim", "tgpu_hierarchy_set_lambda", "tgpu_hierarchy_set_helmholtz", "tgpu_prolong_add_linear", "tgpu_vec_transfer_pair",
    "tgpu_vcycle_update", "tgpu_gmg_solve", "tgpu_boundary_sides", "tgpu_boundary_vec_create", "tgpu_fold_boundary",
    "tgpu_fmg",
]

lib.tgpu_last_error.restype = C.c_char_p
lib.tgpu_version.restype = C.c_char_p
_vp = C.c_void_p
for _name, _args in {
    "tgpu_init": [C.c_int, C.POINTER(_vp)], "tgpu_finalize": [_vp], "tgpu_set_stream": [_vp, _vp], "tgpu_sync": [_vp],
    "tgpu_kernel_launches": [_vp, C.POINTER(C.c_int64)], "tgpu_timer_start": [_vp],
    "tgpu_timer_stop": [_vp, C.POINTER(C.c_double)],
    "tgpu_profile_begin": [_vp], "tgpu_profile_end": [_vp, C.POINTER(C.c_int), C.POINTER(C.POINTER(ProfileEntry))],
    "tgpu_mesh_load": [C.c_char_p, C.c_int, C.POINTER(_vp)], "tgpu_mesh_uniform": [C.c_int, C.c_int, C.POINTER(_vp)],
    "tgpu_mesh_refine_leaves": [_vp], "tgpu_mesh_destroy": [_vp],
    "tgpu_mesh_refine_box": [_vp, C.POINTER(C.c_double), C.POINTER(C.c_double)],
    "tgpu_mesh_info": [_vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)],
    "tgpu_mesh_extract_levels": [_vp, C.c_int, C.POINTER(C.c_int), C.POINTER(C.POINTER(LevelDesc))],
    "tgpu_mesh_level_ids": [_vp, C.c_int, C.POINTER(C.POINTER(C.c_int32)), C.POINTER(C.POINTER(C.c_int32)),
                            C.POINTER(C.POINTER(C.c_int32))],
    "tgpu_hierarchy_create": [_vp, C.c_int, C.c_int, C.c_int, C.POINTER(LevelDesc), C.POINTER(_vp)],
    "tgpu_hierarchy_destroy": [_vp], "tgpu_hierarchy_trim": [_vp],
    "tgpu_hierarchy_info": [_vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)],
    "tgpu_level_npatch": [_vp, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64)],
    "tgpu_vec_create": [_vp, C.c_int, C.POINTER(_vp)], "tgpu_vec_destroy": [_vp],
    "tgpu_vec_upload": [_vp, _vp], "tgpu_vec_download": [_vp, _vp],
    "tgpu_vec_upload_async": [_vp, _vp], "tgpu_vec_download_async": [_vp, _vp],
    "tgpu_vec_device_ptr": [_vp, C.POINTER(_vp), C.POINTER(C.c_int64)],
    "tgpu_host_alloc": [C.c_size_t, C.POINTER(_vp)], "tgpu_host_free": [_vp],
    "tgpu_vec_set": [_vp, C.c_double], "tgpu_vec_scale": [_vp, C.c_double], "tgpu_vec_shift": [_vp, C.c_double],
    "tgpu_vec_copy": [_vp, _vp], "tgpu_vec_add": [_vp, _vp], "tgpu_vec_add_scaled": [_vp, C.c_double, _vp],
    "tgpu_vec_add_scaled2": [_vp, C.c_double, _vp, C.c_double, _vp],
    "tgpu_vec_scale_then_add": [_vp, C.c_double, _vp],
    "tgpu_vec_scale_then_add_scaled": [_vp, C.c_double, C.c_double, _vp],
    "tgpu_vec_scale_then_add_scaled2": [_vp, C.c_double, C.c_double, _vp, C.c_double, _vp],
    "tgpu_vec_two_norm": [_vp, C.POINTER(C.c_double)], "tgpu_vec_inf_norm": [_vp, C.POINTER(C.c_double)],
    "tgpu_vec_dot": [_vp, _vp, C.POINTER(C.c_double)],
    "tgpu_apply": [_vp, C.c_int, _vp, _vp], "tgpu_residual": [_vp, C.c_int, _vp, _vp, _vp],
    "tgpu_smooth": [_vp, C.c_int, _vp, _vp], "tgpu_smooth_jacobi": [_vp, C.c_int, _vp, _vp, C.c_double],
    "tgpu_restrict": [_vp, C.c_int, _vp, _vp], "tgpu_prolong_add": [_vp, C.c_int, _vp, _vp],
    "tgpu_residual_restrict": [_vp, C.c_int, _vp, _vp, _vp], "tgpu_prolong_add_linear": [_vp, C.c_int, _vp, _vp],
    "tgpu_cycle_opts_default": [C.POINTER(CycleOpts)], "tgpu_vcycle": [_vp, C.POINTER(CycleOpts), _vp, _vp],
    "tgpu_bicgstab": [_vp, C.POINTER(CycleOpts), _vp, _vp, C.c_double, C.c_int, C.POINTER(C.c_int),
                      C.POINTER(C.c_double)],
    "tgpu_vcycle_host": [_vp, C.POINTER(CycleOpts), _vp, _vp],
    "tgpu_vcycle_update": [_vp, C.POINTER(CycleOpts), _vp, _vp, C.POINTER(C.c_double)],
    "tgpu_gmg_solve": [_vp, C.POINTER(CycleOpts), _vp, _vp, C.c_double, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_double),
                       C.POINTER(C.c_double)],
    "tgpu_boundary_sides": [_vp, C.POINTER(C.c_int64), C.POINTER(C.POINTER(C.c_int32)), C.POINTER(C.POINTER(C.c_int8))],
    "tgpu_boundary_vec_create": [_vp, C.POINTER(_vp)], "tgpu_fold_boundary": [_vp, _vp, _vp],
    "tgpu_fmg": [_vp, C.POINTER(CycleOpts), C.c_int, _vp, _vp, _vp],
    "tgpu_init_trig_rhs": [_vp, _vp, _vp],
    "tgpu_init_neumann_rhs": [_vp, C.c_int, _vp, _vp],
    "tgpu_vec_integrate": [_vp, _vp, C.POINTER(C.c_double), C.POINTER(C.c_double)],
    "tgpu_mesh_partition": [_vp, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(_vp)], "tgpu_part_destroy": [_vp],
    "tgpu_part_info": [_vp, C.POINTER(C.c_int), C.POINTER(C.c_int)],
    "tgpu_part_level": [_vp, C.c_int, C.POINTER(LevelDesc), C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                        C.POINTER(C.POINTER(C.c_int32)), C.POINTER(C.POINTER(C.c_int32)), C.POINTER(C.POINTER(C.c_int32)),
                        C.POINTER(C.c_int32)],
    "tgpu_part_peer": [_vp, C.c_int, C.c_int, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.POINTER(C.c_int32)),
                       C.POINTER(C.POINTER(C.c_int32)), C.POINTER(C.c_int32), C.POINTER(C.POINTER(C.c_int32)),
                       C.POINTER(C.POINTER(C.c_int32))],
    "tgpu_part_level_interior": [_vp, C.c_int, C.POINTER(C.c_int32)],
    "tgpu_comm_unique_id": [_vp], "tgpu_comm_init": [_vp, _vp, C.c_int, C.c_int],
    "tgpu_hierarchy_create_distributed": [_vp, _vp, C.POINTER(_vp)],
    "tgpu_hierarchy_force_generic_kernels": [_vp, C.c_int], "tgpu_hierarchy_set_lambda": [_vp, C.c_double],
    "tgpu_hierarchy_set_helmholtz": [_vp, C.c_double],
    "tgpu_mesh_set_neumann": [_vp, C.c_int],
    "tgpu_vcycle_host_async": [_vp, C.POINTER(CycleOpts), _vp, _vp], "tgpu_vcycle_host_wait": [_vp],
    "tgpu_vec_transfer_pair": [_vp, _vp, _vp, _vp, _vp],
}.items():
    getattr(lib, _name).argtypes = _args
    getattr(lib, _name).restype = C.c_int


def check(rc):
    if rc != 0:
        raise TgpuError("tgpu error %d: %s" % (rc, lib.tgpu_last_error().decode()))


class Context:
    def __init__(self, device=0):
        self._p = _vp()
        check(lib.tgpu_init(device, C.byref(self._p)))

    def set_stream(self, cuda_stream):
        check(lib.tgpu_set_stream(self._p, _vp(cuda_stream)))

    def sync(self):
        check(lib.tgpu_sync(self._p))

    def kernel_launches(self):
        n = C.c_int64()
        check(lib.tgpu_kernel_launches(self._p, C.byref(n)))
        return n.value

    def timer_start(self):
        check(lib.tgpu_timer_start(self._p))

    def timer_stop(self):
        ms = C.c_double()
        check(lib.tgpu_timer_stop(self._p, C.byref(ms)))
        return ms.value

    def comm_init(self, unique_id, rank, nranks):
        check(lib.tgpu_comm_init(self._p, C.c_char_p(unique_id), rank, nranks))

    def profile_begin(self):
        check(lib.tgpu_profile_begin(self._p))

    def profile_end(self):
        """-> list of (kernel name, level, milliseconds) for every launch since profile_begin"""
        n, ent = C.c_int(), C.POINTER(ProfileEntry)()
        check(lib.tgpu_profile_end(self._p, C.byref(n), C.byref(ent)))
        return [(ent[i].kernel.decode(), ent[i].level, ent[i].ms) for i in range(n.value)]

    def close(self):
        if self._p:
            lib.tgpu_finalize(self._p)
            self._p = _vp()


class Mesh:
    """Tree<D> + ThundereggDomGen<D> level extraction (host side)."""

    def __init__(self, ptr):
        self._p = ptr
        self._nlevels = 0
        self._descs = None

    @classmethod
    def load(cls, path, D):
        p = _vp()
        check(lib.tgpu_mesh_load(os.fsencode(path), D, C.byref(p)))
        return cls(p)

    @classmethod
    def uniform(cls, D, num_levels):
        p = _vp()
        check(lib.tgpu_mesh_uniform(D, num_levels, C.byref(p)))
        return cls(p)

    def refine_leaves(self, times=1):
        for _ in range(times):
            check(lib.tgpu_mesh_refine_leaves(self._p))
        return self

    def set_neumann(self, on=True):
        check(lib.tgpu_mesh_set_neumann(self._p, 1 if on else 0))
        return self

    def refine_box(self, lo, hi):
        a, b = (C.c_double * 3)(*lo), (C.c_double * 3)(*hi)
        check(lib.tgpu_mesh_refine_box(self._p, a, b))
        return self

    def info(self):
        D, nl, nn = C.c_int(), C.c_int(), C.c_int()
        check(lib.tgpu_mesh_info(self._p, C.byref(D), C.byref(nl), C.byref(nn)))
        return D.value, nl.value, nn.value

    def extract_levels(self, n):
        nl = C.c_int()
        descs = C.POINTER(LevelDesc)()
        check(lib.tgpu_mesh_extract_levels(self._p, n, C.byref(nl), C.byref(descs)))
        self._nlevels, self._descs, self._n = nl.value, descs, n
        return nl.value, descs

    def level_arrays(self, n):
        """numpy copies of the extracted level tables (for cross-checks against the reference)."""
        D = self.info()[0]
        nl, descs = self.extract_levels(n)
        S, Q = 2 * D, 1 << (D - 1)
        out = []
        for l in range(nl):
            d = descs[l]
            P = d.npatch
            ids, pids, rl = (C.POINTER(C.c_int32)(), C.POINTER(C.c_int32)(), C.POINTER(C.c_int32)())
            check(lib.tgpu_mesh_level_ids(self._p, l, C.byref(ids), C.byref(pids), C.byref(rl)))
            arr = lambda ptr, shape, dt: np.ctypeslib.as_array(ptr, shape=shape).astype(dt).copy()  # noqa: E731
            out.append(dict(
                npatch=P, ids=arr(ids, (P,), np.int32), parent_id=arr(pids, (P,), np.int32),
                refine_level=arr(rl, (P,), np.int32), spacings=arr(d.spacing, (P, D), np.float64),
                starts=arr(d.starts, (P, D), np.float64), neumann=arr(d.neumann_bits, (P,), np.int32),
                nbr_type=arr(d.nbr_type, (P, S), np.int32), nbr_idx=arr(d.nbr_idx, (P, S, Q), np.int32),
                orth_on_coarse=arr(d.orth_on_coarse, (P, S), np.int32), parent_idx=arr(d.parent_idx, (P,), np.int32),
                orth_on_parent=arr(d.orth_on_parent, (P,), np.int32)))
        return out

    def close(self):
        if self._p:
            lib.tgpu_mesh_destroy(self._p)
            self._p = _vp()


def _desc_arrays(d, D):
    S, Q, P = 2 * D, 1 << (D - 1), d.npatch
    arr = lambda ptr, shape, dt: np.ctypeslib.as_array(ptr, shape=shape).astype(dt).copy()  # noqa: E731
    return dict(npatch=P, spacings=arr(d.spacing, (P, D), np.float64), starts=arr(d.starts, (P, D), np.float64),
                neumann=arr(d.neumann_bits, (P,), np.int32), nbr_type=arr(d.nbr_type, (P, S), np.int32),
                nbr_idx=arr(d.nbr_idx, (P, S, Q), np.int32), orth_on_coarse=arr(d.orth_on_coarse, (P, S), np.int32),
                parent_idx=arr(d.parent_idx, (P,), np.int32), orth_on_parent=arr(d.orth_on_parent, (P,), np.int32))


class Partition:
    """Patches of every level split over `nranks` GPUs + the halo-exchange plan of rank `rank`."""

    def __init__(self, mesh, n, rank, nranks, min_patches_per_rank=8):
        self._p = _vp()
        self.D = mesh.info()[0]
        self.n, self.rank, self.nranks = n, rank, nranks
        check(lib.tgpu_mesh_partition(mesh._p, n, rank, nranks, min_patches_per_rank, C.byref(self._p)))
        a, b = C.c_int(), C.c_int()
        check(lib.tgpu_part_info(self._p, C.byref(a), C.byref(b)))
        self.nlevels, self.ndist = a.value, b.value

    def level(self, l):
        d = LevelDesc()
        no, nh, npe = C.c_int32(), C.c_int32(), C.c_int32()
        og, hg, ho = (C.POINTER(C.c_int32)() for _ in range(3))
        check(lib.tgpu_part_level(self._p, l, C.byref(d), C.byref(no), C.byref(nh), C.byref(og), C.byref(hg), C.byref(ho), C.byref(npe)))
        out = _desc_arrays(d, self.D)
        as_np = lambda ptr, n: np.ctypeslib.as_array(ptr, shape=(n,)).copy() if n else np.zeros(0, np.int32)  # noqa: E731
        ni = C.c_int32()
        check(lib.tgpu_part_level_interior(self._p, l, C.byref(ni)))
        out.update(n_interior=ni.value, n_owned=no.value, n_halo=nh.value, owned_global=as_np(og, no.value), halo_global=as_np(hg, nh.value),
                   halo_owner=as_np(ho, nh.value), peers=[])
        for k in range(npe.value):
            peer, ns, nr = C.c_int32(), C.c_int32(), C.c_int32()
            sp, ss, rs, rd = (C.POINTER(C.c_int32)() for _ in range(4))
            check(lib.tgpu_part_peer(self._p, l, k, C.byref(peer), C.byref(ns), C.byref(sp), C.byref(ss), C.byref(nr), C.byref(rs), C.byref(rd)))
            out["peers"].append(dict(peer=peer.value, send_patch=as_np(sp, ns.value), send_side=as_np(ss, ns.value),
                                     recv_slot=as_np(rs, nr.value), recv_side=as_np(rd, nr.value)))
        return out

    def close(self):
        if self._p:
            lib.tgpu_part_destroy(self._p)
            self._p = _vp()


def comm_unique_id():
    buf = C.create_string_buffer(128)
    check(lib.tgpu_comm_unique_id(buf))
    return buf.raw


class Vec:
    """Vector<D> of one level, resident in HBM."""

    def __init__(self, hier, level):
        self.hier, self.level = hier, level
        self._p = _vp()
        check(lib.tgpu_vec_create(hier._p, level, C.byref(self._p)))
        self.ncells = hier.ncells(level)

    def upload(self, a):
        a = np.ascontiguousarray(a, dtype=np.float64).ravel()
        if a.size != self.ncells:
            raise ValueError("size mismatch: %d vs %d" % (a.size, self.ncells))
        check(lib.tgpu_vec_upload(self._p, a.ctypes.data_as(_vp)))
        return self

    def download(self):
        a = np.empty(self.ncells, dtype=np.float64)
        check(lib.tgpu_vec_download(self._p, a.ctypes.data_as(_vp)))
        return a

    def device_ptr(self):
        p, n = _vp(), C.c_int64()
        check(lib.tgpu_vec_device_ptr(self._p, C.byref(p), C.byref(n)))
        return p.value

    def set(self, a): check(lib.tgpu_vec_set(self._p, a))
    def scale(self, a): check(lib.tgpu_vec_scale(self._p, a))
    def shift(self, a): check(lib.tgpu_vec_shift(self._p, a))
    def copy(self, b): check(lib.tgpu_vec_copy(self._p, b._p))
    def add(self, b): check(lib.tgpu_vec_add(self._p, b._p))
    def add_scaled(self, alpha, b): check(lib.tgpu_vec_add_scaled(self._p, alpha, b._p))
    def add_scaled2(self, alpha, a, beta, b): check(lib.tgpu_vec_add_scaled2(self._p, alpha, a._p, beta, b._p))
    def scale_then_add(self, alpha, b): check(lib.tgpu_vec_scale_then_add(self._p, alpha, b._p))
    def scale_then_add_scaled(self, alpha, beta, b): check(lib.tgpu_vec_scale_then_add_scaled(self._p, alpha, beta, b._p))

    def scale_then_add_scaled2(self, alpha, beta, b, gamma, c):
        check(lib.tgpu_vec_scale_then_add_scaled2(self._p, alpha, beta, b._p, gamma, c._p))

    def two_norm(self):
        r = C.c_double()
        check(lib.tgpu_vec_two_norm(self._p, C.byref(r)))
        return r.value

    def inf_norm(self):
        r = C.c_double()
        check(lib.tgpu_vec_inf_norm(self._p, C.byref(r)))
        return r.value

    def dot(self, b):
        r = C.c_double()
        check(lib.tgpu_vec_dot(self._p, b._p, C.byref(r)))
        return r.value

    def close(self):
        if self._p:
            lib.tgpu_vec_destroy(self._p)
            self._p = _vp()


class PinnedBuffer:
    def __init__(self, ncells):
        self._p = _vp()
        check(lib.tgpu_host_alloc(ncells * 8, C.byref(self._p)))
        self.array = np.ctypeslib.as_array(C.cast(self._p, C.POINTER(C.c_double)), shape=(ncells,))

    def close(self):
        if self._p:
            lib.tgpu_host_free(self._p)
            self._p = _vp()


class Hierarchy:
    """Device-resident level hierarchy = what GMG::CycleFactory{2,3}d::getCycle builds
    (GMG/CycleFactory3d.cpp:69-134), flattened into neighbour tables."""

    def __init__(self, ctx, D, n, nlevels, descs):
        self.ctx, self.D, self.n, self.nlevels = ctx, D, n, nlevels
        self._p = _vp()
        check(lib.tgpu_hierarchy_create(ctx._p, D, n, nlevels, descs, C.byref(self._p)))

    @classmethod
    def from_mesh(cls, ctx, mesh, n):
        nl, descs = mesh.extract_levels(n)
        return cls(ctx, mesh.info()[0], n, nl, descs)

    @classmethod
    def from_partition(cls, ctx, part):
        self = cls.__new__(cls)
        self.ctx, self.D, self.n, self.nlevels = ctx, part.D, part.n, part.nlevels
        self._p = _vp()
        check(lib.tgpu_hierarchy_create_distributed(ctx._p, part._p, C.byref(self._p)))
        return self

    def trim(self):
        """free lazily allocated work space (Krylov vectors, host-buffer slots, cached graphs, pooled vector storage)"""
        check(lib.tgpu_hierarchy_trim(self._p))

    def set_lambda(self, lam):
        """the patch solver's shift (FftwPatchSolver(domain, lambda), PatchSolvers/FftwPatchSolver.h:66,170)"""
        check(lib.tgpu_hierarchy_set_lambda(self._p, lam))

    def set_helmholtz(self, lam):
        """operator A + lam I on every level, with the patch solver's shift lam too (lam finite and <= 0; 0: Poisson)"""
        check(lib.tgpu_hierarchy_set_helmholtz(self._p, lam))

    def force_generic_kernels(self, on=True):
        check(lib.tgpu_hierarchy_force_generic_kernels(self._p, 1 if on else 0))

    def npatch(self, level):
        a, b = C.c_int64(), C.c_int64()
        check(lib.tgpu_level_npatch(self._p, level, C.byref(a), C.byref(b)))
        return a.value

    def ncells(self, level):
        a, b = C.c_int64(), C.c_int64()
        check(lib.tgpu_level_npatch(self._p, level, C.byref(a), C.byref(b)))
        return b.value

    def new_vec(self, level=0, data=None):
        v = Vec(self, level)
        if data is not None:
            v.upload(data)
        return v

    def apply(self, level, u, out): check(lib.tgpu_apply(self._p, level, u._p, out._p))
    def residual(self, level, f, u, r): check(lib.tgpu_residual(self._p, level, f._p, u._p, r._p))
    def smooth(self, level, f, u): check(lib.tgpu_smooth(self._p, level, f._p, u._p))
    def smooth_jacobi(self, level, f, u, omega): check(lib.tgpu_smooth_jacobi(self._p, level, f._p, u._p, omega))
    def restrict(self, fine_level, fine, coarse): check(lib.tgpu_restrict(self._p, fine_level, fine._p, coarse._p))
    def prolong_add(self, fine_level, coarse, fine): check(lib.tgpu_prolong_add(self._p, fine_level, coarse._p, fine._p))

    def prolong_add_linear(self, fine_level, coarse, fine):
        check(lib.tgpu_prolong_add_linear(self._p, fine_level, coarse._p, fine._p))

    def residual_restrict(self, fine_level, f, u, coarse_f):
        check(lib.tgpu_residual_restrict(self._p, fine_level, f._p, u._p, coarse_f._p))

    def vcycle(self, f, u, opts=None):
        check(lib.tgpu_vcycle(self._p, C.byref(opts) if opts is not None else None, f._p, u._p))

    def vcycle_host(self, f_pinned, u_pinned, opts=None):
        check(lib.tgpu_vcycle_host(self._p, C.byref(opts) if opts is not None else None, f_pinned._p, u_pinned._p))

    def vcycle_host_async(self, f_pinned, u_pinned, opts=None):
        """pipelined form for a stream of independent right-hand sides; results are valid after vcycle_host_wait()"""
        check(lib.tgpu_vcycle_host_async(self._p, C.byref(opts) if opts is not None else None, f_pinned._p, u_pinned._p))

    def copy_pair(self, dst_dev, src_pinned, src_dev, dst_pinned):
        """host -> dst_dev and src_dev -> host concurrently (the copies of one pipelined e2e step, nothing else)"""
        check(lib.tgpu_vec_transfer_pair(self._p, dst_dev._p, src_pinned._p, src_dev._p, dst_pinned._p))

    def vcycle_host_wait(self):
        check(lib.tgpu_vcycle_host_wait(self._p))

    def bicgstab(self, f, u, opts=None, tol=1e-12, max_it=1000, precondition=True):
        if precondition and opts is None:
            opts = CycleOpts.default()
        its, rel = C.c_int(), C.c_double()
        check(lib.tgpu_bicgstab(self._p, C.byref(opts) if precondition else None, f._p, u._p, tol, max_it,
                                C.byref(its), C.byref(rel)))
        return its.value, rel.value

    def vcycle_update(self, f, u, opts=None):
        """u <- u + Cycle(f - A u) from the iterate in u; -> ||f - A u|| / ||f|| of the result"""
        rel = C.c_double()
        check(lib.tgpu_vcycle_update(self._p, C.byref(opts) if opts is not None else None, f._p, u._p, C.byref(rel)))
        return rel.value

    def gmg_solve(self, f, u, opts=None, tol=1e-10, max_it=100, history=False):
        """stationary multigrid from the iterate in u until ||f - A u|| <= tol ||f||; -> (cycles, relative residual) and,
        with history=True, the relative residual before the first cycle and after each one"""
        its, rel = C.c_int(), C.c_double()
        hist = (C.c_double * max(max_it + 1, 1))() if history else None
        check(lib.tgpu_gmg_solve(self._p, C.byref(opts) if opts is not None else None, f._p, u._p, tol, max_it, C.byref(its),
                                 C.byref(rel), hist))
        if history:
            return its.value, rel.value, list(hist[:its.value + 1])
        return its.value, rel.value

    def boundary_sides(self):
        """-> (patch, side): the domain-boundary sides of level 0's owned patches, ascending; row k of a boundary vector
        holds side k's n^(D-1) values in face order"""
        cnt, pa, sa = C.c_int64(), C.POINTER(C.c_int32)(), C.POINTER(C.c_int8)()
        check(lib.tgpu_boundary_sides(self._p, C.byref(cnt), C.byref(pa), C.byref(sa)))
        if cnt.value == 0:
            return np.zeros(0, np.int32), np.zeros(0, np.int8)
        return (np.ctypeslib.as_array(pa, shape=(cnt.value,)).copy(), np.ctypeslib.as_array(sa, shape=(cnt.value,)).copy())

    def new_boundary_vec(self, data=None):
        """boundary data of level 0: Dirichlet values / outward normal derivatives, one row per boundary_sides() entry"""
        v = Vec.__new__(Vec)
        v.hier, v.level, v._p = self, -1, _vp()
        check(lib.tgpu_boundary_vec_create(self._p, C.byref(v._p)))
        n = C.c_int64()
        check(lib.tgpu_vec_device_ptr(v._p, None, C.byref(n)))
        v.ncells = n.value
        if data is not None:
            v.upload(data)
        return v

    def fold_boundary(self, b, f):
        """f -= 2 b / h^2 (Dirichlet sides), b / h (Neumann sides) on the boundary cells of level 0"""
        check(lib.tgpu_fold_boundary(self._p, b._p, f._p))

    def fmg(self, f, u, b=None, opts=None, cycles=2):
        """full multigrid u <- FMG(f); b: the Dirichlet values folded into f (None: homogeneous)"""
        check(lib.tgpu_fmg(self._p, C.byref(opts) if opts is not None else None, cycles, f._p, b._p if b is not None else None, u._p))

    def init_trig_rhs(self, f, exact=None):
        check(lib.tgpu_init_trig_rhs(self._p, f._p, exact._p if exact is not None else None))

    def init_neumann_rhs(self, f, exact=None, problem="trig"):
        """Init::initNeumann (apps/shared/Init.cpp:57-151) on the 3D manufactured problems `trig` / `gauss`"""
        check(lib.tgpu_init_neumann_rhs(self._p, {"trig": 0, "gauss": 1}[problem], f._p, exact._p if exact is not None else None))

    def integrate(self, v):
        """(Domain::integrate(v), Domain::volume()), Domain.h:237-278"""
        a, b = C.c_double(), C.c_double()
        check(lib.tgpu_vec_integrate(self._p, v._p, C.byref(a), C.byref(b)))
        return a.value, b.value

    def close(self):
        if self._p:
            lib.tgpu_hierarchy_destroy(self._p)
            self._p = _vp()
