"""ctypes bindings of the two C-ABI libraries (include/nst.h, include/nsg.h).

libnst.so (host topology) and libnsg.so (CUDA hot path) are built in-tree by `make` /
`__graft_entry__.build()`.  There is no Python or CPU fallback for the device path: if
libnsg.so is missing, or no CUDA device exists, the first device call raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))

i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
i64p = np.ctypeslib.ndpointer(dtype=np.int64, flags="C_CONTIGUOUS")
f64p = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
u8p = np.ctypeslib.ndpointer(dtype=np.uint8, flags="C_CONTIGUOUS")
vp = C.c_void_p
i64 = C.c_int64
i32 = C.c_int32


class NstError(RuntimeError):
    pass


class NsgError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"nsg error {code}: {msg}")
        self.code = code


class InletParams(C.Structure):
    _fields_ = [("u_m", C.c_double), ("H", C.c_double), ("y0", C.c_double), ("time_factor", C.c_double)]


class PartInfo(C.Structure):
    _fields_ = [(n, i64) for n in ("n_own_u", "n_own_p", "n_ghost_u", "n_ghost_p", "n_cells", "n_owned_cells",
                                   "n_vertices", "nnz_jac", "nnz_pm")] + [("n_neighbors", i32), ("n_send", i64),
                                                                         ("n_recv", i64)]


class NsgParams(C.Structure):
    _fields_ = [("nu", C.c_double), ("rho", C.c_double), ("p_out", C.c_double), ("deltat", C.c_double),
                ("forcing", C.c_double * 2), ("neumann_id", i32), ("use_mass", i32), ("stokes", i32),
                ("dirichlet_diag", i32)]


def _opt(ptr_type):
    """ndpointer that also accepts None (NULL)."""
    base = ptr_type

    class _P(base):
        @classmethod
        def from_param(cls, obj):
            if obj is None:
                return None
            return base.from_param(obj)

    return _P


_NST_SIGS = {
    "nst_last_error": (C.c_char_p, []),
    "nst_mesh_read_msh": (C.c_int, [C.c_char_p, C.c_int, C.POINTER(vp)]),
    "nst_mesh_create": (C.c_int, [i64, f64p, i64, i32p, i64, _opt(i32p), _opt(i32p), C.POINTER(vp)]),
    "nst_mesh_refine": (C.c_int, [vp, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.POINTER(vp)]),
    "nst_mesh_tag_boundary_box": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, C.c_int]),
    "nst_mesh_free": (None, [vp]),
    "nst_mesh_n_vertices": (i64, [vp]),
    "nst_mesh_n_cells": (i64, [vp]),
    "nst_mesh_n_edges": (i64, [vp]),
    "nst_mesh_n_boundary_edges": (i64, [vp]),
    "nst_mesh_n_inverted": (i64, [vp]),
    "nst_mesh_xy": (C.POINTER(C.c_double), [vp]),
    "nst_mesh_cells": (C.POINTER(i32), [vp]),
    "nst_mesh_cell_edges": (C.POINTER(i32), [vp]),
    "nst_mesh_edge_vertices": (C.POINTER(i32), [vp]),
    "nst_mesh_edge_tag": (C.POINTER(i32), [vp]),
    "nst_mesh_boundary_faces": (C.c_int, [vp, i32p, i32p, i32p]),
    "nst_partition_rcb": (C.c_int, [vp, C.c_int, i32p]),
    "nst_dofs_distribute": (C.c_int, [vp, C.c_int, _opt(i32p), C.POINTER(vp)]),
    "nst_dofs_free": (None, [vp]),
    "nst_dofs_n_u": (i64, [vp]),
    "nst_dofs_n_p": (i64, [vp]),
    "nst_dofs_cell_dofs": (C.POINTER(i32), [vp]),
    "nst_dofs_vertex_node": (C.POINTER(i32), [vp]),
    "nst_dofs_edge_node": (C.POINTER(i32), [vp]),
    "nst_dofs_vertex_p": (C.POINTER(i32), [vp]),
    "nst_dofs_part_n_u": (C.POINTER(i64), [vp]),
    "nst_dofs_part_n_p": (C.POINTER(i64), [vp]),
    "nst_sparsity": (C.c_int, [vp, vp, C.c_int, C.POINTER(i64), _opt(i64p), _opt(i32p)]),
    "nst_dirichlet_values": (C.c_int, [vp, vp, C.c_int, i32p, i32p, i32p, C.POINTER(InletParams), C.POINTER(i64),
                                       _opt(i32p), _opt(f64p)]),
    "nst_dofs_support_points": (C.c_int, [vp, vp, f64p]),
    "nst_part_build": (C.c_int, [vp, vp, C.c_int, _opt(i32p), C.c_int, C.POINTER(vp)]),
    "nst_part_build_ex": (C.c_int, [vp, vp, C.c_int, _opt(i32p), C.c_int, C.c_int, C.POINTER(vp)]),
    "nst_part_free": (None, [vp]),
    "nst_part_get_info": (C.c_int, [vp, C.POINTER(PartInfo)]),
    "nst_part_l2g": (C.POINTER(i64), [vp]),
    "nst_part_cell_ids": (C.POINTER(i32), [vp]),
    "nst_part_cell_dofs": (C.POINTER(i32), [vp]),
    "nst_part_cell_vertices": (C.POINTER(i32), [vp]),
    "nst_part_xy": (C.POINTER(C.c_double), [vp]),
    "nst_part_cell_owned": (C.POINTER(C.c_uint8), [vp]),
    "nst_part_jac_rowptr": (C.POINTER(i64), [vp]),
    "nst_part_jac_col": (C.POINTER(i32), [vp]),
    "nst_part_pm_rowptr": (C.POINTER(i64), [vp]),
    "nst_part_pm_col": (C.POINTER(i32), [vp]),
    "nst_part_neighbors": (C.POINTER(i32), [vp]),
    "nst_part_send_ptr": (C.POINTER(i64), [vp]),
    "nst_part_send_idx": (C.POINTER(i32), [vp]),
    "nst_part_recv_ptr": (C.POINTER(i64), [vp]),
    "nst_part_recv_idx": (C.POINTER(i32), [vp]),
    "nst_part_n_boundary_faces": (i64, [vp]),
    "nst_part_bface_cell": (C.POINTER(i32), [vp]),
    "nst_part_bface_face": (C.POINTER(i32), [vp]),
    "nst_part_bface_tag": (C.POINTER(i32), [vp]),
}

_NSG_SIGS = {
    "nsg_last_error": (C.c_char_p, []),
    "nsg_create": (C.c_int, [C.c_int, C.POINTER(vp)]),
    "nsg_destroy": (None, [vp]),
    "nsg_set_stream": (C.c_int, [vp, vp]),
    "nsg_set_pattern": (C.c_int, [vp, i64, i64, i64, i64, i64p, i32p, i64p, i32p]),
    "nsg_set_pattern_from_cells": (C.c_int, [vp, i64, i64, i64, i64, i64, i32p]),
    "nsg_get_pattern_sizes": (C.c_int, [vp, C.POINTER(i64), C.POINTER(i64)]),
    "nsg_get_pattern": (C.c_int, [vp, i64p, i32p, i64p, i32p]),
    "nsg_set_mesh": (C.c_int, [vp, i64, i64, f64p, i32p, i32p, i64, i32p, i32p, i32p]),
    "nsg_set_halo": (C.c_int, [vp, i32, i32p, i64p, i32p, i64p, i32p]),
    "nsg_comm_unique_id": (C.c_int, [C.c_char_p]),
    "nsg_comm_init": (C.c_int, [vp, C.c_int, C.c_int, C.c_char_p]),
    "nsg_comm_ipc_handle": (C.c_int, [vp, C.c_char_p]),
    "nsg_comm_set_peers": (C.c_int, [vp, C.c_char_p]),
    "nsg_comm_release_peers": (C.c_int, [vp]),
    "nsg_params_default": (None, [C.POINTER(NsgParams)]),
    "nsg_set_params": (C.c_int, [vp, C.POINTER(NsgParams)]),
    "nsg_assemble": (C.c_int, [vp]),
    "nsg_apply_dirichlet": (C.c_int, [vp, i64, i32p, f64p, i32]),
    "nsg_residual_norm": (C.c_int, [vp, C.POINTER(C.c_double)]),
    "nsg_solve": (C.c_int, [vp, i32, C.c_double, i32, i32, i32, C.POINTER(i32), C.POINTER(C.c_double)]),
    "nsg_gmres_history": (i64, [vp, _opt(f64p), i64]),
    "nsg_last_solve_info": (C.c_int, [vp, i32p]),
    "nsg_last_inner_iterations": (i64, [vp]),
    "nsg_update_solution": (C.c_int, [vp]),
    "nsg_push_time_level": (C.c_int, [vp]),
    "nsg_set_solution": (C.c_int, [vp, f64p]),
    "nsg_set_solution_old": (C.c_int, [vp, f64p]),
    "nsg_set_delta": (C.c_int, [vp, f64p]),
    "nsg_get_solution": (C.c_int, [vp, f64p]),
    "nsg_get_solution_ghosted": (C.c_int, [vp, f64p]),
    "nsg_get_delta": (C.c_int, [vp, f64p]),
    "nsg_get_residual": (C.c_int, [vp, f64p]),
    "nsg_get_matrix_values": (C.c_int, [vp, f64p]),
    "nsg_get_pm_values": (C.c_int, [vp, f64p]),
    "nsg_set_solution_ghosted": (C.c_int, [vp, f64p]),
    "nsg_boundary_force": (C.c_int, [vp, i32, f64p]),
    "nsg_set_cell_ownership": (C.c_int, [vp, i32p, u8p]),
    "nsg_eval_points": (C.c_int, [vp, i64, f64p, i32, f64p, _opt(f64p), _opt(i64p)]),
    "nsg_points_index_info": (C.c_int, [vp, f64p]),
    "nsg_spmv": (C.c_int, [vp, f64p, f64p]),
    "nsg_precond_apply": (C.c_int, [vp, i32, f64p, f64p]),
    "nsg_ilu_apply": (C.c_int, [vp, i32, f64p, f64p]),
    "nsg_time_kernel": (C.c_int, [vp, i32, i32, C.POINTER(C.c_double)]),
    "nsg_set_tuning": (C.c_int, [vp, i32, i32]),
    "nsg_get_counters": (C.c_int, [vp, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64)]),
    "nsg_get_phase_ms": (C.c_int, [vp, C.POINTER(C.c_double)]),
}


def _bind(lib, sigs):
    for name, (res, args) in sigs.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    return lib


_nst = None
_nsg = None


def nst():
    global _nst
    if _nst is None:
        path = os.environ.get("NST_LIB", os.path.join(_HERE, "libnst.so"))  # NST_LIB: A/B builds of the same ABI
        if not os.path.exists(path):
            raise NstError(f"{path} is missing: run `make` (or __graft_entry__.build()) first")
        _nst = _bind(C.CDLL(path), _NST_SIGS)
    return _nst


def nsg():
    """The CUDA library. Loading needs libcudart/libnccl but no GPU; nsg_create needs a GPU."""
    global _nsg
    if _nsg is None:
        path = os.environ.get("NSG_LIB", os.path.join(_HERE, "libnsg.so"))  # NSG_LIB: A/B builds of the same ABI
        if not os.path.exists(path):
            raise NsgError(-1, f"{path} is missing: the CUDA extension was not built and there is no fallback; "
                               "run `make` (or __graft_entry__.build())")
        _nsg = _bind(C.CDLL(path), _NSG_SIGS)
    return _nsg


def nst_check(rc):
    if rc != 0:
        raise NstError(f"nst error {rc}: {nst().nst_last_error().decode()}")


def nsg_check(rc):
    if rc != 0:
        raise NsgError(rc, nsg().nsg_last_error().decode())


def as_array(ptr, n, dtype):
    """Copy n elements out of a library-owned buffer."""
    if n == 0:
        return np.zeros(0, dtype=dtype)
    return np.ctypeslib.as_array(ptr, shape=(int(n),)).astype(dtype, copy=True)
