"""ctypes binding of libsemk.so (the C ABI declared in include/semk.h).

This is the stub a maintainer of the reference would add (see INTEGRATION.md).
There is deliberately NO fallback: if the shared library is missing or a CUDA
device is required and absent, the call raises -- the product never routes
through a CPU implementation.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libsemk.so")

# status codes / flags (mirror include/semk.h)
OK, ERR_INVALID, ERR_CUDA, ERR_JACOBIAN, ERR_BREAKDOWN, ERR_UNSUPPORTED = 0, -1, -2, -3, -4, -5
NODE_ID_MASK, NODE_SHARED, NODE_DIRICHLET = 0x3FFFFFFF, 0x40000000, 0x80000000
MASK_IN, MASK_OUT, DIRICHLET_IDENTITY = 1, 2, 4
MAX_N1 = 17

(PA_PATCH_NODE_PTR, PA_PNODE, PA_PATCH_NPRIV, PA_PATCH_SLOT_BASE, PA_ELOC,
 PA_ELEM_OF_SLOT, PA_SHARED_NODE, PA_SHARED_PTR, PA_SHARED_SLOT, PA_PATCH_NNODES,
 PA_PNBLK, PA_ELBLK, PA_SHARED_REC, PA_SHARED_EXT, PA_SHARED_CHUNK,
 PA_PATCH_HDR, PA_PATCH_MAXNODE, PA_CHUNK_MAXPATCH, PA_REC_MAXPATCH, PA_INVBLK) = range(20)
(PS_N_PATCH, PS_N_PNODE, PS_N_SLOTS, PS_N_SHARED, PS_MAX_PATCH_NODES,
 PS_N_SLOT_ELEMS, PS_ELOC_STRIDE, PS_PN_STRIDE, PS_EL_STRIDE, PS_N_SHARED_CHUNK,
 PS_N_SHARED_REC, PS_N_PN_UNIQUE, PS_N_EL_UNIQUE, PS_N_INV_UNIQUE, PS_INV_WIDTH,
 PS_INV_STRIDE) = range(16)
PS_COUNT = 16

PLAN_ARRAY_DTYPES = {
    PA_PATCH_NODE_PTR: np.int32, PA_PNODE: np.uint32, PA_PATCH_NPRIV: np.int32,
    PA_PATCH_SLOT_BASE: np.int32, PA_ELOC: np.uint16,
    PA_ELEM_OF_SLOT: np.int64, PA_SHARED_NODE: np.uint32, PA_SHARED_PTR: np.int32,
    PA_SHARED_SLOT: np.int32, PA_PATCH_NNODES: np.int32, PA_PNBLK: np.uint32,
    PA_ELBLK: np.uint16, PA_SHARED_REC: np.uint32, PA_SHARED_EXT: np.uint32,
    PA_SHARED_CHUNK: np.uint32, PA_PATCH_HDR: np.uint32, PA_PATCH_MAXNODE: np.uint32,
    PA_CHUNK_MAXPATCH: np.int32, PA_REC_MAXPATCH: np.int32, PA_INVBLK: np.uint16,
}


class SemkError(RuntimeError):
    def __init__(self, code, msg):
        RuntimeError.__init__(self, "libsemk error %d: %s" % (code, msg))
        self.code = code


class SolverFailure(Exception):
    """PCG breakdown (the reference's solver-failure convention,
    sem/rootfind.py:15-19)."""


class semk_op(C.Structure):
    _fields_ = [
        ("n1", C.c_int32), ("elems_per_patch", C.c_int32),
        ("n_elem", C.c_int64), ("n_nodes", C.c_int64), ("n_patch", C.c_int64),
        ("max_patch_nodes", C.c_int64), ("max_ctas", C.c_int64),
        ("g_patch_stride", C.c_int64), ("G", C.c_void_p),
        ("patch_hdr", C.c_void_p), ("pnode", C.c_void_p), ("pn_patch_stride", C.c_int64),
        ("eloc", C.c_void_p), ("eloc_patch_stride", C.c_int64),
        ("inv", C.c_void_p), ("inv_patch_stride", C.c_int64), ("inv_width", C.c_int64),
        ("n_slots", C.c_int64), ("slot_buf", C.c_void_p),
        ("n_shared", C.c_int64), ("shared_rec", C.c_void_p), ("shared_ext", C.c_void_p),
        ("n_shared_chunk", C.c_int64), ("shared_chunk", C.c_void_p),
        ("partials", C.c_void_p), ("D_host", C.c_void_p), ("dirichlet", C.c_void_p),
        ("kernel_variant", C.c_int64),
        ("box_ld", C.c_int64),
        ("separable", C.c_int64),
    ]


class semk_sc_op(C.Structure):
    _fields_ = [
        ("n1", C.c_int32), ("n_ext_loc", C.c_int32),
        ("n_elem", C.c_int64), ("n_ext", C.c_int64), ("s_stride", C.c_int64),
        ("S", C.c_void_p), ("l2g_ext", C.c_void_p), ("y_loc", C.c_void_p),
        ("node_ptr", C.c_void_p), ("node_pos", C.c_void_p), ("dirichlet", C.c_void_p),
        ("partials", C.c_void_p),
    ]


SC_SCHUR, SC_RHS, SC_BACKSOLVE, SC_STORE, SC_STORE_INV = 1, 2, 4, 8, 16


class semk_sc_top(C.Structure):
    _fields_ = [("n_agg", C.c_int64), ("agg", C.c_void_p), ("aptr", C.c_void_p),
                ("aidx", C.c_void_p), ("A3inv", C.c_void_p), ("A3inv_f32", C.c_void_p)]


class semk_sc_coarse(C.Structure):
    _fields_ = [
        ("n_v", C.c_int64), ("Ace", C.c_void_p), ("vert_c", C.c_void_p), ("y_loc_c", C.c_void_p),
        ("vptr", C.c_void_p), ("vpos", C.c_void_p), ("dirichlet_c", C.c_void_p),
        ("partials", C.c_void_p), ("pv", C.c_void_p), ("pw", C.c_void_p), ("rptr", C.c_void_p),
        ("ridx", C.c_void_p), ("rw", C.c_void_p),
        ("ell_width", C.c_int64), ("ell_cols", C.c_void_p), ("ell_vals", C.c_void_p),
    ]


COMM_MAX_WORLD = 8


class semk_comm(C.Structure):
    _fields_ = [("rank", C.c_int32), ("world", C.c_int32), ("capacity", C.c_int64),
                ("regions", C.c_void_p * COMM_MAX_WORLD), ("status", C.c_void_p)]


class semk_halo(C.Structure):
    _fields_ = [("n_col", C.c_int64), ("mine", C.c_void_p), ("left", C.c_void_p),
                ("right", C.c_void_p), ("epoch", C.c_uint64), ("status", C.c_void_p)]


class semk_ml_dist(C.Structure):
    _fields_ = [("comm", C.POINTER(semk_comm)), ("halo_f", C.POINTER(semk_halo)),
                ("halo_c", C.POINTER(semk_halo)), ("n_owned_f", C.c_int64),
                ("n_owned_c", C.c_int64)]


class semk_ml_opts(C.Structure):
    _fields_ = [("rtol", C.c_double), ("inner_rtol", C.c_double), ("maxiter", C.c_int32),
                ("inner_maxiter", C.c_int32), ("levels", C.c_int32), ("flexible", C.c_int32),
                ("inner_chunk", C.c_int32), ("reserved", C.c_int32)]


class semk_ml_info(C.Structure):
    _fields_ = [("iterations", C.c_int32), ("status", C.c_int32), ("rel_residual", C.c_double),
                ("true_rel_residual", C.c_double), ("bnorm", C.c_double),
                ("inner_iterations", C.c_int64), ("inner_solves", C.c_int32),
                ("reserved", C.c_int32)]


class semk_stokes_op(C.Structure):
    _fields_ = [("plan", semk_op), ("n_fac", C.c_int32), ("reserved", C.c_int32),
                ("n_ess", C.c_int64), ("ess_dof", C.c_void_p)]


class semk_stage(C.Structure):
    _fields_ = [("patch_end", C.c_int64), ("chunk_end", C.c_int64), ("rec_end", C.c_int64),
                ("u_need", C.c_int64), ("y_final", C.c_int64)]


class semk_pcg_info(C.Structure):
    _fields_ = [("iterations", C.c_int32), ("status", C.c_int32),
                ("rel_residual", C.c_double), ("bnorm", C.c_double)]


class semk_bdiag(C.Structure):
    _fields_ = [("n", C.c_int64), ("node", C.c_void_p), ("val", C.c_void_p),
                ("partials", C.c_void_p)]


_P, _I, _L, _D = C.c_void_p, C.c_int, C.c_int64, C.c_double

# name -> (restype, argtypes); every symbol include/semk.h declares
SIGNATURES = {
    "semk_version": (_I, []),
    "semk_last_error": (C.c_char_p, []),
    "semk_device_available": (_I, []),
    "semk_hostplan_create": (_I, [_I, _L, _L, _P, _P, _L, _I, _P, C.POINTER(_P)]),
    "semk_hostplan_create_mt": (_I, [_I, _L, _L, _P, _P, _L, _I, _P, _I, C.POINTER(_P)]),
    "semk_hostplan_scalar": (_L, [_P, _I]),
    "semk_hostplan_array": (_P, [_P, _I, C.POINTER(_L)]),
    "semk_hostplan_destroy": (None, [_P]),
    "semk_partials_len": (_L, [_L, _L]),
    "semk_patch_smem_bytes": (_L, [_I, _I, _L, _L, _L, _L]),
    "semk_resident_ctas": (_L, [_I, _I, _L, _L, _L, _L]),
    "semk_resident_ctas_variant": (_L, [_I, _I, _I, _L, _L, _L, _L]),
    "semk_resident_ctas_sep": (_L, [_I, _I, _I, _I, _L, _L, _L, _L]),
    "semk_patch_smem_bytes_sep": (_L, [_I, _I, _I, _L, _L, _L, _L]),
    "semk_geom_factors_f64": (_I, [_I, _L, _P, _P, _P, _P, _P, _P, _P, _P, _L, _I, _P, _P, _P,
                                   _P, _P, _P, _P]),
    "semk_field_grad_f64": (_I, [_I, _L, _P, _P, _P, _P, _P, _P, _P, _L, _P, _P, _P, _P, _I, _P,
                                 _P, _P, _P, _P, _P, _P]),
    "semk_gfactors_from_invj_f64": (_I, [_I, _L, _P, _P, _P, _P, _L, _I, _P]),
    "semk_poisson_apply_f64": (_I, [C.POINTER(semk_op), _P, _P, _I, _P, _P]),
    "semk_poisson_apply_atomic_f64": (_I, [_I, _L, _L, _P, _P, _P, _L, _I, _P, _P, _P, _P, _I,
                                           _P]),
    "semk_poisson_apply_host_f64": (_I, [C.POINTER(semk_op), _P, _P, _P, _P, _I, _P]),
    "semk_assemble_f64": (_I, [C.POINTER(semk_op), _P, _P, _I, _D, _P]),
    "semk_poisson_local_diag_f64": (_I, [C.POINTER(semk_op), _P, _P, _P]),
    "semk_weighted_local_f64": (_I, [_I, _L, _L, _P, _P, _P, _P, _P, _P]),
    "semk_vec_partials_len": (_L, [_L]),
    "semk_pcg_init_f64": (_I, [_L, _L, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "semk_pcg_update_xr_f64": (_I, [_L, _L, _P, _P, _P, _P, _P, _P, _P, _P]),
    "semk_pcg_update_p_f64": (_I, [_L, _P, _P, _P, _P, _P, _P]),
    "semk_pcg_update_px_f64": (_I, [_L, _P, _P, _P, _P, _P, _P, _P]),
    "semk_dot_f64": (_I, [_L, _P, _P, _P, _P, _P]),
    "semk_pcg_solve_f64": (_I, [C.POINTER(semk_op), _P, _P, _P, _P, _P, _P, _D, _I, _I,
                                C.POINTER(semk_pcg_info), _P]),
    "semk_poisson_apply_bdiag_f64": (_I, [C.POINTER(semk_op), C.POINTER(semk_bdiag), _P, _P, _I,
                                          _P, _P]),
    "semk_pcg_solve_bdiag_f64": (_I, [C.POINTER(semk_op), C.POINTER(semk_bdiag), _P, _P, _P, _P,
                                      _P, _P, _D, _I, _I, C.POINTER(semk_pcg_info), _P]),
    "semk_face_sum_f64": (_I, [_L, _P, _P, _P, _P, _P]),
    "semk_poisson_apply_host_staged_f64":(_I, [C.POINTER(semk_op), C.POINTER(semk_stage), _I, _P, _P,
                                                _P, _P, _I, _P]),
    "semk_poisson_apply_host_batch_f64": (_I, [C.POINTER(semk_op), C.POINTER(semk_stage), _I, _I,
                                               C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                               _P, _P, _P, _P, _I, _P]),
    "semk_scratch_row_stride": (_I, [_I, _I]),
    "semk_scale_gfactors_f64": (_I, [_I, _L, _P, _P, _P, _L, _I, _P]),
    "semk_sc_element_f64": (_I, [_I, _L, _P, _P, _L, _I, _P, _P, _P, _P, _P, _D, _I, _P, _L, _P,
                                 _P, _P, _P, _P, _P, _P]),
    "semk_sc_element_react_f64": (_I, [_I, _L, _P, _P, _L, _I, _P, _P, _P, _P, _P, _D, _I, _P, _L,
                                       _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "semk_sc_load_stored_f64": (_I, [_I, _L, _P, _P, _P, _P, _P, _P, _D, _P, _P, _P]),
    "semk_sc_backsolve_stored_f64": (_I, [_I, _L, _P, _P, _P, _P, _P, _P]),
    "semk_sc_block_max_cols": (_I, [_I]),
    "semk_sc_element_block_f64": (_I, [_I, _L, _P, _L, _I, _P, _P, _P, _P, _P, _I, _I, _P, _L,
                                       C.c_uint32, _P, _P, _L, _P, _L, _P, _L, _P, _P]),
    "semk_sc_load_stored_block_f64": (_I, [_I, _L, _P, _P, _P, _P, _P, _I, _P, _L, C.c_uint32,
                                           _P, _P, _L, _P, _L, _P]),
    "semk_sc_backsolve_stored_block_f64": (_I, [_I, _L, _P, _P, _L, _P, _P, _I, _P, _L, _P]),
    "semk_sc_element_dense_f64": (_I, [_I, _L, _P, _P, _P, _I, _P, _L, _P, _P, _P, _P, _P]),
    "semk_sc_apply_f64": (_I, [C.POINTER(semk_sc_op), _P, _P, _I, _P, _P]),
    "semk_sc_assemble_f64": (_I, [C.POINTER(semk_sc_op), _P, _P, _I, _D, _P]),
    "semk_sc_pcg_solve_f64": (_I, [C.POINTER(semk_sc_op), _P, _P, _P, _P, _P, _P, _D, _I, _I,
                                   C.POINTER(semk_pcg_info), _P]),
    "semk_sc_coarse_elem_f64": (_I, [C.POINTER(semk_sc_op), _P, _P, _P]),
    "semk_sc_coarse_apply_f64": (_I, [_L, C.POINTER(semk_sc_coarse), _P, _P, _I, _P, _P]),
    "semk_sc_coarse_assemble_f64": (_I, [_L, C.POINTER(semk_sc_coarse), _P, _P, _P]),
    "semk_sc_coarse_ell_build_f64": (_I, [C.POINTER(semk_sc_coarse), _I, _P, _P, _P, _P]),
    "semk_sc_coarse_ell_apply_f64": (_I, [C.POINTER(semk_sc_coarse), _P, _P, _P, _P]),
    "semk_sc_top_assemble_f64": (_I, [C.POINTER(semk_sc_coarse), _L, _P, _P, _P, _P, _P]),
    "semk_comm_region_bytes": (_L, [C.c_int32, _L]),
    "semk_comm_allreduce_f64": (_I, [C.POINTER(semk_comm), _P, _L, _P]),
    "semk_pcg_dist_solve_f64": (_I, [C.POINTER(semk_op), C.POINTER(semk_sc_op),
                                     C.POINTER(semk_halo), C.POINTER(semk_comm), _L, _P, _P, _P,
                                     _P, _P, _P, _D, _I, _I, C.POINTER(semk_pcg_info), _P]),
    "semk_sc_mlpcg_solve_f64": (_I, [C.POINTER(semk_sc_op), C.POINTER(semk_sc_coarse),
                                     C.POINTER(semk_sc_top), C.POINTER(semk_ml_dist), _P, _P, _P,
                                     _P, _P, _P, _P, _P, C.POINTER(semk_ml_opts),
                                     C.POINTER(semk_ml_info), _P]),
    "semk_vec_resid_f64": (_I, [_L, _P, _P, _P, _P, _P, _P]),
    "semk_vec_scale_f64": (_I, [_L, _P, _P, _P, _P]),
    "semk_vec_axpy2_f64": (_I, [_L, _D, _P, _P, _P, _P, _P]),
    "semk_vec_xpay_f64": (_I, [_L, _D, _P, _P, _P]),
    "semk_sc_restrict_f64": (_I, [C.POINTER(semk_sc_coarse), _P, _L, _P, _P]),
    "semk_sc_prolong_add_f64": (_I, [_L, C.POINTER(semk_sc_coarse), _P, _P, _P]),
    "semk_values_at_nodes_f64": (_I, [_I, _L, _P, _P, _P, _P, _P, _P]),
    "semk_locate_points_f64": (_I, [_I, _L, _P, _P, _P, _P, _P, _D, _D, _D, _D, _I, _I, _P, _P, _L,
                                    _P, _I, _D, _P, _P, _P]),
    "semk_interpolate_points_f64": (_I, [_I, _L, _P, _P, _P, _P, _P, _P, _P, _P]),
    "semk_halo_region_bytes": (_L, [_L]),
    "semk_peer_alloc": (_I, [_L, C.POINTER(_P), _P]),
    "semk_peer_open": (_I, [_P, C.POINTER(_P)]),
    "semk_peer_close": (_I, [_P]),
    "semk_peer_free": (_I, [_P]),
    "semk_halo_exchange_f64": (_I, [_L, _L, _P, _P, _P, _P, _P, _P, C.c_uint64, _P, _P, _P]),
    "semk_poisson_apply_range_f64": (_I, [C.POINTER(semk_op), _P, _P, _I, _L, _L, _L, _L, _L, _L, _P]),
    "semk_poisson_apply_halo_f64": (_I, [C.POINTER(semk_op), _P, _P, _I, _L, _L, _L,
                                         C.POINTER(semk_halo), _P, _P]),
    "semk_host_structured_maps": (_I, [_L, _L, C.c_int32, _L, _P, C.c_int32]),
    "semk_host_sc_numbering": (_I, [_L, _L, C.c_int32, _P, _P, C.c_int32, _P, C.c_int32, _P,
                                    C.c_int32, _L, C.POINTER(_L), C.POINTER(_L), _P, C.c_int32]),
    "semk_stokes_smem_bytes": (_L, [_I, _I, _L, _L, _L, _L]),
    "semk_stokes_factors_f64": (_I, [_I, _L, _P, _P, _P, _P, _P, _L, _I, _P]),
    "semk_stokes_linearize_f64": (_I, [_I, _L, _P, _P, _P, _P, _P, _P, _P, _D, _P, _L, _I, _P]),
    "semk_stokes_apply_f64": (_I, [C.POINTER(semk_stokes_op), _P, _P, _I, _D, _P]),
    "semk_stokes_local_diag_f64": (_I, [C.POINTER(semk_stokes_op), _P, _L, _P, _P, _P, _P, _P]),
    "semk_scatter_fix_f64": (_I, [_L, _P, _P, _P, _P]),
    "semk_stokes_prec_gamma_f64": (_I, [_L, _P, _P, _P, _P]),
    "semk_stokes_prec_rhs_f64": (_I, [_L, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "semk_stokes_prec_out_f64": (_I, [_L, _P, _P, _P, _P, _P, _P]),
    "semk_sc_rhs_finish_f64": (_I, [_L, _P, _P, _P, _P, _P]),
    "semk_multi_dot_partials_len": (_L, [_I]),
    "semk_multi_dot_f64": (_I, [_L, _I, _P, _L, _P, _P, _P, _P]),
    "semk_multi_axpy_f64": (_I, [_L, _I, _P, _L, _P, _D, _P, _P]),
    "semk_vec_scale_add_f64": (_I, [_L, _D, _P, _P, _P, _P]),
    "semk_block2_apply_f64": (_I, [_L, _P, _P, _P, _P]),
    "semk_block_gram_partials_len": (_L, [_I, _I]),
    "semk_block_gram_f64": (_I, [_L, _I, _P, _L, _I, _P, _L, _P, _P, _P, _P]),
    "semk_block_gram_dfma_f64": (_I, [_L, _I, _P, _L, _I, _P, _L, _P, _P, _P, _P]),
    "semk_block_gram_dmma_f64": (_I, [_L, _I, _P, _L, _I, _P, _L, _P, _P, _P, _P]),
    "semk_block_combine_f64": (_I, [_L, _I, _P, _L, _I, _P, _D, _P, _L, _P]),
}

_lib = None


def load():
    """Load libsemk.so (once).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "libsemk.so not found at %s -- build it with "
                "`python -c 'import __graft_entry__ as g; g.build()'` or "
                "spectralelementmethod_b200/csrc/build.sh.  There is no CPU fallback." % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def host_threads():
    """Threads for the host-side table helpers: all processors, shared between the ranks of
    one box (torchrun exports OMP_NUM_THREADS=1, which is not what set-up code wants)."""
    forced = os.environ.get("SEMK_HOST_THREADS")
    if forced:
        return max(1, int(forced))
    n = os.cpu_count() or 1
    local = int(os.environ.get("LOCAL_WORLD_SIZE", "1") or 1)
    return max(1, min(64, n // max(local, 1)))


def last_error():
    return load().semk_last_error().decode("utf-8", "replace")


def check(code):
    """Map a libsemk status to the reference's exception conventions
    (SURVEY.md 8b 'Error conventions')."""
    if code == OK:
        return
    msg = last_error()
    if code == ERR_INVALID:
        raise ValueError(msg)
    if code == ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    if code == ERR_JACOBIAN:
        raise AssertionError(msg)
    if code == ERR_BREAKDOWN:
        raise SolverFailure(msg)
    raise SemkError(code, msg)


def require_device():
    """Fail loudly when no CUDA device is usable (no CPU fallback)."""
    if not load().semk_device_available():
        raise RuntimeError("spectralelementmethod_b200: no CUDA device available; "
                           "the operator engine has no CPU fallback")


def hostplan(n1, l2g, n_nodes, elem_order=None, elems_per_patch=16, dirichlet=None, threads=None,
             arrays=None):
    """Run the host plan builder (``threads``: for its per-patch passes; default
    ``host_threads()``; same tables for any count); returns (scalars dict, arrays dict of
    numpy copies).  ``arrays``: the SEMK_PA_* tables to copy out (default: all; the full
    per-patch node and index tables are several hundred MB at config 2 and the device only
    needs their deduplicated blocks)."""
    lib = load()
    l2g = np.ascontiguousarray(l2g, dtype=np.uint32).reshape(-1, n1 * n1)
    n_elem = l2g.shape[0]
    order_p = None
    if elem_order is not None:
        elem_order = np.ascontiguousarray(elem_order, dtype=np.int64)
        if elem_order.ndim != 1 or elem_order.size < n_elem:
            raise ValueError("elem_order must have one entry per element (plus -1 padding slots)")
        order_p = elem_order.ctypes.data
    dir_p = None
    if dirichlet is not None:
        dirichlet = np.ascontiguousarray(dirichlet).astype(np.uint8, copy=False)
        if dirichlet.shape != (n_nodes,):
            raise ValueError("dirichlet mask must have one entry per node")
        dir_p = dirichlet.ctypes.data
    handle = _P()
    n_order = 0 if elem_order is None else int(elem_order.size)
    check(lib.semk_hostplan_create_mt(int(n1), n_elem, int(n_nodes), l2g.ctypes.data, order_p, n_order,
                                      int(elems_per_patch), dir_p,
                                      int(host_threads() if threads is None else threads),
                                      C.byref(handle)))
    try:
        scalars = {k: int(lib.semk_hostplan_scalar(handle, k)) for k in range(PS_COUNT)}
        want = None if arrays is None else set(arrays)
        arrays = {}
        for k, dt in PLAN_ARRAY_DTYPES.items():
            if want is not None and k not in want:
                continue
            nb = _L(0)
            ptr = lib.semk_hostplan_array(handle, k, C.byref(nb))
            if nb.value:
                buf = (C.c_char * nb.value).from_address(ptr)
                arrays[k] = np.frombuffer(buf, dtype=dt).copy()
            else:
                arrays[k] = np.zeros(0, dtype=dt)
    finally:
        lib.semk_hostplan_destroy(handle)
    return scalars, arrays
