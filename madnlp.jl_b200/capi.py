"""ctypes binding of the C ABI in include/b200kkt.h (libb200kkt.so, built in-tree by csrc/Makefile).

This is the same boundary a MadNLP.jl maintainer would bind with `ccall` (INTEGRATION.md); the Python host
layer above it only mirrors the reference's plugin interface.  There is NO fallback: if the shared library is
missing the import fails loudly, and every numeric entry point needs a CUDA device.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libb200kkt.so")

B2_OK = 0
B2_ERR_INVALID, B2_ERR_CUDA, B2_ERR_SYMBOLIC, B2_ERR_FACTORIZATION, B2_ERR_SOLVE, B2_ERR_NO_DEVICE = 1, 2, 3, 4, 5, 6
ORDER_METIS_ND, ORDER_MINDEG, ORDER_NATURAL, ORDER_USER = 0, 1, 2, 3
B2_PIVOT_STATIC, B2_PIVOT_BUNCH_KAUFMAN = 0, 1
B2_PIVOT_KIND_1X1, B2_PIVOT_KIND_2X2_FIRST, B2_PIVOT_KIND_2X2_SECOND, B2_PIVOT_KIND_PERTURBED = 0, 1, 2, 3


class B2Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"b200kkt error {code}: {msg}")
        self.code = code


# exception types of the reference (src/LinearSolvers/linearsolvers.jl:133-137)
class SymbolicException(B2Error):
    pass


class FactorizationException(B2Error):
    pass


class SolveException(B2Error):
    pass


class InertiaException(RuntimeError):
    pass


class Options(C.Structure):
    _fields_ = [
        ("ordering", C.c_int32), ("nemin", C.c_int32), ("relax_zeros", C.c_double), ("pivot_eps", C.c_double),
        ("use_cuda_graph", C.c_int32), ("small_front_max", C.c_int32), ("n_parts", C.c_int32), ("part_rank", C.c_int32),
        ("kkt_n_primal", C.c_int32), ("fuse_max_fronts", C.c_int32), ("dep_schedule", C.c_int32), ("chain_merge_f", C.c_int32),
        ("pivoting", C.c_int32), ("reserved", C.c_int32 * 3),
    ]


class Stats(C.Structure):
    _fields_ = [(k, C.c_int64) for k in (
        "n", "nnz_a", "nnz_l", "flops", "n_supernodes", "n_levels", "max_front", "n_small_fronts", "n_big_fronts",
        "factor_bytes", "workspace_bytes", "sep_rows", "n_factor_launches", "n_solve_launches", "n_perturbed")]

    def as_dict(self):
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


class SymbolicSizes(C.Structure):
    _fields_ = [(k, C.c_int64) for k in (
        "n", "n_supernodes", "n_rows", "n_children", "n_rel", "n_amap", "n_levels", "lval_size", "cb_size")]


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            f"(or `make -C madnlp.jl_b200/csrc`). The B200 KKT path has no CPU fallback.")
    return C.CDLL(LIB_PATH)


lib = _load()

_p = C.c_void_p
_i32, _i64, _f64 = C.c_int32, C.c_int64, C.c_double
_PP = C.POINTER(C.c_void_p)

# name -> (restype, argtypes); every symbol declared in include/b200kkt.h appears here
PROTOTYPES = {
    "b2_last_error": (C.c_char_p, []),
    "b2_version": (C.c_int, []),
    "b2_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "b2_options_default": (C.c_int, [C.POINTER(Options)]),
    "b2_create": (C.c_int, [_i32, _i64, _p, _p, _p, C.POINTER(Options), _p, _PP]),
    "b2_create_symbolic_only": (C.c_int, [_i32, _i64, _p, _p, C.POINTER(Options), _p, _PP]),
    "b2_destroy": (C.c_int, [_p]),
    "b2_set_values_ptr": (C.c_int, [_p, _p]),
    "b2_factorize": (C.c_int, [_p, _p]),
    "b2_inertia": (C.c_int, [_p, C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_i64), _p]),
    "b2_inertia_enqueue": (C.c_int, [_p, _p]),
    "b2_inertia_fetch": (C.c_int, [_p, C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_i64)]),
    "b2_solve": (C.c_int, [_p, _p, _i32, _p]),
    "b2_improve": (C.c_int, [_p, C.POINTER(_i32)]),
    "b2_get_stats": (C.c_int, [_p, C.POINTER(Stats)]),
    "b2_get_perm": (C.c_int, [_p, _p]),
    "b2_exchange_buffer": (C.c_int, [_p, _PP, C.POINTER(_i64), C.POINTER(_i64)]),
    "b2_exchange_vector": (C.c_int, [_p, _PP, C.POINTER(_i64)]),
    "b2_inertia_parts": (C.c_int, [_p, C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_i64), _p]),
    "b2_factorize_local": (C.c_int, [_p, _p]),
    "b2_factorize_top": (C.c_int, [_p, _p]),
    "b2_solve_fwd_local": (C.c_int, [_p, _p, _p]),
    "b2_solve_top": (C.c_int, [_p, _p, _p]),
    "b2_solve_bwd_local": (C.c_int, [_p, _p, _p]),
    "b2_owned_mask": (C.c_int, [_p, _p]),
    "b2_symbolic_query": (C.c_int, [_p, C.POINTER(SymbolicSizes)]),
    "b2_symbolic_export": (C.c_int, [_p] + [_p] * 13),
    "b2_symbolic_owner": (C.c_int, [_p, _p]),
    "b2_symbolic_exchange": (C.c_int, [_p, _p, C.POINTER(_i64), C.POINTER(_i64)]),
    "b2_debug_get_factor": (C.c_int, [_p, _p, _p]),
    "b2_debug_profile_front": (C.c_int, [_p, _i32, _i32, _p]),
    "b2d_debug_trace": (C.c_int, [_p, _p, _i64, C.POINTER(_i64)]),
    "b2_debug_trace": (C.c_int, [_p, _p, _p, _p, _p, _i64, C.POINTER(_i64)]),
    "b2d_create": (C.c_int, [_i32, _i32, _p, C.POINTER(Options), _PP]),
    "b2d_destroy": (C.c_int, [_p]),
    "b2d_factorize": (C.c_int, [_p, _p]),
    "b2d_inertia": (C.c_int, [_p, C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_i64), _p]),
    "b2d_inertia_enqueue": (C.c_int, [_p, _p]),
    "b2d_inertia_fetch": (C.c_int, [_p, C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_i64)]),
    "b2d_solve": (C.c_int, [_p, _p, _i32, _p]),
    "b2d_pivot_info": (C.c_int, [_p, _p, _p, C.POINTER(_i64), C.POINTER(_i64)]),
    "b2_condensed_symbolic_device": (C.c_int, [_i32, _i32, _p, _p, _p, _p, _PP, C.POINTER(_i64), _p]),
    "b2_coo_to_csc_device": (C.c_int, [_i32, _i32, _i64, _p, _p, _p, _p, _p, C.POINTER(_i64), _p]),
    "b2d_ozaki_plan_create": (C.c_int, [_i32, _i32, _PP]),
    "b2d_ozaki_plan_destroy": (C.c_int, [_p]),
    "b2d_condensed_assemble_ozaki": (C.c_int, [_p, _i32, _i32, _i32, _i32] + [_p] * 9),
    "b2d_ozaki_plan_status": (C.c_int, [_p, C.POINTER(_i32), _p]),
    "b2d_kkt_create": (C.c_int, [_i32, _i32, _i32, _p, _PP]),
    "b2d_kkt_destroy": (C.c_int, [_p]),
    "b2d_kkt_solve_pre": (C.c_int, [_p] * 10 + [_p]),
    "b2d_kkt_solve_post": (C.c_int, [_p] * 12 + [_p]),
    "b2d_kkt_mul": (C.c_int, [_p] * 10 + [_f64, _f64, _p, _p, _p]),
    "b2d_gemv_n": (C.c_int, [_i32, _i32, _i32, _p, _p, _p, _f64, _f64, _p]),
    "b2d_gemv_t": (C.c_int, [_i32, _i32, _i32, _p, _p, _p, _f64, _f64, _p]),
    "b2d_symv_lower": (C.c_int, [_i32, _i32, _p, _p, _p, _f64, _f64, _p]),
    "b2_coo_to_csc": (C.c_int, [_i32, _i32, _i64, _p, _p, _p, _p, _p, C.POINTER(_i64)]),
    "b2_transfer_plan_create": (C.c_int, [_i64, _i64, _p, _PP]),
    "b2_transfer_plan_destroy": (C.c_int, [_p]),
    "b2_transfer": (C.c_int, [_p, _p, _p, _p]),
    "b2_condensed_symbolic": (C.c_int, [_i32, _i32, _p, _p, _p, _p, _PP, C.POINTER(_i64)]),
    "b2_condensed_pattern": (C.c_int, [_p, _p, _p]),
    "b2_condensed_plan_sizes": (C.c_int, [_p, C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_i64)]),
    "b2_condensed_plan_destroy": (C.c_int, [_p]),
    "b2_condensed_assemble": (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _p]),
    "b2d_condensed_assemble": (C.c_int, [_i32, _i32, _i32, _i32, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "b2_bounds_create": (C.c_int, [_i64, _i64, _i64, _p, _p, _PP]),
    "b2_bounds_destroy": (C.c_int, [_p]),
    "b2_set_aug_diagonal": (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _p]),
    "b2_regularize_diagonal": (C.c_int, [_i64, _i64, _f64, _f64, _p, _p, _p, _p]),
    "b2_reduce_rhs": (C.c_int, [_p, _i64, _p, _p, _p, _p]),
    "b2_finish_aug_solve": (C.c_int, [_p, _i64, _p, _p, _p, _p, _p, _p]),
    "b2_spmv_plan_create": (C.c_int, [_i32, _i32, _p, _p, _PP]),
    "b2_spmv_plan_destroy": (C.c_int, [_p]),
    "b2_spmv_n": (C.c_int, [_p, _p, _p, _p, _f64, _f64, _p]),
    "b2_spmv_t": (C.c_int, [_p, _p, _p, _p, _f64, _f64, _p]),
    "b2_spmv_symlower": (C.c_int, [_p, _p, _p, _p, _f64, _f64, _p]),
    "b2_kktmul": (C.c_int, [_p, _i64, _p, _p, _p, _p, _p, _p, _f64, _f64, _p, _p, _p]),
    "b2_condensed_solve_pre": (C.c_int, [_p, _p, _i64, _i64, _p, _p, _p, _p, _p, _p, _p, _p]),
    "b2_condensed_solve_post": (C.c_int, [_p, _p, _i64, _i64, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "b2_condensed_kkt_mul": (C.c_int, [_p, _p, _p, _i64, _i64, _p, _p, _p, _p, _p, _p, _p, _p, _f64, _f64, _p, _p, _p]),
    "b2_condensed_kkt_mul_norm": (C.c_int, [_p, _p, _p, _i64, _i64, _p, _p, _p, _p, _p, _p, _p, _p, _f64, _f64, _p, _p, _p, _p]),
    "b2_get_alpha_max": (C.c_int, [_p, _p, _p, _p, _p, _f64, _p, _p]),
    "b2_get_alpha_z": (C.c_int, [_p, _p, _p, _p, _p, _f64, _p, _p]),
    "b2_get_varphi": (C.c_int, [_p, _f64, _p, _p, _p, _f64, _p, _p]),
    "b2_get_varphi_d": (C.c_int, [_p, _p, _p, _p, _p, _p, _f64, _p, _p]),
    "b2_get_inf_du": (C.c_int, [_p, _p, _p, _p, _p, _f64, _p, _p]),
    "b2_get_inf_compl": (C.c_int, [_p, _p, _p, _p, _p, _p, _f64, _f64, _p, _p]),
    "b2_get_average_complementarity": (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _p]),
    "b2_get_min_complementarity": (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _p]),
    "b2_get_rel_search_norm": (C.c_int, [_p, _i64, _p, _p, _p, _p]),
    "b2_get_sd": (C.c_int, [_p, _i64, _p, _p, _p, _f64, _p, _p]),
    "b2_get_sc": (C.c_int, [_p, _p, _p, _f64, _p, _p]),
    "b2_set_aug_rhs": (C.c_int, [_p, _i64, _p, _p, _p, _p, _p, _p, _p, _p, _f64, _p, _p]),
    "b2_richardson_begin": (C.c_int, [_i64, _p, _p, _p, _p, _p]),
    "b2_richardson_update": (C.c_int, [_i64, _p, _p, _p, _p, _p]),
    "b2_copy_many": (C.c_int, [_i32, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(_i64), _p]),
    "b2_norm_inf": (C.c_int, [_i64, _p, _p, _p]),
    "b2_axpy": (C.c_int, [_i64, _f64, _p, _p, _p]),
    "b2_copy": (C.c_int, [_i64, _p, _p, _p]),
    "b2_fill": (C.c_int, [_i64, _f64, _p, _p]),
}

for _name, (_res, _args) in PROTOTYPES.items():
    _fn = getattr(lib, _name)          # AttributeError here = header/library mismatch: fail loudly
    _fn.restype = _res
    _fn.argtypes = _args


def last_error() -> str:
    return (lib.b2_last_error() or b"").decode()


_EXC = {B2_ERR_SYMBOLIC: SymbolicException, B2_ERR_FACTORIZATION: FactorizationException, B2_ERR_SOLVE: SolveException}


def check(rc: int):
    if rc != B2_OK:
        raise _EXC.get(rc, B2Error)(rc, last_error())


def device_count() -> int:
    n = C.c_int(0)
    rc = lib.b2_device_count(C.byref(n))
    return n.value if rc == B2_OK else 0


def require_device():
    if device_count() == 0:
        raise B2Error(B2_ERR_NO_DEVICE, "no CUDA device visible; the B200 KKT path has no CPU fallback")


def default_options(**kw) -> Options:
    o = Options()
    check(lib.b2_options_default(C.byref(o)))
    for k, v in kw.items():
        if not hasattr(o, k):
            raise TypeError(f"unknown b2 option {k!r}")
        setattr(o, k, v)
    return o


def ptr(t):
    """device/host pointer of a torch tensor or numpy array (or None)."""
    if t is None:
        return None
    if hasattr(t, "data_ptr"):
        return t.data_ptr()
    return t.ctypes.data


def stream_ptr(stream=None):
    if stream is None:
        import torch
        return torch.cuda.current_stream().cuda_stream
    return getattr(stream, "cuda_stream", stream)
