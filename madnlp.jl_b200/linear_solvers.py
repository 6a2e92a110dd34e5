"""Host-side mirror of MadNLP's AbstractLinearSolver plugin surface
(src/LinearSolvers/linearsolvers.jl:13-95) for the B200 back-ends.

Same method names and meaning as the reference (Python spelling: `factorize!` -> `factorize`):
    Solver(A; opt)            constructor, A kept BY REFERENCE, symbolic analysis happens here
    factorize()               numeric factorisation of the current values of A
    solve_linear_system(x)    in place
    is_inertia() / inertia()  -> (num_pos, num_zero, num_neg)   (code order, src/IPM/solver.jl:626)
    improve()                 -> bool
    introduce(), input_type, default_options(), is_supported(T), is_async()
Everything numeric is a call through the C ABI (capi.py) into hand-written sm_100a kernels.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import capi
from .capi import lib, check


@dataclass
class DeviceCSC:
    """Lower-triangular SparseMatrixCSC{Float64,Int32} with the value vector on the device
    (cf. CuSparseMatrixCSC in lib/MadNLPGPU).  colptr/rowval are 0-based host arrays."""
    m: int
    n: int
    colptr: np.ndarray   # int32 [n+1], host
    rowval: np.ndarray   # int32 [nnz], host
    nzval: "object"      # torch.cuda float64 [nnz]

    @property
    def nnz(self):
        return int(self.colptr[-1])


class B200SparseSolver:
    """Supernodal multifrontal LDL^T with static pivoting on one B200
    (role of CUDSSSolver, lib/MadNLPGPU/ext/MadNLPGPUCUDAExt/cudss.jl:88-214)."""
    input_type = "csc"

    def __init__(self, csc: DeviceCSC, opt: capi.Options | None = None, stream=None):
        capi.require_device()
        assert csc.m == csc.n
        self.csc = csc                      # kept by reference (cudss.jl:154-158)
        self.opt = opt if opt is not None else self.default_options()
        self._h = C.c_void_p()
        self.colptr = np.ascontiguousarray(csc.colptr, dtype=np.int32)
        self.rowval = np.ascontiguousarray(csc.rowval, dtype=np.int32)
        check(lib.b2_create(csc.n, int(self.colptr[-1]), self.colptr.ctypes.data, self.rowval.ctypes.data,
                            csc.nzval.data_ptr(), C.byref(self.opt), None, C.byref(self._h)))
        self.n = csc.n
        self.stream = stream

    def __del__(self):
        h = getattr(self, "_h", None)
        if h and lib is not None:
            lib.b2_destroy(h)
            self._h = None

    @staticmethod
    def default_options(**kw):
        return capi.default_options(**kw)

    @staticmethod
    def is_supported(dtype) -> bool:
        return np.dtype(dtype) == np.float64

    def introduce(self) -> str:
        return f"b200kkt multifrontal LDL^T v{lib.b2_version()}"

    def is_async(self) -> bool:
        return True                          # returns before the GPU is done (linearsolvers.jl:67-69)

    def factorize(self):
        check(lib.b2_factorize(self._h, capi.stream_ptr(self.stream)))
        return self

    def solve_linear_system(self, x):
        assert x.is_cuda and x.dtype.is_floating_point and x.is_contiguous()
        nrhs = 1 if x.dim() == 1 else x.shape[0]
        check(lib.b2_solve(self._h, x.data_ptr(), nrhs, capi.stream_ptr(self.stream)))
        return x

    def is_inertia(self) -> bool:
        return True

    def inertia(self):
        p, z, n = C.c_int64(), C.c_int64(), C.c_int64()
        check(lib.b2_inertia(self._h, C.byref(p), C.byref(z), C.byref(n), capi.stream_ptr(self.stream)))
        return (p.value, z.value, n.value)

    def inertia_enqueue(self):
        """queue the D2H copy of the pivot counts; `inertia_fetch` is valid once the stream has been synchronised"""
        check(lib.b2_inertia_enqueue(self._h, capi.stream_ptr(self.stream)))

    def inertia_fetch(self):
        p, z, n = C.c_int64(), C.c_int64(), C.c_int64()
        check(lib.b2_inertia_fetch(self._h, C.byref(p), C.byref(z), C.byref(n)))
        return (p.value, z.value, n.value)

    def improve(self) -> bool:
        ch = C.c_int32(0)
        check(lib.b2_improve(self._h, C.byref(ch)))
        return bool(ch.value)

    def stats(self) -> dict:
        st = capi.Stats()
        check(lib.b2_get_stats(self._h, C.byref(st)))
        return st.as_dict()

    def perm(self) -> np.ndarray:
        p = np.empty(self.n, dtype=np.int32)
        check(lib.b2_get_perm(self._h, p.ctypes.data))
        return p


class B200DenseSolver:
    """Blocked dense LDL^T on the fp64 tensor pipe (role of LapackCUDASolver / LapackCPUSolver{BUNCHKAUFMAN},
    src/LinearSolvers/lapack.jl:164-172, cusolver.jl:150-187).  `A` is an N x N column-major device matrix kept by
    reference; only its lower triangle is read.

    Pivoting: ``default_options(pivoting="static")`` (default) takes 1 x 1 pivots in order and perturbs |d| < pivot_eps;
    ``pivoting="bunchkaufman"`` takes Bunch-Kaufman 1 x 1 / 2 x 2 pivots with the search bounded to each 128 x 128 diagonal
    block (N <= 128 * number of SMs)."""
    input_type = "dense"
    PIVOTING = {"static": capi.B2_PIVOT_STATIC, "bunchkaufman": capi.B2_PIVOT_BUNCH_KAUFMAN}

    def __init__(self, A, opt: capi.Options | None = None, stream=None):
        capi.require_device()
        self.A = A                           # torch.cuda float64, shape (N, N), memory = column-major matrix
        N = A.shape[0]
        assert A.shape[0] == A.shape[1] and A.is_contiguous()
        self.n = N
        self.opt = opt if opt is not None else self.default_options()
        self._h = C.c_void_p()
        check(lib.b2d_create(N, N, A.data_ptr(), C.byref(self.opt), C.byref(self._h)))
        self.stream = stream

    def __del__(self):
        h = getattr(self, "_h", None)
        if h and lib is not None:
            lib.b2d_destroy(h)
            self._h = None

    @classmethod
    def default_options(cls, **kw):
        if isinstance(kw.get("pivoting"), str):
            if kw["pivoting"] not in cls.PIVOTING:
                raise ValueError(f"pivoting must be one of {sorted(cls.PIVOTING)}, not {kw['pivoting']!r}")
            kw["pivoting"] = cls.PIVOTING[kw["pivoting"]]
        return capi.default_options(**kw)

    @staticmethod
    def is_supported(dtype) -> bool:
        return np.dtype(dtype) == np.float64

    def introduce(self) -> str:
        mode = "Bunch-Kaufman pivoting" if self.opt.pivoting == capi.B2_PIVOT_BUNCH_KAUFMAN else "static pivoting"
        return f"b200kkt dense LDL^T (DMMA, {mode}) v{lib.b2_version()}"

    def pivot_info(self):
        """pivots of the last factorisation: (perm, kind, n_2x2, n_perturbed) with perm[new] = old and kind[i] one of
        capi.B2_PIVOT_KIND_*; a static-pivoting solver reports the identity and only 1 x 1 pivots"""
        perm = np.empty(self.n, dtype=np.int32)
        kind = np.empty(self.n, dtype=np.int8)
        n2, npert = C.c_int64(), C.c_int64()
        check(lib.b2d_pivot_info(self._h, perm.ctypes.data, kind.ctypes.data, C.byref(n2), C.byref(npert)))
        return perm, kind, n2.value, npert.value

    def is_async(self) -> bool:
        return True

    def factorize(self):
        check(lib.b2d_factorize(self._h, capi.stream_ptr(self.stream)))
        return self

    def solve_linear_system(self, x):
        nrhs = 1 if x.dim() == 1 else x.shape[0]
        check(lib.b2d_solve(self._h, x.data_ptr(), nrhs, capi.stream_ptr(self.stream)))
        return x

    def is_inertia(self) -> bool:
        return True

    def inertia(self):
        p, z, n = C.c_int64(), C.c_int64(), C.c_int64()
        check(lib.b2d_inertia(self._h, C.byref(p), C.byref(z), C.byref(n), capi.stream_ptr(self.stream)))
        return (p.value, z.value, n.value)

    def inertia_enqueue(self):
        check(lib.b2d_inertia_enqueue(self._h, capi.stream_ptr(self.stream)))

    def inertia_fetch(self):
        p, z, n = C.c_int64(), C.c_int64(), C.c_int64()
        check(lib.b2d_inertia_fetch(self._h, C.byref(p), C.byref(z), C.byref(n)))
        return (p.value, z.value, n.value)

    def improve(self) -> bool:
        return False
