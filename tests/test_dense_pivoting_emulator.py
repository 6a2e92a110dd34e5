"""Bunch-Kaufman pivoting of the dense solver, checked on its numpy restatement (tests/bk_emulator.py) without a GPU:
the factor reconstructs P A P', its inertia is LAPACK's (dsytrf through the oracle) and numpy's, the transformed solve the
device runs has a backward-stable residual, and the static path these matrices defeat really is defeated."""
import numpy as np
import pytest

import bk_emulator as E
import madnlp_oracle as o


CASES = E.pivot_test_matrices()


def _eig_inertia(A):
    ev = np.linalg.eigvalsh(A)
    return int(np.sum(ev > 0)), int(np.sum(ev == 0)), int(np.sum(ev < 0))


def _check_factor(A, F):
    N = len(A)
    assert sorted(F.perm) == list(range(N))
    # a block permutation: every row stays inside its 128-row block
    assert (F.perm // E.DB == np.arange(N) // E.DB).all()
    Lb = F.l_bd()
    P = A[np.ix_(F.perm, F.perm)]
    scale = (np.abs(Lb) * np.abs(F.lam)) @ np.abs(Lb).T           # |L| |Lambda| |L|': the backward-error scale
    assert np.abs(P - Lb @ np.diag(F.lam) @ Lb.T).max() <= 1e-13 * scale.max()
    # pairs: (first, second), a rotation, one positive and one negative eigenvalue
    first = np.flatnonzero(F.kind == E.KIND_2X2_FIRST)
    assert (F.kind[first + 1] == E.KIND_2X2_SECOND).all()
    assert int(np.sum(F.kind == E.KIND_2X2_SECOND)) == len(first)
    assert np.allclose(F.rot[first] ** 2 + F.rot[first + 1] ** 2, 1.0, rtol=0, atol=1e-15)
    assert (F.lam[first] * F.lam[first + 1] < 0).all()
    assert (first // E.DB == (first + 1) // E.DB).all()          # a pair never straddles two blocks
    assert (np.diag(F.L) == 1.0).all() and (F.L[first + 1, first] == 0.0).all()


@pytest.mark.parametrize("name", sorted(CASES))
def test_emulator_factor_inertia_and_solve(name):
    A = CASES[name]
    F = E.bk_factor(A)
    _check_factor(A, F)
    inertia = F.inertia()
    assert inertia[1] == 0
    assert inertia == _eig_inertia(A)
    assert inertia == o.LapackCPUSolver(np.asfortranarray(A)).factorize().inertia()
    b = np.random.default_rng(len(A)).standard_normal(len(A))
    x = F.solve(b)
    assert np.abs(A @ x - b).max() <= 1e-12 * (np.abs(A).sum(axis=1).max() * np.abs(x).max() + np.abs(b).max())
    # the static path perturbs a pivot of every one of these matrices
    assert E.static_inertia(A)[1] > 0
    assert F.n_2x2() > 0


def test_emulator_spd_takes_plain_1x1_pivots():
    A = E.spd(200, 6)
    F = E.bk_factor(A)
    _check_factor(A, F)
    assert (F.perm == np.arange(200)).all()
    assert (F.kind == E.KIND_1X1).all() and (F.rot == 0).all()
    assert F.inertia() == (200, 0, 0)
    # ... and is then plain LDL^T: D = the pivots of the unpivoted elimination
    Lc = np.linalg.cholesky(A)
    assert np.allclose(F.lam, np.diag(Lc) ** 2, rtol=1e-12, atol=0)


def test_emulator_zero_column_is_perturbed_and_counted():
    """a numerically zero remaining column (|a_pp| and lambda below eps): sign(d) * eps, counted as a zero"""
    A = np.diag([2.0, 0.0, -3.0, 1e-15])
    F = E.bk_factor(A)
    assert list(F.kind) == [E.KIND_1X1, E.KIND_PERTURBED, E.KIND_1X1, E.KIND_PERTURBED]
    assert F.lam[1] == 1e-13 and F.lam[3] == 1e-13
    assert F.inertia() == (1, 2, 1)


def test_schur2_diagonalises():
    rng = np.random.default_rng(0)
    for _ in range(100):
        a, b, c = rng.standard_normal(3) * 10.0 ** rng.integers(-3, 3, 3)
        cs, sn, l1, l2 = E.schur2(a, b, c)
        Q = np.array([[cs, sn], [-sn, cs]])
        D = np.array([[a, b], [b, c]])
        assert np.abs(Q @ np.diag([l1, l2]) @ Q.T - D).max() <= 1e-14 * np.abs(D).max()


# ------------------------------------------------------------------------------------------------ C ABI (host side)
def test_pivoting_option_defaults_to_static_and_the_sparse_solver_rejects_bunch_kaufman():
    import ctypes as C
    from madnlp_jl_b200 import capi
    from madnlp_jl_b200.linear_solvers import B200DenseSolver
    opt = capi.default_options()
    assert opt.pivoting == capi.B2_PIVOT_STATIC == 0
    assert C.sizeof(capi.Options) == 72                        # pivoting took one of the reserved words
    assert B200DenseSolver.default_options(pivoting="bunchkaufman").pivoting == capi.B2_PIVOT_BUNCH_KAUFMAN
    assert B200DenseSolver.default_options(pivoting="static").pivoting == capi.B2_PIVOT_STATIC
    with pytest.raises(ValueError):
        B200DenseSolver.default_options(pivoting="rook")
    colptr = np.array([0, 2, 3], dtype=np.int32); rowval = np.array([0, 1, 1], dtype=np.int32)
    h = C.c_void_p()
    opt.pivoting = capi.B2_PIVOT_BUNCH_KAUFMAN
    assert capi.lib.b2_create_symbolic_only(2, 3, colptr.ctypes.data, rowval.ctypes.data, C.byref(opt), None, C.byref(h)) == capi.B2_ERR_INVALID
    assert "sparse solver" in capi.last_error()
    assert capi.lib.b2_create(2, 3, colptr.ctypes.data, rowval.ctypes.data, None, C.byref(opt), None, C.byref(h)) == capi.B2_ERR_INVALID
    assert capi.lib.b2d_pivot_info(None, None, None, None, None) == capi.B2_ERR_INVALID
