"""Bunch-Kaufman pivoting of the dense solver on the device (B2_PIVOT_BUNCH_KAUFMAN through B200DenseSolver): inertia equal
to LAPACK dsytrf and to the eigenvalues, the same pivots as the numpy restatement (tests/bk_emulator.py) wherever no
decision is within rounding of its threshold, backward-stable solves, on matrices that defeat static pivoting; the
DenseCondensedKKTSystem with a nonconvex Hessian and du_diag = 0; graph capture and re-factorisation; the C ABI."""
import ctypes as C

import numpy as np
import pytest

import bk_emulator as E
import madnlp_oracle as o
import madnlp_jl_b200 as pkg

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

W = pkg.workloads
capi = pkg.capi


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _colmajor(A):
    """device tensor whose memory is the column-major matrix A (what b2d_* reads)"""
    return _dev(np.asarray(A, dtype=np.float64).T)


def _solver(buf, **kw):
    from madnlp_jl_b200.linear_solvers import B200DenseSolver
    return B200DenseSolver(buf, B200DenseSolver.default_options(**kw))


def _rel_residual(A, x, b):
    return np.abs(A @ x - b).max() / (np.abs(A).sum(axis=1).max() * np.abs(x).max() + np.abs(b).max())


def _eig_inertia(A):
    ev = np.linalg.eigvalsh(A)
    return int(np.sum(ev > 0)), int(np.sum(ev == 0)), int(np.sum(ev < 0))


CASES = E.pivot_test_matrices(sizes=(7, 128, 129, 300, 513, 1000, 4096))


@pytest.mark.parametrize("name", list(CASES))
def test_bunch_kaufman_inertia_pivots_and_residual(name):
    """N <= 512 runs the step-by-step schedule, larger N the look-ahead one (general branch)"""
    _need_gpu()
    A = CASES[name]
    N = len(A)
    b = np.random.default_rng(N).standard_normal(N)
    M = _solver(_colmajor(A), pivoting="bunchkaufman")
    assert "Bunch-Kaufman" in M.introduce()
    M.factorize()
    inertia = M.inertia()
    perm, kind, n2, npert = M.pivot_info()
    assert npert == 0 and inertia[1] == 0
    assert inertia == _eig_inertia(A) == o.LapackCPUSolver(np.asfortranarray(A)).factorize().inertia()
    F = E.bk_factor(A)
    assert n2 == int(np.sum(kind == E.KIND_2X2_FIRST)) > 0
    if F.margin > 1e-6:
        assert (perm == F.perm).all() and (kind == F.kind).all()
    x = M.solve_linear_system(_dev(b)).cpu().numpy()
    assert _rel_residual(A, x, b) <= 1e-12
    # the static solver on the same matrix perturbs a pivot or loses the solution
    S = _solver(_colmajor(A))
    S.factorize()
    xs = S.solve_linear_system(_dev(b)).cpu().numpy()
    assert S.inertia()[1] > 0 or _rel_residual(A, xs, b) > 1e-6


def test_bunch_kaufman_on_spd_is_static_pivoting():
    _need_gpu()
    A = E.spd(600, 6)
    b = np.random.default_rng(1).standard_normal(600)
    M = _solver(_colmajor(A), pivoting="bunchkaufman"); M.factorize()
    S = _solver(_colmajor(A)); S.factorize()
    perm, kind, n2, npert = M.pivot_info()
    assert (perm == np.arange(600)).all() and (kind == E.KIND_1X1).all() and n2 == 0 and npert == 0
    assert M.inertia() == S.inertia() == (600, 0, 0)
    x = M.solve_linear_system(_dev(b)).cpu().numpy()
    xs = S.solve_linear_system(_dev(b)).cpu().numpy()
    assert np.abs(x - xs).max() <= 1e-12 * np.abs(xs).max()


def _kkt_pair(qp, it, hess, opt):
    from madnlp_jl_b200 import kkt as K
    cb = o.Callback(qp.n, qp.m, [], [], [], [], qp.ind_ineq, qp.ind_lb, qp.ind_ub)
    kc = o.DenseCondensedKKTSystem(cb)
    kg = K.DenseCondensedKKTSystem(cb, opt_linear_solver=opt)
    for k in (kc, kg):
        k.initialize()
    kc.hess[:] = hess; kc.jac[:] = qp.A
    kg.set_dense(hess_np=hess, jac_np=qp.A)
    for name in ("reg", "du_diag", "l_diag", "u_diag", "l_lower", "u_lower"):
        getattr(kc, name)[:] = it[name]
        getattr(kg, name).copy_(_dev(it[name]))
    o.set_aug_diagonal_(kc); kc.build_kkt()
    kg.set_aug_diagonal_(); kg.build_kkt()
    kc.linear_solver.factorize(); kg.linear_solver.factorize()
    return kc, kg


def _refined(kc, kg, rhs):
    from madnlp_jl_b200 import kkt as K
    from madnlp_jl_b200.richardson import RichardsonIterator
    b = o.UnreducedKKTVector.for_kkt(kc); b.full()[:] = rhs
    x = o.UnreducedKKTVector.for_kkt(kc); w = o.UnreducedKKTVector.for_kkt(kc)
    okc, _, _ = o.solve_refine(x, kc, b, w)
    dc = x.full().copy()
    bg = K.UnreducedKKTVector.for_kkt(kg); bg.values.copy_(_dev(rhs))
    xg = K.UnreducedKKTVector.for_kkt(kg); wg = K.UnreducedKKTVector.for_kkt(kg)
    okg = RichardsonIterator(kg).solve_refine(xg, bg, wg)
    return dc, okc, xg.values.cpu().numpy(), okg


def test_dense_condensed_nonconvex_zero_dual_block():
    """nonconvex Hessian (-1e6 P: its negative curvature survives the barrier terms) and du_diag = 0: inertia of the pivoted
    solver = LapackCPUSolver's, refined directions agree"""
    _need_gpu()
    from madnlp_jl_b200.linear_solvers import B200DenseSolver
    qp = W.dense_qp(n=320, m=130, n_eq=24, seed=3)
    it = W.dense_qp_iterate(qp, mu=1e-3, seed=4)
    assert (it["du_diag"] == 0).all()
    kc, kg = _kkt_pair(qp, it, -1e6 * qp.P, B200DenseSolver.default_options(pivoting="bunchkaufman"))
    inertia = kg.linear_solver.inertia()
    assert inertia == kc.linear_solver.inertia()
    assert inertia[2] > qp.m - len(qp.ind_ineq)                    # nonconvex: more negative eigenvalues than equality rows
    assert kg.linear_solver.pivot_info()[3] == 0
    dc, okc, dg, okg = _refined(kc, kg, it["rhs"])
    assert okc and okg
    assert np.abs(dg - dc).max() / np.abs(dc).max() <= 1e-8


@pytest.mark.parametrize("n_eq", [0, 24])
def test_dense_condensed_convex_same_as_static(n_eq):
    """the convex QP of test_dense_condensed_qp: pivoted and static modes agree"""
    _need_gpu()
    from madnlp_jl_b200.linear_solvers import B200DenseSolver
    qp = W.dense_qp(n=320, m=130, n_eq=n_eq, seed=3)
    it = W.dense_qp_iterate(qp, mu=1e-3, seed=4)
    kc, kp = _kkt_pair(qp, it, qp.P, B200DenseSolver.default_options(pivoting="bunchkaufman"))
    _, ks = _kkt_pair(qp, it, qp.P, None)
    assert kp.linear_solver.inertia() == ks.linear_solver.inertia() == kc.linear_solver.inertia() == (qp.n, 0, n_eq)
    _, _, dp, okp = _refined(kc, kp, it["rhs"])
    _, _, ds, oks = _refined(kc, ks, it["rhs"])
    assert okp and oks
    assert np.abs(dp - ds).max() / np.abs(ds).max() <= 1e-8


def test_graph_capture_and_refactorisation_leave_no_stale_pivots():
    """use_cuda_graph on / off give identical results; one handle re-factorising matrices with different pivot patterns
    gives bit for bit what a fresh handle gives"""
    _need_gpu()
    N = 1000
    mats = [E.random_indefinite(N, 21), E.augmented(700, 300, 22), E.spd(N, 23), E.random_indefinite(N, 21)]
    b = np.random.default_rng(3).standard_normal(N)
    buf = _colmajor(mats[0])
    Mg = _solver(buf, pivoting="bunchkaufman", use_cuda_graph=1)
    Mn = _solver(buf, pivoting="bunchkaufman", use_cuda_graph=0)
    first = None
    for A in mats:
        buf.copy_(_colmajor(A))
        out = []
        for M in (Mg, Mn, _solver(_colmajor(A), pivoting="bunchkaufman")):
            M.factorize()
            perm, kind, n2, npert = M.pivot_info()
            x = M.solve_linear_system(_dev(b)).cpu().numpy()
            out.append((M.inertia(), perm, kind, x))
        for r in out[1:]:
            assert r[0] == out[0][0]
            assert (r[1] == out[0][1]).all() and (r[2] == out[0][2]).all() and (r[3] == out[0][3]).all()
        assert _rel_residual(A, out[0][3], b) <= 1e-12
        if first is None:
            first = out[0]
    assert (out[0][3] == first[3]).all()                            # the first matrix again, after three others


def test_abi_pivoting_option():
    _need_gpu()
    lib = capi.lib
    assert capi.default_options().pivoting == capi.B2_PIVOT_STATIC
    # the sparse solver has no pivoted mode
    colptr = np.array([0, 2, 3], dtype=np.int32); rowval = np.array([0, 1, 1], dtype=np.int32)
    nz = _dev(np.array([1.0, 0.1, 2.0]))
    h = C.c_void_p()
    opt = capi.default_options(pivoting=capi.B2_PIVOT_BUNCH_KAUFMAN)
    assert lib.b2_create(2, 3, colptr.ctypes.data, rowval.ctypes.data, nz.data_ptr(), C.byref(opt), None, C.byref(h)) == capi.B2_ERR_INVALID
    # unknown mode, and more 128-row blocks than SMs: rejected before anything is allocated
    A = _colmajor(np.eye(4))
    assert lib.b2d_create(4, 4, A.data_ptr(), C.byref(capi.default_options(pivoting=2)), C.byref(h)) == capi.B2_ERR_INVALID
    nsm = torch.cuda.get_device_properties(0).multi_processor_count
    big = 128 * nsm + 1
    assert lib.b2d_create(big, big, A.data_ptr(), C.byref(opt), C.byref(h)) == capi.B2_ERR_INVALID
    assert "SMs" in capi.last_error()
    # a static handle reports the identity
    Ad = E.random_indefinite(300, 5)
    S = _solver(_colmajor(Ad))
    assert "static pivoting" in S.introduce()
    S.factorize()
    perm, kind, n2, npert = S.pivot_info()
    assert (perm == np.arange(300)).all() and (kind == 0).all() and n2 == 0
    assert npert == S.inertia()[1] > 0
