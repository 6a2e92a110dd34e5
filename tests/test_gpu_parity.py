"""Parity of the CUDA hot path with the CPU oracle, through the C ABI (via the host mirror of MadNLP's interface).

Bars (SURVEY.md 8c): assembly = BIT-EXACT (integer/index work + fixed summation order); factor/solve = fp64 within
the stated tolerance (step direction rel. inf-norm <= 1e-8 on well-conditioned systems, <= 1e-6 on the ill-conditioned
IPM iterates after Richardson refinement), inertia triple IDENTICAL to the oracle (LAPACK Bunch-Kaufman / eigenvalues).
"""
import numpy as np
import pytest

import madnlp_oracle as o
import madnlp_jl_b200 as pkg

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

W = pkg.workloads


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _cb(st):
    return o.Callback(st.nvar, st.ncon, st.jac_I, st.jac_J, st.hess_I, st.hess_J, st.ind_ineq, st.ind_lb, st.ind_ub)


def _load(kkt_gpu, kkt_cpu, it, dense=False):
    """put one iterate into both the oracle and the device KKT system and assemble"""
    for k, put in ((kkt_cpu, lambda dst, v: dst.__setitem__(slice(None), v)),
                   (kkt_gpu, lambda dst, v: dst.copy_(_dev(v)))):
        k.initialize()
        put(k.get_jacobian(), it.jac); put(k.get_hessian(), it.hess)
        put(k.reg, it.reg + 1e-8); put(k.du_diag, it.du_diag)
        put(k.l_diag, it.l_diag); put(k.u_diag, it.u_diag); put(k.l_lower, it.l_lower); put(k.u_lower, it.u_lower)
        k.compress_jacobian(); k.compress_hessian()
    o.set_aug_diagonal_(kkt_cpu); kkt_cpu.build_kkt()
    kkt_gpu.set_aug_diagonal_(); kkt_gpu.build_kkt()


# ------------------------------------------------------------------------------------------------ assembly
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_transfer_bit_exact(seed):
    """A5 build_kkt!(::SparseKKTSystem) = transfer! (src/matrixtools.jl:79-88): duplicates, empty slots, ragged."""
    _need_gpu()
    from madnlp_jl_b200 import kkt as K
    import ctypes as C
    rng = np.random.default_rng(seed)
    m, n, nnz = 301, 257, 5000
    I = rng.integers(0, m, nnz); J = rng.integers(0, n, nnz)
    I[:500] = I[500:1000]; J[:500] = J[500:1000]
    V = rng.standard_normal(nnz) * 10.0 ** rng.integers(-8, 8, nnz)
    cp0, rv0, mp0 = o.coo_to_csc(I, J, m, n)
    ref = np.zeros(len(rv0)); o.transfer(ref, V, mp0)
    cp, rv, mp = K.coo_to_csc(I, J, m, n)
    plan = K._transfer_plan(mp, len(rv))
    out = torch.full((len(rv),), 7.0, dtype=torch.float64, device="cuda")
    pkg.capi.check(pkg.capi.lib.b2_transfer(plan.h, out.data_ptr(), _dev(V).data_ptr(), None))
    torch.cuda.synchronize()
    assert (out.cpu().numpy() == ref).all()


@pytest.mark.parametrize("case", ["hs15", "case30_synth", "case300_synth"])
def test_condensed_assembly_bit_exact(case):
    """A7 build_kkt!(::SparseCondensedKKTSystem) incl. compress_* and set_aug_diagonal (A1, A3, A4): bit-exact."""
    _need_gpu()
    from madnlp_jl_b200 import kkt as K
    if case == "hs15":
        cb = o.HS15Model.callback()
        it = W.IPMIterate(jac=o.HS15Model.jac_coord(np.array([0.3, 0.7])), hess=o.HS15Model.hess_coord(np.array([0.3, 0.7]), np.array([0.5, -0.2])),
                          reg=np.zeros(4), du_diag=np.array([-1e-3, -2e-3]), l_diag=-np.array([0.3, 0.7]), u_diag=-np.array([0.2]),
                          l_lower=np.array([1e-2, 3e-3]), u_lower=np.array([5e-2]), rhs=np.ones(9), mu=0.1)
    else:
        model, st = W.acopf_case(case)
        cb = _cb(st)
        it = W.ipm_iterates(model, st, 1, seed=11)[0]
        it.du_diag[:] = -1e-6
    kc = o.SparseCondensedKKTSystem(cb)
    kg = K.SparseCondensedKKTSystem(cb)
    assert (kg.aug_com.colptr == kc.aug_colptr).all() and (kg.aug_com.rowval == kc.aug_rowval).all()
    _load(kg, kc, it)
    torch.cuda.synchronize()
    assert (kg.pr_diag.cpu().numpy() == kc.pr_diag).all()
    assert (kg.jt_csc.nzval.cpu().numpy() == kc.jt_nz).all()
    assert (kg.hess_com.nzval.cpu().numpy() == kc.hess_nz).all()
    assert (kg.diag_buffer.cpu().numpy() == kc.diag_buffer).all()
    assert (kg.aug_com.nzval.cpu().numpy() == kc.aug_nz).all()


def test_augmented_assembly_bit_exact():
    """A5 on the SparseKKTSystem value vector layout [pr_diag|hess|jac|-1|du_diag] (augmented.jl:77-107)."""
    _need_gpu()
    from madnlp_jl_b200 import kkt as K
    model, st = W.acopf_case("case30_synth", relax_equality=False)
    cb = _cb(st)
    it = W.ipm_iterates(model, st, 1, seed=5)[0]
    kc = o.SparseKKTSystem(cb, o.DenseLDLInertiaSolver)
    kg = K.SparseKKTSystem(cb)
    _load(kg, kc, it)
    torch.cuda.synchronize()
    assert (kg.V.cpu().numpy() == kc.V).all()
    assert (kg.aug_com.nzval.cpu().numpy() == kc.aug_nz).all()
    assert (kg.jac_com.nzval.cpu().numpy() == kc.jac_nz).all()


# ------------------------------------------------------------------------------------------------ factor / solve
def test_2x2_known_answer_through_sparse_and_dense_solver():
    """The reference's KAT (MadNLPTests.jl:24-51) for both input types (:csc and :dense)."""
    _need_gpu()
    from madnlp_jl_b200.linear_solvers import B200SparseSolver, B200DenseSolver, DeviceCSC
    sol = np.array([0.8542713567839195, 1.4572864321608041])
    csc = DeviceCSC(2, 2, np.array([0, 2, 3], dtype=np.int32), np.array([0, 1, 1], dtype=np.int32), _dev(np.array([1.0, 0.1, 2.0])))
    M = B200SparseSolver(csc)
    assert isinstance(M.introduce(), str)
    M.improve()
    M.factorize()
    assert M.inertia() == (2, 0, 0)
    x = M.solve_linear_system(_dev(np.array([1.0, 3.0])))
    assert np.abs(x.cpu().numpy() - sol).max() < 1e-14
    A = _dev(np.array([[1.0, 0.1], [0.0, 2.0]]))          # memory = column-major [[1,0],[.1,2]] (lower triangle filled)
    D = B200DenseSolver(A)
    D.factorize()
    assert D.inertia() == (2, 0, 0)
    x = D.solve_linear_system(_dev(np.array([1.0, 3.0])))
    assert np.abs(x.cpu().numpy() - sol).max() < 1e-14


HS15_EXPECTED = np.array([0.24987493746873435, 0.00497512437810945, -1.0, -0.7501250625312657, -0.9989999999999999,
                          -0.7493749374687343, -1.001, -1.0007501250625312, 0.9997501250625312])


@pytest.mark.parametrize("kind", ["sparse", "condensed", "dense_condensed"])
def test_hs15_kkt_system_like_reference(kind):
    """test/kkt_test.jl:27-48 / MadNLPTests.test_kkt_system (MadNLPTests.jl:53-110) on the device."""
    _need_gpu()
    from madnlp_jl_b200 import kkt as K
    cb = o.HS15Model.callback()
    typ = dict(sparse=K.SparseKKTSystem, condensed=K.SparseCondensedKKTSystem, dense_condensed=K.DenseCondensedKKTSystem)[kind]
    kkt = K.create_kkt_system(typ, cb)
    n = kkt.num_variables()
    kkt.initialize()
    if kind == "dense_condensed":
        kkt.set_dense(hess_np=o.HS15Model.hess_dense(o.HS15Model.x0, o.HS15Model.y0), jac_np=o.HS15Model.jac_dense(o.HS15Model.x0))
    else:
        kkt.get_jacobian().copy_(_dev(o.HS15Model.jac_coord(o.HS15Model.x0)))
        kkt.get_hessian().copy_(_dev(o.HS15Model.hess_coord(o.HS15Model.x0, o.HS15Model.y0)))
    kkt.compress_jacobian(); kkt.compress_hessian()
    kkt.l_lower.fill_(1e-3); kkt.u_lower.fill_(1e-3)
    kkt.set_aug_diagonal_()
    kkt.build_kkt()
    kkt.linear_solver.factorize()
    x = K.UnreducedKKTVector.for_kkt(kkt)
    x.values.fill_(1.0)
    out1 = kkt.solve_kkt(x)
    assert out1 is x
    y = x.copy(); y.values.zero_()
    out2 = kkt.mul(y, x)
    assert out2 is y
    assert np.allclose(y.values.cpu().numpy(), 1.0, rtol=np.sqrt(np.finfo(float).eps), atol=0)
    assert np.abs(x.values.cpu().numpy() - HS15_EXPECTED).max() < 1e-12
    ni, mi, pi = kkt.linear_solver.inertia()
    assert kkt.is_inertia_correct(ni, mi, pi)
    kkt.regularize_diagonal(1.0, 1.0)
    assert n in (2, 4)


def _refined_direction_cpu(kc, rhs):
    b = o.UnreducedKKTVector.for_kkt(kc); b.full()[:] = rhs
    x = o.UnreducedKKTVector.for_kkt(kc); w = o.UnreducedKKTVector.for_kkt(kc)
    ok, nit, ratio = o.solve_refine(x, kc, b, w)
    return x.full().copy(), ok, ratio


def _refined_direction_gpu(kg, rhs):
    from madnlp_jl_b200 import kkt as K
    from madnlp_jl_b200.richardson import RichardsonIterator
    b = K.UnreducedKKTVector.for_kkt(kg); b.values.copy_(_dev(rhs))
    x = K.UnreducedKKTVector.for_kkt(kg); w = K.UnreducedKKTVector.for_kkt(kg)
    itr = RichardsonIterator(kg)
    ok = itr.solve_refine(x, b, w)
    return x.values.cpu().numpy(), ok, itr.residual_ratio


@pytest.mark.parametrize("case,seed", [("case30_synth", 1), ("case300_synth", 2), ("case1354_pegase", 3)])
def test_condensed_opf_step_direction_and_inertia(case, seed):
    """configs[2]-style: condensed AC-OPF KKT, step direction vs the oracle (dsytrf-based) and identical inertia."""
    _need_gpu()
    from madnlp_jl_b200 import kkt as K
    model, st = W.acopf_case(case)
    cb = _cb(st)
    its = W.ipm_iterates(model, st, 3, seed=seed)
    big = st.nvar > 4000
    kc = o.SparseCondensedKKTSystem(cb, o.UmfpackStandInSolver if big else o.DenseLDLInertiaSolver)
    kg = K.SparseCondensedKKTSystem(cb)
    for it in its:
        _load(kg, kc, it)
        kc.linear_solver.factorize(); kg.linear_solver.factorize()
        inertia = kg.linear_solver.inertia()
        if not big:
            assert inertia == kc.linear_solver.inertia()
        assert kg.is_inertia_correct(*inertia)
        dc, okc, rc = _refined_direction_cpu(kc, it.rhs)
        dg, okg, rg = _refined_direction_gpu(kg, it.rhs)
        assert okc and okg and rg < 1e-8
        assert np.abs(dg - dc).max() / np.abs(dc).max() <= 1e-6
        # unrefined single solve of the condensed system itself, well inside fp64 backward stability
        b = np.random.default_rng(seed).standard_normal(kg.n)
        xg = kg.linear_solver.solve_linear_system(_dev(b)).cpu().numpy()
        Kfull = o.tril_to_full(kc.aug_colptr, kc.aug_rowval, kc.aug_nz, kc.n)
        res = np.abs(Kfull @ xg - b).max() / (abs(Kfull).max() * np.abs(xg).max() + np.abs(b).max())
        assert res < 1e-12


@pytest.mark.parametrize("dep_schedule,chain_merge_f", [(3, 0), (5, 0), (1, 48), (0, 0)])
def test_schedule_and_amalgamation_options_give_the_same_answers(dep_schedule, chain_merge_f):
    """b2_options.dep_schedule (bit 0: single-launch factorisation, bit 1: single-launch flag-driven sweeps, bit 2: hybrid sweeps --
    fused bottom subtrees + one flag-driven launch for the tree above them; 0: level launches) and
    chain_merge_f (only children absorbed while the front stays team-class) change the schedule / the supernode partition, never the
    mathematics: same inertia as the oracle, refined direction within 1e-6, single-solve residual within fp64 backward stability."""
    _need_gpu()
    from madnlp_jl_b200 import kkt as K
    model, st = W.acopf_case("case300_synth")
    cb = _cb(st)
    it = W.ipm_iterates(model, st, 1, seed=5)[0]
    kc = o.SparseCondensedKKTSystem(cb, o.DenseLDLInertiaSolver)
    opt = pkg.capi.default_options(dep_schedule=dep_schedule, chain_merge_f=chain_merge_f)
    kg = K.create_kkt_system(K.SparseCondensedKKTSystem, cb, None, opt)
    _load(kg, kc, it)
    kc.linear_solver.factorize(); kg.linear_solver.factorize()
    assert kg.linear_solver.inertia() == kc.linear_solver.inertia()
    dc, okc, rc = _refined_direction_cpu(kc, it.rhs)
    dg, okg, rg = _refined_direction_gpu(kg, it.rhs)
    assert okc and okg and rg < 1e-8
    assert np.abs(dg - dc).max() / np.abs(dc).max() <= 1e-6
    b = np.random.default_rng(11).standard_normal(kg.n)
    xg = kg.linear_solver.solve_linear_system(_dev(b)).cpu().numpy()
    Kfull = o.tril_to_full(kc.aug_colptr, kc.aug_rowval, kc.aug_nz, kc.n)
    assert np.abs(Kfull @ xg - b).max() / (abs(Kfull).max() * np.abs(xg).max() + np.abs(b).max()) < 1e-12


def test_negative_curvature_is_counted():
    """A10: an indefinite condensed matrix must report the same (pos, zero, neg) as the oracle and fail is_inertia_correct."""
    _need_gpu()
    from madnlp_jl_b200 import kkt as K
    model, st = W.acopf_case("case300_synth")
    cb = _cb(st)
    # large multipliers + loose slack boxes -> the indefinite Lagrangian Hessian dominates J'DJ (oracle: 237 negatives)
    it = W.ipm_iterates(model, st, 1, seed=9, y_scale=1e3, eq_box=(1e-1, 1.0))[0]
    kc = o.SparseCondensedKKTSystem(cb, o.DenseLDLInertiaSolver)
    kg = K.SparseCondensedKKTSystem(cb)
    _load(kg, kc, it)
    kc.linear_solver.factorize(); kg.linear_solver.factorize()
    ref = kc.linear_solver.inertia()
    assert ref[2] > 0
    assert kg.linear_solver.inertia() == ref
    assert not kg.is_inertia_correct(*ref)


def test_augmented_kkt_solve_and_inertia():
    """SparseKKTSystem (true indefinite LDL^T, inertia (n_tot, 0, m)) on a small AC-OPF with equalities kept."""
    _need_gpu()
    from madnlp_jl_b200 import kkt as K
    model, st = W.acopf_case("case300_synth", relax_equality=False)
    cb = _cb(st)
    it = W.ipm_iterates(model, st, 1, seed=4)[0]
    it.du_diag[:] = -1e-8
    kc = o.SparseKKTSystem(cb, o.DenseLDLInertiaSolver)
    kg = K.SparseKKTSystem(cb)
    _load(kg, kc, it)
    kc.linear_solver.factorize(); kg.linear_solver.factorize()
    assert kg.linear_solver.inertia() == kc.linear_solver.inertia() == (kg.n_tot, 0, kg.m)
    dc, okc, rc = _refined_direction_cpu(kc, it.rhs)
    dg, okg, rg = _refined_direction_gpu(kg, it.rhs)
    assert okc and okg
    assert np.abs(dg - dc).max() / np.abs(dc).max() <= 1e-6


def test_big_front_path_3d_grid():
    """Fronts beyond the shared-memory classes (HBM-resident, blocked DMMA update): 3-D augmented KKT, config 5 style.
    delta = 1e-2 keeps the quasi-definite LDL^T well conditioned (growth ~ 1/delta with static pivoting), so the
    solution itself can be compared; the delta = 1e-8 variant is checked through residual + inertia only."""
    _need_gpu()
    import scipy.sparse.linalg as spla
    from madnlp_jl_b200.linear_solvers import B200SparseSolver, DeviceCSC
    for nx, delta, res_tol, sol_tol in ((14, 1e-2, 1e-13, 1e-9), (14, 1e-8, 1e-9, None), (22, 1e-2, 1e-13, 1e-9)):
        N, n_tot, m, I, J, V = W.augmented_grid_kkt(nx, nx, nx, delta=delta)
        cp, rv, mp = o.coo_to_csc(I, J, N, N)
        nz = np.zeros(len(rv)); o.transfer(nz, V, mp)
        csc = DeviceCSC(N, N, cp, rv, _dev(nz))
        M = B200SparseSolver(csc, B200SparseSolver.default_options(kkt_n_primal=n_tot))
        st = M.stats()
        assert st["n_big_fronts"] > 0 and st["max_front"] > 168
        M.factorize()
        assert M.inertia() == (n_tot, 0, m)
        b = np.random.default_rng(0).standard_normal(N)
        x = M.solve_linear_system(_dev(b)).cpu().numpy()
        Kf = o.tril_to_full(cp, rv, nz, N)
        assert np.abs(Kf @ x - b).max() / (abs(Kf).max() * np.abs(x).max() + np.abs(b).max()) < res_tol
        if sol_tol is not None:
            xr = spla.splu(Kf.tocsc()).solve(b)
            assert np.abs(x - xr).max() / np.abs(xr).max() < sol_tol
            # a smaller shared-memory limit forces more fronts through the big path; same answer
            M2 = B200SparseSolver(csc, B200SparseSolver.default_options(kkt_n_primal=n_tot, small_front_max=40, use_cuda_graph=0))
            M2.factorize()
            assert M2.inertia() == (n_tot, 0, m)
            x2 = M2.solve_linear_system(_dev(b)).cpu().numpy()
            assert np.abs(x2 - x).max() / np.abs(x).max() < 1e-10


@pytest.mark.parametrize("n_eq", [0, 24])
def test_dense_condensed_qp(n_eq):
    """configs[1] structure at a size the oracle finishes in seconds: DenseCondensedKKTSystem assembly (A8),
    dense LDL^T + inertia (neg == n_eq) and solve_kkt vs LAPACK dsytrf/dsytrs."""
    _need_gpu()
    from madnlp_jl_b200 import kkt as K
    qp = W.dense_qp(n=320, m=130, n_eq=n_eq, seed=3)
    it = W.dense_qp_iterate(qp, mu=1e-3, seed=4)
    ns = qp.m - n_eq
    cb = o.Callback(qp.n, qp.m, [], [], [], [], qp.ind_ineq, qp.ind_lb, qp.ind_ub)
    kc = o.DenseCondensedKKTSystem(cb)
    kg = K.DenseCondensedKKTSystem(cb)
    for k in (kc, kg):
        k.initialize()
    kc.hess[:] = qp.P; kc.jac[:] = qp.A
    kg.set_dense(hess_np=qp.P, jac_np=qp.A)
    for name in ("reg", "du_diag", "l_diag", "u_diag", "l_lower", "u_lower"):
        getattr(kc, name)[:] = it[name]
        getattr(kg, name).copy_(_dev(it[name]))
    o.set_aug_diagonal_(kc); kc.build_kkt()
    kg.set_aug_diagonal_(); kg.build_kkt()
    N = qp.n + n_eq
    aug = kg.aug_com.cpu().numpy().T                     # back to the mathematical (row, col) view
    assert np.abs(np.tril(aug) - np.tril(kc.aug_com)).max() / np.abs(kc.aug_com).max() < 1e-13
    kc.linear_solver.factorize(); kg.linear_solver.factorize()
    assert kg.linear_solver.inertia() == kc.linear_solver.inertia() == (qp.n, 0, n_eq)
    assert kg.is_inertia_correct(*kg.linear_solver.inertia())
    dc, okc, rc = _refined_direction_cpu(kc, it["rhs"])
    dg, okg, rg = _refined_direction_gpu(kg, it["rhs"])
    assert okc and okg
    assert np.abs(dg - dc).max() / np.abs(dc).max() <= 1e-8
    assert ns == kg.ns and N == kg.N


def test_ipm_replay_regularises_like_the_reference():
    """inertia_correction!(InertiaBased) replay (src/IPM/solver.jl:611-670): a nonconvex iterate must trigger the
    primal regularisation schedule 1e-4, x100, x8 ... until the inertia is correct, then return a direction."""
    _need_gpu()
    from madnlp_jl_b200 import kkt as K
    from madnlp_jl_b200.ipm import IPMLinearAlgebra
    model, st = W.acopf_case("case30_synth")
    cb = _cb(st)
    kg = K.SparseCondensedKKTSystem(cb)
    kg.initialize()
    la = IPMLinearAlgebra(kg)
    good = W.ipm_iterates(model, st, 1, seed=2)[0]
    bad = W.ipm_iterates(model, st, 1, seed=2, y_scale=1e2, eq_box=(1e-1, 1.0))[0]
    for it, expect_reg in ((good, False), (bad, True)):
        d = {k: _dev(getattr(it, k)) for k in ("jac", "hess", "reg", "du_diag", "l_diag", "u_diag", "l_lower", "u_lower", "rhs")}
        before = la.cnt["regularized"]
        la.load_iterate(d)
        assert la.step(mu=it.mu)
        assert (la.cnt["regularized"] > before) == expect_reg
        assert kg.is_inertia_correct(*la.last_inertia)


def test_host_pipeline_returns_the_same_directions_as_serial_steps():
    """ipm.HostIteratePipeline (double-buffered H2D of iterate i+1 / D2H of direction i-1 on copy streams, the asynchronous
    form of SparseWrapperModel's pinned staging, lib/MadNLPGPU/src/wrappers.jl:173-196): the directions that arrive in the pinned
    host buffers must be BIT-identical to the ones of copy -> step -> copy, for every iterate and across slot reuse."""
    _need_gpu()
    from madnlp_jl_b200 import kkt as K
    from madnlp_jl_b200.ipm import IPMLinearAlgebra, HostIteratePipeline
    fields = ("jac", "hess", "reg", "du_diag", "l_diag", "u_diag", "l_lower", "u_lower", "rhs")
    model, st = W.acopf_case("case300_synth")
    its = W.ipm_iterates(model, st, 5, seed=4)
    host = [{k: torch.from_numpy(np.ascontiguousarray(getattr(it, k))).pin_memory() for k in fields} for it in its]
    kg = K.SparseCondensedKKTSystem(_cb(st))
    kg.initialize()
    la = IPMLinearAlgebra(kg)
    serial = []
    for rep in range(2):                                  # second pass: captured graphs replay
        for i, it in enumerate(its):
            la.load_iterate_host(host, i)
            assert la.step(mu=it.mu)
            if rep:
                serial.append(la.d.values.cpu().numpy().copy())
    pipe = HostIteratePipeline(la, fields)
    assert pipe.h2d_bytes == sum(v.numel() * 8 for v in host[0].values()) and pipe.d2h_bytes == la.d.values.numel() * 8
    got = []
    slot = pipe.prefetch(host[0])
    for i, it in enumerate(its):
        pipe.load(slot)
        nxt = None
        if i + 1 < len(its):
            if i % 2:                                     # both placements of the prefetch: before the step / inside it
                nxt = pipe.prefetch(host[i + 1])
                assert la.step(mu=it.mu)
            else:
                box = []
                assert la.step(mu=it.mu, after_prologue=lambda: box.append(pipe.prefetch(host[i + 1])))
                nxt = box[0]
        else:
            assert la.step(mu=it.mu)
        hs = pipe.push_result()
        pipe.ev_d_out[hs].synchronize()
        got.append(pipe.d_host[hs].numpy().copy())
        slot = nxt
    pipe.drain()
    torch.cuda.synchronize()
    for a, b in zip(got, serial):
        assert np.array_equal(a, b)


def test_bench_dump_outputs_agree_with_the_reference_arm(tmp_path):
    """bench.py --dump-outputs, both arms with the same arguments: the last timed step of the device-resident loop has the reference
    arm's inertia and its step direction within 1e-6 (refined, as above); the pipelined host-facing loop returns it bit for bit."""
    _need_gpu()
    import os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    args = ["--steps", "3", "--warmup", "1", "--workload", "case300_synth", "--no-secondary", "--cpu-sample-steps", "0"]
    got = {}
    for impl in ("b200", "reference"):
        out = subprocess.run([sys.executable, "bench.py", "--impl", impl, *args, "--dump-outputs", str(tmp_path / impl)],
                             cwd=root, capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stderr[-2000:]
        got[impl] = {f[:-len(".npy")]: np.load(tmp_path / impl / f) for f in os.listdir(tmp_path / impl)}
    g, r = got["b200"], got["reference"]
    assert sorted(g) == ["direction", "direction_e2e", "inertia"] and sorted(r) == ["direction", "inertia"]
    assert all(a.dtype == np.float64 for a in (*g.values(), *r.values()))
    assert np.array_equal(g["inertia"], r["inertia"])
    assert np.abs(g["direction"] - r["direction"]).max() / np.abs(r["direction"]).max() <= 1e-6
    assert np.array_equal(g["direction_e2e"], g["direction"])


def test_golden_fixture_on_device():
    """The committed HS15 fixture (tests/golden/hs15_kkt.json): factor + solve the stored condensed and augmented
    matrices through the C ABI and reproduce the stored solve_kkt vector / inertia."""
    _need_gpu()
    import json, os
    from madnlp_jl_b200.linear_solvers import B200SparseSolver, DeviceCSC
    g = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "hs15_kkt.json")))
    for key, n, npr in (("hs15_sparse", 6, 4), ("hs15_condensed", 2, 0)):
        e = g[key]
        csc = DeviceCSC(n, n, np.array(e["colptr"], dtype=np.int32), np.array(e["rowval"], dtype=np.int32), _dev(np.array(e["nzval"])))
        M = B200SparseSolver(csc, B200SparseSolver.default_options(kkt_n_primal=npr))
        M.factorize()
        assert list(M.inertia()) == e["inertia"]
    k = g["kat_2x2"]
    cp, rv, mp = o.coo_to_csc(np.array(k["row"]), np.array(k["col"]), 2, 2)
    nz = np.zeros(len(rv)); o.transfer(nz, np.array(k["val"]), mp)
    M = B200SparseSolver(DeviceCSC(2, 2, cp, rv, _dev(nz)))
    M.factorize()
    x = M.solve_linear_system(_dev(np.array(k["b"]))).cpu().numpy()
    assert np.abs(x - np.array(k["x"])).max() < 1e-14 and list(M.inertia()) == k["inertia"]


@pytest.mark.parametrize("rows,cols", [(1, 1), (130, 320), (515, 77), (2048, 4096)])
def test_dense_matvec_kernels(rows, cols):
    """b2d_gemv_n / b2d_gemv_t / b2d_symv_lower (the mat-vecs of AbstractDenseKKTSystem mul!/solve_kkt!) vs numpy fp64;
    tolerance: 1e-13 relative to |A||x| (different summation order only)."""
    _need_gpu()
    from madnlp_jl_b200.capi import lib, check
    rng = np.random.default_rng(rows * 7 + cols)
    A = rng.standard_normal((rows, cols))
    x = rng.standard_normal(cols); xt = rng.standard_normal(rows)
    y0 = rng.standard_normal(rows); yt0 = rng.standard_normal(cols)
    Ad = _dev(A.T.copy())                                  # column-major storage, lda = rows
    st = torch.cuda.current_stream().cuda_stream
    xd, xtd = _dev(x), _dev(xt)                            # (named: a temporary would be freed before the launch)
    for alpha, beta in ((1.0, 0.0), (-0.5, 2.0)):
        y = _dev(y0.copy()); yt = _dev(yt0.copy())
        if beta == 0.0:
            y.fill_(float("nan")); yt.fill_(float("nan"))  # beta == 0 must not read y (BLAS convention)
        check(lib.b2d_gemv_n(rows, cols, rows, Ad.data_ptr(), xd.data_ptr(), y.data_ptr(), alpha, beta, st))
        check(lib.b2d_gemv_t(rows, cols, rows, Ad.data_ptr(), xtd.data_ptr(), yt.data_ptr(), alpha, beta, st))
        ref = alpha * (A @ x) + (beta * y0 if beta else 0.0)
        reft = alpha * (A.T @ xt) + (beta * yt0 if beta else 0.0)
        scale = np.abs(A) @ np.abs(x) + np.abs(y0) + 1.0
        scalet = np.abs(A.T) @ np.abs(xt) + np.abs(yt0) + 1.0
        assert (np.abs(y.cpu().numpy() - ref) / scale).max() < 1e-13
        assert (np.abs(yt.cpu().numpy() - reft) / scalet).max() < 1e-13
    n = min(rows, cols)
    S = rng.standard_normal((n, n)); S = S + S.T
    low = np.tril(S) + np.triu(np.full((n, n), np.nan), 1)  # the upper triangle must never be read
    xs = rng.standard_normal(n); ys0 = rng.standard_normal(n)
    ys = _dev(ys0.copy()); lowd = _dev(low.T.copy()); xsd = _dev(xs)
    check(lib.b2d_symv_lower(n, n, lowd.data_ptr(), xsd.data_ptr(), ys.data_ptr(), 0.75, -1.0, st))
    ref = 0.75 * (S @ xs) - ys0
    assert (np.abs(ys.cpu().numpy() - ref) / (np.abs(S) @ np.abs(xs) + np.abs(ys0) + 1.0)).max() < 1e-13


def test_fused_richardson_kernels_are_bit_identical():
    """b2_richardson_begin/update == (norm_inf; fill; copy / axpy; copy; norm_inf) and b2_condensed_kkt_mul_norm == (mul; norm_inf), bit for bit;
    b2_copy_many == the individual copies (ragged lengths, an empty segment)."""
    _need_gpu()
    import ctypes as C
    from madnlp_jl_b200 import kkt as K
    from madnlp_jl_b200.capi import lib, check
    st = torch.cuda.current_stream().cuda_stream
    rng = np.random.default_rng(11)
    n = 100003
    b, w, x = (_dev(rng.standard_normal(n)) for _ in range(3))
    w2, x2 = w.clone(), x.clone()
    norms = torch.full((2,), 7.0, dtype=torch.float64, device="cuda")
    check(lib.b2_richardson_update(n, b.data_ptr(), w.data_ptr(), x.data_ptr(), norms.data_ptr(), st))
    check(lib.b2_axpy(n, 1.0, w2.data_ptr(), x2.data_ptr(), st)); check(lib.b2_copy(n, b.data_ptr(), w2.data_ptr(), st))
    assert torch.equal(x, x2) and torch.equal(w, w2)
    assert float(norms[0]) == 0.0 and float(norms[1]) == float(x2.abs().max())
    nb = torch.full((1,), 3.0, dtype=torch.float64, device="cuda")
    check(lib.b2_richardson_begin(n, b.data_ptr(), w.data_ptr(), x.data_ptr(), nb.data_ptr(), st))     # ||b||; x = 0; w = b
    assert torch.equal(w, b) and float(x.abs().max()) == 0.0 and float(nb[0]) == float(b.abs().max())
    # mul with fused norm on a condensed KKT system
    model, stt = W.acopf_case("case30_synth")
    it = W.ipm_iterates(model, stt, 1, seed=5)[0]
    kc = o.SparseCondensedKKTSystem(_cb(stt)); kg = K.SparseCondensedKKTSystem(_cb(stt))
    _load(kg, kc, it)
    xv = K.UnreducedKKTVector.for_kkt(kg); wa = K.UnreducedKKTVector.for_kkt(kg); wb = K.UnreducedKKTVector.for_kkt(kg)
    xv.values.copy_(_dev(rng.standard_normal(xv.values.numel())))
    r0 = _dev(rng.standard_normal(xv.values.numel())); wa.values.copy_(r0); wb.values.copy_(r0)
    acc = torch.zeros(1, dtype=torch.float64, device="cuda")
    kg.mul(wa, xv, -1.0, 1.0)
    kg.mul_norm(wb, xv, -1.0, 1.0, acc)
    assert torch.equal(wa.values, wb.values) and float(acc[0]) == float(wa.values.abs().max())
    # copy_many
    lens = [0, 1, 255, 70001]
    src = [_dev(rng.standard_normal(max(k, 1)))[:k] for k in lens]
    dst = [torch.zeros(max(k, 1), dtype=torch.float64, device="cuda")[:k] for k in lens]
    cnt = len(lens)
    check(lib.b2_copy_many(cnt, (C.c_void_p * cnt)(*[s.data_ptr() for s in src]), (C.c_void_p * cnt)(*[d.data_ptr() for d in dst]),
                           (C.c_int64 * cnt)(*lens), st))
    assert all(torch.equal(s, d) for s, d in zip(src, dst))


@pytest.mark.parametrize("n_tot,m,seed", [(0, 0, 0), (7, 3, 1), (1000, 400, 2), (300001, 120007, 3)])
def test_ipm_reductions_match_the_reference_formulas(n_tot, m, seed):
    """SURVEY 8f rows 2/4: the line-search scalars (src/IPM/kernels.jl:263-388,675-695) and set_aug_rhs! (:113-130) as
    single-pass device kernels vs their scalar restatement.  min/max results: exact (same terms, order-free);
    sums: relative 1e-12 of the sum of magnitudes (different association); twice the same call: bit-identical."""
    _need_gpu()
    import ctypes as C
    from madnlp_jl_b200.capi import lib, check
    rng = np.random.default_rng(seed)
    st = torch.cuda.current_stream().cuda_stream
    has_lb = rng.random(n_tot) < 0.6; has_ub = rng.random(n_tot) < 0.5
    ind_lb = np.flatnonzero(has_lb).astype(np.int64); ind_ub = np.flatnonzero(has_ub).astype(np.int64)
    nlb, nub = len(ind_lb), len(ind_ub)
    x = rng.standard_normal(n_tot)
    xl = np.where(has_lb, x - rng.uniform(1e-6, 2.0, n_tot), -np.inf)
    xu = np.where(has_ub, x + rng.uniform(1e-6, 2.0, n_tot), np.inf)
    zl = np.where(has_lb, rng.uniform(1e-8, 3.0, n_tot), 0.0); zu = np.where(has_ub, rng.uniform(1e-8, 3.0, n_tot), 0.0)
    f, jacl, dx = (rng.standard_normal(n_tot) for _ in range(3))
    dzl, dzu = rng.standard_normal(nlb), rng.standard_normal(nub)
    c, l = rng.standard_normal(m), rng.standard_normal(m)
    mu, tau, sd, sc, s_max, obj = 1e-3, 0.99, 1.7, 2.3, 100.0, 4.25
    h = C.c_void_p()
    check(lib.b2_bounds_create(n_tot, nlb, nub, ind_lb.ctypes.data, ind_ub.ctypes.data, C.byref(h)))
    D = {k: _dev(v) for k, v in dict(x=x, xl=xl, xu=xu, zl=zl, zu=zu, f=f, jacl=jacl, dx=dx, dzl=dzl, dzu=dzu, c=c, l=l).items()}
    P = lambda k: D[k].data_ptr()
    out = torch.zeros(16, dtype=torch.float64, device="cuda")
    O = lambda k: out[k:k + 1].data_ptr()

    def run():
        check(lib.b2_get_alpha_max(h, P("x"), P("xl"), P("xu"), P("dx"), tau, O(0), st))
        check(lib.b2_get_alpha_z(h, P("zl"), P("zu"), P("dzl"), P("dzu"), tau, O(1), st))
        check(lib.b2_get_varphi(h, obj, P("x"), P("xl"), P("xu"), mu, O(2), st))
        check(lib.b2_get_varphi_d(h, P("f"), P("x"), P("xl"), P("xu"), P("dx"), mu, O(3), st))
        check(lib.b2_get_inf_du(h, P("f"), P("zl"), P("zu"), P("jacl"), sd, O(4), st))
        check(lib.b2_get_inf_compl(h, P("x"), P("xl"), P("xu"), P("zl"), P("zu"), mu, sc, O(5), st))
        check(lib.b2_get_average_complementarity(h, P("x"), P("xl"), P("xu"), P("zl"), P("zu"), O(6), st))
        check(lib.b2_get_min_complementarity(h, P("x"), P("xl"), P("xu"), P("zl"), P("zu"), O(7), st))
        check(lib.b2_get_rel_search_norm(h, n_tot, P("x"), P("dx"), O(8), st))
        check(lib.b2_get_sd(h, m, P("l"), P("zl"), P("zu"), s_max, O(9), st))
        check(lib.b2_get_sc(h, P("zl"), P("zu"), s_max, O(10), st))
        return out.cpu().numpy().copy()

    g = run()
    assert (run() == g).all()                                               # deterministic reduction tree
    xlr, xur = x[ind_lb], x[ind_ub]
    ref = [o.get_alpha_max(x, xl, xu, dx, tau), o.get_alpha_z(zl[ind_lb], zu[ind_ub], dzl, dzu, tau),
           o.get_varphi(obj, xlr, xl[ind_lb], xu[ind_ub], xur, mu), o.get_varphi_d(f, x, xl, xu, dx, mu),
           o.get_inf_du(f, zl, zu, jacl, sd), o.get_inf_compl(xlr, xl[ind_lb], zl[ind_lb], xu[ind_ub], xur, zu[ind_ub], mu, sc),
           o.get_average_complementarity(xlr, xl[ind_lb], zl[ind_lb], xur, xu[ind_ub], zu[ind_ub]),
           o.get_min_complementarity(xlr, xl[ind_lb], zl[ind_lb], xur, xu[ind_ub], zu[ind_ub]),
           o.get_rel_search_norm(x, dx), o.get_sd(l, zl[ind_lb], zu[ind_ub], s_max), o.get_sc(zl[ind_lb], zu[ind_ub], s_max)]
    for k in (0, 1, 4, 5, 7, 8):                                            # min / max: exact
        assert g[k] == ref[k], (k, g[k], ref[k])
    mags = {2: abs(obj) + np.abs(mu * np.log(np.concatenate([xlr - xl[ind_lb], xu[ind_ub] - xur]))).sum() if nlb + nub else abs(obj),
            3: np.abs((f - mu / (x - xl) + mu / (xu - x)) * dx).sum(), 6: 3.0 * 2.0, 9: 1.0 + g[9], 10: 1.0 + g[10]}
    for k in (2, 3, 6, 9, 10):                                              # sums: association differs
        assert abs(g[k] - ref[k]) <= 1e-12 * (mags[k] + 1.0), (k, g[k], ref[k])
    # set_aug_rhs!: elementwise, bit-exact
    p = torch.zeros(n_tot + m + nlb + nub, dtype=torch.float64, device="cuda")
    check(lib.b2_set_aug_rhs(h, m, P("x"), P("xl"), P("xu"), P("f"), P("zl"), P("zu"), P("jacl"), P("c"), mu, p.data_ptr(), st))
    assert (p.cpu().numpy() == o.set_aug_rhs(x, xl, xu, f, zl, zu, jacl, c, mu, ind_lb, ind_ub)).all()
    # a NaN anywhere propagates through min like Julia's
    if n_tot > 3:
        D["dx"][3] = float("nan")
        check(lib.b2_get_alpha_max(h, P("x"), P("xl"), P("xu"), P("dx"), tau, O(0), st))
        assert np.isnan(float(out[0])) == np.isnan(o.get_alpha_max(x, xl, xu, np.where(np.arange(n_tot) == 3, np.nan, dx), tau))
    lib.b2_bounds_destroy(h)


@pytest.mark.parametrize("n,m,n_eq", [(640, 300, 0), (515, 333, 40), (1024, 512, 0)])
def test_dense_assembly_on_tensor_cores_matches_oracle(n, m, n_eq, monkeypatch):
    """A8 with the contraction on tcgen05.mma.kind::i8 (Ozaki digits, csrc/ozaki_kernels.cuh): ragged sizes (n, ns not multiples of the
    128 / 64 tile and K-block sizes: zero padding), equality rows, D spanning 18 decades.  Bar: 1e-13 of max|K| against the oracle's
    fp64 assembly (Dense/condensed.jl:157-186), and agreement with the DMMA kernel to the same bar."""
    _need_gpu()
    from madnlp_jl_b200 import kkt as K
    qp = W.dense_qp(n=n, m=m, n_eq=n_eq, seed=7)
    it = W.dense_qp_iterate(qp, mu=1e-5, seed=8)
    cb = o.Callback(qp.n, qp.m, [], [], [], [], qp.ind_ineq, qp.ind_lb, qp.ind_ub)
    kc = o.DenseCondensedKKTSystem(cb); kc.initialize(); kc.hess[:] = qp.P; kc.jac[:] = qp.A
    out = {}
    for flag in ("1", "0"):
        monkeypatch.setenv("B2_OZAKI", flag)
        kg = K.DenseCondensedKKTSystem(cb); kg.initialize(); kg.set_dense(hess_np=qp.P, jac_np=qp.A)
        for name in ("reg", "du_diag", "l_diag", "u_diag", "l_lower", "u_lower"):
            getattr(kc, name)[:] = it[name]
            getattr(kg, name).copy_(_dev(it[name]))
        kg.set_aug_diagonal_(); kg.build_kkt()
        out[flag] = np.tril(kg.aug_com.cpu().numpy().T)
        assert kg.tensor_core_status() is (True if flag == "1" else None)
    o.set_aug_diagonal_(kc); kc.build_kkt()
    ref = np.tril(kc.aug_com); scale = np.abs(kc.aug_com).max()
    assert np.abs(out["1"] - ref).max() / scale <= 1e-13
    assert np.abs(out["0"] - ref).max() / scale <= 1e-13
