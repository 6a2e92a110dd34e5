#!/usr/bin/env python
"""b2d_factorize / b2d_solve with static and Bunch-Kaufman pivoting (b2_options.pivoting), CUDA events, median of 20 after 3
warm-ups with L2 flushed between repeats, at N in {1024, 4096} on two matrices:
  c2   the DenseCondensedKKTSystem matrix of workloads.dense_qp (n = N - 256, m = n / 2, n_eq = 256) at an IPM-like iterate
  aug  an indefinite augmented matrix [[H, J'], [J, 0]] (H a random bilinear form with zero diagonal, n = 3N/4, m = N/4)
Prints the inertia and the number of 2 x 2 / perturbed pivots beside each time.  --trace: per-kind device time of one
pivoted factorisation at N = 4096 (B2_DENSE_TRACE stamps; a separate run, tracing perturbs the timings)."""
import argparse, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[1024, 4096])
    ap.add_argument("--trace", action="store_true")
    args = ap.parse_args()
    if args.trace:
        os.environ["B2_DENSE_TRACE"] = "1"
    import numpy as np, torch
    import ctypes as C
    import madnlp_jl_b200 as pkg
    from madnlp_jl_b200 import kkt as K
    from madnlp_jl_b200.linear_solvers import B200DenseSolver
    W = pkg.workloads
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device="cuda")

    def timeit(fn, reps=20, warm=3):
        for _ in range(warm):
            fn()
        ts = []
        for _ in range(reps):
            flush.fill_(1.0)
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record(); e1.synchronize()
            ts.append(e0.elapsed_time(e1))
        return float(np.median(ts))

    class _CB:
        def __init__(self, qp):
            self.nvar, self.ncon = qp.n, qp.m
            self.jac_I = self.jac_J = self.hess_I = self.hess_J = []
            self.ind_ineq, self.ind_lb, self.ind_ub = qp.ind_ineq, qp.ind_lb, qp.ind_ub

    def c2_matrix(N):
        n = N - 256
        qp = W.dense_qp(n=n, m=n // 2, n_eq=256, seed=1)
        it = W.dense_qp_iterate(qp, mu=1e-3, seed=2)
        kg = K.DenseCondensedKKTSystem(_CB(qp)); kg.initialize(); kg.set_dense(hess_np=qp.P, jac_np=qp.A)
        for name in ("reg", "du_diag", "l_diag", "u_diag", "l_lower", "u_lower"):
            getattr(kg, name).copy_(torch.from_numpy(it[name]).cuda())
        kg.set_aug_diagonal_(); kg.build_kkt()
        torch.cuda.synchronize()
        return kg.aug_com.clone()                      # memory = column-major N x N, lower triangle

    def aug_matrix(N):
        rng = np.random.default_rng(N)
        n, m = 3 * N // 4, N // 4
        H = np.tril(rng.standard_normal((n, n)), -1); H = H + H.T
        Km = np.zeros((N, N)); Km[:n, :n] = H; Km[n:, :n] = rng.standard_normal((m, n)); Km[:n, n:] = Km[n:, :n].T
        return torch.from_numpy(np.ascontiguousarray(Km.T)).cuda()

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print(f"# {torch.cuda.get_device_name(0)} | nvidia-smi: {smi}")
    print("# b2d_factorize / b2d_solve, CUDA events, median of 20 (3 warm-ups, L2 flushed between repeats), use_cuda_graph=1")
    print(f"{'matrix':<6} {'N':>5} {'pivoting':<13} {'factorize_ms':>12} {'solve_ms':>9} {'inertia':>18} {'n_2x2':>6} "
          f"{'n_perturbed':>11} {'rel_residual':>12}")
    for N in args.sizes:
        for mname, build in (("c2", c2_matrix), ("aug", aug_matrix)):
            A = build(N)
            Af = torch.tril(A.t()) + torch.tril(A.t(), -1).t()
            b = torch.randn(N, dtype=torch.float64, device="cuda")
            for piv in ("static", "bunchkaufman"):
                M = B200DenseSolver(A, B200DenseSolver.default_options(pivoting=piv))
                t_fac = timeit(M.factorize)
                inertia = M.inertia()
                _, _, n2, npert = M.pivot_info()
                xc = b.clone()
                t_sol = timeit(lambda: M.solve_linear_system(xc))
                x = M.solve_linear_system(b.clone())
                res = float((Af @ x - b).abs().max() / (Af.abs().sum(1).max() * x.abs().max() + b.abs().max()))
                print(f"{mname:<6} {N:>5} {piv:<13} {t_fac:>12.3f} {t_sol:>9.3f} {str(inertia):>18} {n2:>6} {npert:>11} {res:>12.2e}",
                      flush=True)
                if args.trace and piv == "bunchkaufman" and N == max(args.sizes):
                    M.factorize(); torch.cuda.synchronize()
                    cnt = C.c_int64()
                    pkg.capi.check(pkg.capi.lib.b2d_debug_trace(M._h, None, 0, C.byref(cnt)))
                    st = np.zeros(cnt.value, dtype=np.uint64)
                    pkg.capi.check(pkg.capi.lib.b2d_debug_trace(M._h, st.ctypes.data, cnt.value, C.byref(cnt)))
                    st = st.reshape(-1, 8, 2).astype(np.float64)
                    ok = st[:, :, 1] > 0
                    t0 = st[:, :, 0][ok].min()
                    names = ["diag", "near_trsm", "near_syrk", "panel_trsm", "col_update", "trailing", "inverse", "bk_diag"]
                    span = (st[:, :, 1] - st[:, :, 0]) * ok
                    print(f"#   trace {mname} N={N}: wall {(st[:, :, 1][ok].max() - t0) / 1e3:.1f} us; per kind (sum of launch spans, us): " +
                          ", ".join(f"{names[k]} {span[:, k].sum() / 1e3:.1f}" for k in range(8) if ok[:, k].any()), flush=True)
                del M


if __name__ == "__main__":
    main()
