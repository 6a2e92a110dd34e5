/*
 * b200kkt.h -- C ABI of the B200-native KKT hot path (assembly -> LDL^T + inertia -> solve).
 *
 * This is the drop-in boundary a MadNLP.jl maintainer binds with `ccall` (see INTEGRATION.md
 * and madnlp.jl_b200/julia/B200KKT.jl).  Plain pointers and sizes only; no exceptions cross
 * the boundary: every entry point returns a status code (B2_OK == 0) and b2_last_error()
 * gives the message.  All matrix values are fp64; all sparse indices are 0-based int32
 * (the reference uses 1-based Int32: src/KKT/Sparse/augmented.jl:20, condensed.jl:11,17);
 * COO->CSC maps are int64 like the reference's Vector{Int} (src/matrixtools.jl:91).
 *
 * Pointer suffix convention:  *_h = host memory,  *_d = device memory (cuda:current).
 * `stream` arguments are a cudaStream_t passed as void* (NULL = legacy default stream).
 *
 * Reference interface each group replaces (paths relative to MadNLP.jl @ v0.10.1):
 *   b2_*  sparse solver  : AbstractLinearSolver surface, src/LinearSolvers/linearsolvers.jl:13-95,
 *                          as implemented by CUDSSSolver lib/MadNLPGPU/ext/MadNLPGPUCUDAExt/cudss.jl:88-214
 *                          and Ma97Solver lib/MadNLPHSL/src/ma97.jl:29-115.
 *   b2d_* dense solver   : LapackCUDASolver/LapackCPUSolver, src/LinearSolvers/lapack.jl:164-172,
 *                          lib/MadNLPGPU/ext/MadNLPGPUCUDAExt/cusolver.jl:150-187.
 *   b2_coo_to_csc, b2_transfer*          : src/matrixtools.jl:55-95, lib/MadNLPGPU/src/KKT/gpu_sparse.jl:260-302,
 *                                          kernels_sparse.jl:161-167.
 *   b2_condensed_*                       : src/KKT/Sparse/condensed.jl:201-366, gpu_sparse.jl:308-340.
 *   b2d_condensed_assemble               : src/KKT/Dense/condensed.jl:120-186, kernels_dense.jl:81-119.
 *   b2_set_aug_diagonal .. b2_kkt_mul_*  : src/IPM/kernels.jl:4-27,161-204, src/IPM/factorization.jl:41-46,
 *                                          143-167,190-237,303-324, src/KKT/KKTsystem.jl:222-226.
 */
#ifndef B200KKT_H
#define B200KKT_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2_OK                 0
#define B2_ERR_INVALID        1   /* bad argument */
#define B2_ERR_CUDA           2   /* CUDA runtime error (message in b2_last_error) */
#define B2_ERR_SYMBOLIC       3   /* analysis failed         (SymbolicException,      linearsolvers.jl:133) */
#define B2_ERR_FACTORIZATION  4   /* numeric failure         (FactorizationException, linearsolvers.jl:134) */
#define B2_ERR_SOLVE          5   /* solve before factorize  (SolveException,         linearsolvers.jl:135) */
#define B2_ERR_NO_DEVICE      6   /* no CUDA device: the product path has no CPU fallback */

#define B2_ORDER_METIS_ND 0   /* nested dissection (METIS_NodeND, statically linked)        */
#define B2_ORDER_MINDEG   1   /* built-in minimum-degree                                    */
#define B2_ORDER_NATURAL  2   /* identity                                                   */
#define B2_ORDER_USER     3   /* caller-supplied permutation (cf. cudss_perm, cudss.jl:7)   */

const char* b2_last_error(void);
int b2_version(void);
/* number of visible CUDA devices; B2_ERR_NO_DEVICE if none */
int b2_device_count(int* count);

/* ------------------------------------------------------------------ options */
typedef struct b2_options {
    int32_t ordering;        /* B2_ORDER_*                                              */
    int32_t nemin;           /* supernode amalgamation: always merge while width <= nemin */
    double  relax_zeros;     /* additionally merge when explicit-zero fraction below this */
    double  pivot_eps;       /* |d| < pivot_eps -> static perturbation, counted as "zero"  */
    int32_t use_cuda_graph;  /* 1: capture factor/solve launch sequences into CUDA graphs  */
    int32_t small_front_max; /* fronts with order <= this run in the fused shared-memory kernel */
    int32_t n_parts;         /* multi-GPU: number of ranks sharing the elimination tree (1 = off) */
    int32_t part_rank;       /* multi-GPU: this rank                                        */
    int32_t kkt_n_primal;    /* > 0: the matrix is an augmented KKT system [[H, J'],[J, -D]] whose first kkt_n_primal
                                rows are primal; the ordering then eliminates every dual row only after one of its
                                primal neighbours, so that a zero (2,2) block never yields a structurally zero pivot */
    int32_t fuse_max_fronts; /* bottom elimination subtrees with at most this many (warp-class) fronts run inside ONE
                                CTA of a single launch (0 = plain level-by-level schedule)                      */
    int32_t dep_schedule;    /* bit 0 (factorisation), bit 1 (solves): when every front is team-class (order <= 64) run the sweep
                                as ONE launch whose CTAs wait on their children's completion flags instead of on
                                kernel boundaries.  Default 1: measured faster for the factorisation only.
                                bit 2 (hybrid sweeps): the fused bottom subtrees keep their staged kernel, every front above
                                them runs in one flag-driven launch (instead of one launch per level)          */
    int32_t chain_merge_f;   /* > 0: a supernode with exactly ONE child absorbs it whatever the explicit zeros cost, as long as the
                                merged front stays team-class (order <= min(chain_merge_f, 64)): on latency-bound trees every
                                level of the critical path costs ~5 us of hand-off besides its pivots, the zeros nothing.
                                Default 0 = off (measured slower on the OPF trees: the single-child chains sit at the bottom, where the
                                tree is throughput-bound and bigger leaves hurt); kept as an option for trees with long chains on top */
    int32_t pivoting;        /* B2_PIVOT_*: pivoting of the dense solver (b2d_*).  The sparse solver (b2_*) supports only
                                B2_PIVOT_STATIC and rejects any other value                                        */
    int32_t reserved[3];
} b2_options;

#define B2_PIVOT_STATIC         0   /* 1 x 1 pivots in order, |d| < pivot_eps perturbed (default)                      */
#define B2_PIVOT_BUNCH_KAUFMAN  1   /* dense solver: Bunch-Kaufman 1 x 1 / 2 x 2 pivots, search bounded to each 128 x 128
                                       diagonal block; needs ceil(N / 128) <= number of SMs                              */
/* pivot kinds reported by b2d_pivot_info */
#define B2_PIVOT_KIND_1X1        0
#define B2_PIVOT_KIND_2X2_FIRST  1
#define B2_PIVOT_KIND_2X2_SECOND 2
#define B2_PIVOT_KIND_PERTURBED  3  /* numerically zero column: pivot set to +-pivot_eps, counted as a zero eigenvalue */

int b2_options_default(b2_options* opt);

/* ------------------------------------------------------------------ sparse LDL^T */
typedef struct b2_solver b2_solver;

typedef struct b2_stats {
    int64_t n, nnz_a, nnz_l, flops;        /* nnz(L) incl. diagonal and explicit zeros; flops of one factorisation */
    int64_t n_supernodes, n_levels;
    int64_t max_front, n_small_fronts, n_big_fronts;
    int64_t factor_bytes, workspace_bytes; /* device memory held */
    int64_t sep_rows;                      /* multi-GPU: order of the shared (replicated) top tree */
    int64_t n_factor_launches, n_solve_launches;
    int64_t n_perturbed;                   /* pivots perturbed in the last factorisation */
} b2_stats;

/* Analysis (ordering + symbolic factorisation); `nzval_d` is KEPT BY REFERENCE and re-read by
 * every b2_factorize -- the reference's aliasing contract (cudss.jl:154-158, ma97.jl:72-88).
 * colptr_h[n+1], rowval_h[nnz]: lower-triangular CSC pattern on the host, 0-based.
 * user_perm_h: n entries (perm[new]=old) when ordering == B2_ORDER_USER, else NULL. */
int b2_create(int32_t n, int64_t nnz, const int32_t* colptr_h, const int32_t* rowval_h,
              const double* nzval_d, const b2_options* opt, const int32_t* user_perm_h,
              b2_solver** out);
/* analysis only (no device state): for tooling/tests on machines without a GPU; every numeric entry point
 * returns B2_ERR_INVALID on such a handle -- it is NOT a compute fallback. */
int b2_create_symbolic_only(int32_t n, int64_t nnz, const int32_t* colptr_h, const int32_t* rowval_h,
                            const b2_options* opt, const int32_t* user_perm_h, b2_solver** out);
int b2_destroy(b2_solver* s);
/* re-point the aliased value buffer (same pattern) */
int b2_set_values_ptr(b2_solver* s, const double* nzval_d);
/* numeric factorisation of the CURRENT values; asynchronous on `stream` */
int b2_factorize(b2_solver* s, void* stream);
/* (num_pos, num_zero, num_neg) in the reference's code order (src/IPM/solver.jl:626);
 * synchronises `stream`.  Perturbed pivots are reported as zeros (cf. mumps.jl:248-250). */
int b2_inertia(b2_solver* s, int64_t* num_pos, int64_t* num_zero, int64_t* num_neg, void* stream);
/* the same read split in two so that a caller can queue more work behind the factorisation before it blocks:
 * b2_inertia_enqueue() queues the 32-byte D2H copy on `stream`; after the caller has synchronised that stream,
 * b2_inertia_fetch() returns the counts without touching the device.  (b2_inertia == enqueue + synchronise + fetch.) */
int b2_inertia_enqueue(b2_solver* s, void* stream);
int b2_inertia_fetch(b2_solver* s, int64_t* num_pos, int64_t* num_zero, int64_t* num_neg);
/* in-place x <- K^{-1} x, nrhs columns of length n (ld = n); asynchronous on `stream` */
int b2_solve(b2_solver* s, double* x_d, int32_t nrhs, void* stream);
/* raise robustness after a failed refinement (improve!, linearsolvers.jl / ma97.jl:103-111);
 * *changed = 1 if something changed and a re-factorisation is worthwhile */
int b2_improve(b2_solver* s, int32_t* changed);
int b2_get_stats(b2_solver* s, b2_stats* st);
/* copy out the fill-reducing permutation (perm[new]=old), n entries, host */
int b2_get_perm(b2_solver* s, int32_t* perm_h);

/* Multi-GPU (subtree-to-rank) support.  With opt.n_parts = P > 1 every rank analyses the same
 * pattern; rank r factors the subtrees it owns plus (replicated) the shared top tree.  The only
 * exchange is the sum of the subtree roots' update (Schur-complement) blocks, which the host
 * reduces with NCCL:   b2_factorize_local -> allreduce(b2_exchange_buffer) -> b2_factorize_top.
 * b2_solve_* mirror this for the triangular solves (the exchange buffer then holds vectors). */
int b2_exchange_buffer(b2_solver* s, double** buf_d, int64_t* n_factor_doubles, int64_t* n_solve_doubles);
int b2_exchange_vector(b2_solver* s, double** buf_d, int64_t* n_doubles);   /* forward-solve contributions */
/* inertia split for the multi-GPU reduction: counts of the owned subtrees and of the replicated top tree */
int b2_inertia_parts(b2_solver* s, int64_t* local_neg, int64_t* local_zero, int64_t* top_neg, int64_t* top_zero, void* stream);
int b2_factorize_local(b2_solver* s, void* stream);
int b2_factorize_top(b2_solver* s, void* stream);
int b2_solve_fwd_local(b2_solver* s, double* x_d, void* stream);
int b2_solve_top(b2_solver* s, double* x_d, void* stream);      /* after allreduce of the exchange buffer */
int b2_solve_bwd_local(b2_solver* s, double* x_d, void* stream); /* leaves x complete only on owned + top rows */
int b2_owned_mask(b2_solver* s, uint8_t* owned_h);               /* n entries: 1 if this rank finalises x[i] */

/* Debug/test export of the symbolic structure (host arrays, caller-allocated; pass NULL to query sizes):
 * used by tests/ to replay the multifrontal arithmetic in numpy on machines without a GPU. */
typedef struct b2_symbolic_sizes {
    int64_t n, n_supernodes, n_rows, n_children, n_rel, n_amap, n_levels, lval_size, cb_size;
} b2_symbolic_sizes;
int b2_symbolic_query(b2_solver* s, b2_symbolic_sizes* sz);
int b2_symbolic_export(b2_solver* s, int32_t* perm, int32_t* sn_first, int32_t* sn_parent, int32_t* sn_level,
                       int64_t* rows_ptr, int32_t* rows, int64_t* lp_off, int64_t* cb_off,
                       int64_t* rel_ptr, int32_t* rel, int64_t* amap_ptr, int64_t* amap_src, int64_t* amap_dst);
int b2_symbolic_owner(b2_solver* s, int32_t* owner);   /* n_supernodes entries: rank, or -1 for the shared top tree */
/* layout of the multi-GPU exchange: contribution-vector offsets (n_supernodes+1) and the sizes (in doubles) of the
 * leading regions of the update-block / contribution-vector workspaces that are all-reduced */
int b2_symbolic_exchange(b2_solver* s, int64_t* cbv_off, int64_t* exch_cb, int64_t* exch_cbv);
/* test/debug: copy the numeric factor (lval_size doubles, panel layout of b2_symbolic_export) and D (n doubles, permuted
 * order) to the host; synchronises the device. */
int b2_debug_get_factor(b2_solver* s, double* lval_h, double* dvec_h);
/* test/debug: re-factor one warp-class front `reps` times with clock64() stamps at its 8 phase boundaries */
int b2_debug_profile_front(b2_solver* s, int32_t sn, int32_t reps, int64_t* stamps_h);
/* Debug: per-front device timeline of the team-class factor kernels.  With B2_SPARSE_TRACE=1 in the environment at b2_create every
 * front of order <= 64 stamps %globaltimer (ns) when its team starts, when its children have been assembled and when it has
 * finished: stamps_h[3 * sn + {0,1,2}].  Also returns the supernode parents and (w, f) of every front.  *count = number of
 * supernodes; data is copied when capacity >= *count (stamps are zero when tracing is off). */
int b2_debug_trace(b2_solver* s, uint64_t* stamps_h, int32_t* parent_h, int32_t* w_h, int32_t* f_h, int64_t capacity, int64_t* count);

/* ------------------------------------------------------------------ dense LDL^T */
typedef struct b2d_solver b2d_solver;
/* A_d: N x N column-major (ld = lda) on the device, lower triangle read, KEPT BY REFERENCE
 * (lapack.jl:40); the factor is written to an internal buffer (lapack_common.jl:28). */
int b2d_create(int32_t N, int32_t lda, const double* A_d, const b2_options* opt, b2d_solver** out);
int b2d_destroy(b2d_solver* s);
/* Debug: device timeline of the dense look-ahead factorisation.  With B2_DENSE_TRACE=1 in the environment at b2d_create, every kernel
 * of b2d_factorize stamps %globaltimer (ns) at its first entry and last exit; slot = 8 * block column + kind (0 diagonal block, 1 near
 * trsm, 2 near syrk, 3 panel trsm, 4 block-column update, 5 trailing update, 6 inverse, 7 Bunch-Kaufman diagonal block), two
 * uint64 per slot.  *count = number of uint64 values (0 when tracing is off); stamps are copied when capacity >= *count. */
int b2d_debug_trace(b2d_solver* s, uint64_t* stamps_h, int64_t capacity, int64_t* count);
int b2d_factorize(b2d_solver* s, void* stream);
int b2d_inertia(b2d_solver* s, int64_t* num_pos, int64_t* num_zero, int64_t* num_neg, void* stream);
int b2d_inertia_enqueue(b2d_solver* s, void* stream);
int b2d_inertia_fetch(b2d_solver* s, int64_t* num_pos, int64_t* num_zero, int64_t* num_neg);
int b2d_solve(b2d_solver* s, double* x_d, int32_t nrhs, void* stream);
/* Pivots of the last factorisation (host arrays of N entries; any pointer may be NULL); synchronises the device.
 * perm_h[new] = old (the b2_get_perm convention): row `new` of P A P' is row `old` of A.  kind_h: B2_PIVOT_KIND_*.
 * n_2x2: number of 2 x 2 pivots; n_perturbed: number of perturbed pivots.  A static-pivoting handle reports the identity,
 * every kind 1 x 1 and n_2x2 = 0 (its perturbed pivots are counted in n_perturbed only). */
int b2d_pivot_info(b2d_solver* s, int32_t* perm_h, int8_t* kind_h, int64_t* n_2x2, int64_t* n_perturbed);

/* ------------------------------------------------------------------ assembly: COO -> CSC */
/* Host, one-time: CSC pattern of a COO matrix with duplicate merging and the COO->CSC map
 * (src/matrixtools.jl:55-95).  colptr_h[n+1]; rowval_h capacity nnz_coo; map_h[nnz_coo]. */
int b2_coo_to_csc(int32_t m, int32_t n, int64_t nnz_coo, const int32_t* I_h, const int32_t* J_h,
                  int32_t* colptr_h, int32_t* rowval_h, int64_t* map_h, int64_t* nnz_csc);

/* The same construction with device sorts (lib/MadNLPGPU/src/KKT/gpu_sparse.jl:260-302): I_d, J_d, and all outputs are DEVICE arrays
 * (rowval_d capacity nnz_coo); identical output to b2_coo_to_csc.  Synchronises `stream` once to return *nnz_csc. */
int b2_coo_to_csc_device(int32_t m, int32_t n, int64_t nnz_coo, const int32_t* I_d, const int32_t* J_d,
                         int32_t* colptr_d, int32_t* rowval_d, int64_t* map_d, int64_t* nnz_csc, void* stream);

/* Device plan for  dst .= 0; dst[map[k]] += V[k]  (src/matrixtools.jl:79-88) as a race-free,
 * deterministic segmented gather: one thread per destination slot summing its sources in COO
 * order -- bit-identical to the reference's sequential CPU loop. */
typedef struct b2_transfer_plan b2_transfer_plan;
int b2_transfer_plan_create(int64_t nnz_coo, int64_t nnz_csc, const int64_t* map_h, b2_transfer_plan** out);
int b2_transfer_plan_destroy(b2_transfer_plan* p);
int b2_transfer(b2_transfer_plan* p, double* dst_nz_d, const double* V_d, void* stream);

/* ------------------------------------------------------------------ assembly: sparse condensed */
typedef struct b2_condensed_plan b2_condensed_plan;
/* Symbolic (host, one-time): pattern of tril(H) U diag U tril(Jt*Jt') and the dptr/hptr/jptr maps
 * (src/KKT/Sparse/condensed.jl:201-301).  H: n x n lower CSC; Jt: n x m CSC. */
int b2_condensed_symbolic(int32_t n, int32_t m,
                          const int32_t* H_colptr_h, const int32_t* H_rowval_h,
                          const int32_t* Jt_colptr_h, const int32_t* Jt_rowval_h,
                          b2_condensed_plan** out, int64_t* nnz_aug);
/* the same construction with device sorts (condensed.jl:251 on the GPU, lib/MadNLPGPU/src/KKT/gpu_sparse.jl:100-130): patterns are
 * DEVICE arrays; the resulting plan is identical to b2_condensed_symbolic's.  Synchronises `stream`. */
int b2_condensed_symbolic_device(int32_t n, int32_t m,
                                 const int32_t* H_colptr_d, const int32_t* H_rowval_d,
                                 const int32_t* Jt_colptr_d, const int32_t* Jt_rowval_d,
                                 b2_condensed_plan** out, int64_t* nnz_aug, void* stream);
int b2_condensed_pattern(b2_condensed_plan* p, int32_t* colptr_h, int32_t* rowval_h);
int b2_condensed_plan_sizes(b2_condensed_plan* p, int64_t* n_dptr, int64_t* n_hptr, int64_t* n_jptr);
int b2_condensed_plan_destroy(b2_condensed_plan* p);
/* Numeric (device, every iteration), two launches instead of the reference's fill! + 3 kernels
 * (src/KKT/Sparse/condensed.jl:328-366, gpu_sparse.jl:308-340):
 *   diag_buffer = Ss ./ (1 - Sd .* Ss)   with Ss = pr_diag[n:n+m], Sd = du_diag
 *   nz[i] = sum H.nz[..] + pr_diag[..] + sum diag_buffer[c]*Jt.nz[k]*Jt.nz[l]
 * summed per slot in the reference's order (hess, diag, triples) without FMA contraction. */
int b2_condensed_assemble(b2_condensed_plan* p, double* aug_nz_d, const double* pr_diag_d,
                          const double* du_diag_d, const double* H_nz_d, const double* Jt_nz_d,
                          double* diag_buffer_d, void* stream);

/* ------------------------------------------------------------------ assembly: dense condensed */
/* src/KKT/Dense/condensed.jl:157-186.  hess n x n (ld n), jac m x n (ld m), aug N x N (ld N), N = n + n_eq.
 * Only the LOWER triangle of aug is written (what dsytrf('L') and b2d_* read), plus the equality rows. */
int b2d_condensed_assemble(int32_t n, int32_t m, int32_t ns, int32_t n_eq,
                           const int64_t* ind_ineq_d, const int64_t* ind_eq_d,
                           const double* hess_d, const double* jac_d,
                           const double* pr_diag_d, const double* du_diag_d,
                           double* diag_buffer_d, double* aug_d, void* stream);

/* The same assembly with the J' D J contraction on the 5th-generation tensor cores: fp64 is cut into 8 signed 7-bit digits per entry
 * (Ozaki scheme) and the 36 digit-pair products run as exact int8 GEMMs on tcgen05.mma.kind::i8 with TMA-staged operands
 * (csrc/ozaki_kernels.cuh); the result agrees with the fp64 contraction to ~1e-14 of max|W| (parity bar 1e-13,
 * tests/test_gpu_parity_large.py).  The plan owns the digit planes (8 * n_pad * ns_pad bytes), exponents, tile list and tensor maps.
 * ns <= 16384.  b2d_ozaki_plan_status reports whether a (bounded) pipeline wait ever timed out. */
typedef struct b2d_ozaki_plan b2d_ozaki_plan;
int b2d_ozaki_plan_create(int32_t n, int32_t ns, b2d_ozaki_plan** out);
int b2d_ozaki_plan_destroy(b2d_ozaki_plan* p);
int b2d_condensed_assemble_ozaki(b2d_ozaki_plan* p, int32_t n, int32_t m, int32_t ns, int32_t n_eq,
                                 const int64_t* ind_ineq_d, const int64_t* ind_eq_d,
                                 const double* hess_d, const double* jac_d,
                                 const double* pr_diag_d, const double* du_diag_d,
                                 double* diag_buffer_d, double* aug_d, void* stream);
int b2d_ozaki_plan_status(b2d_ozaki_plan* p, int32_t* timed_out, void* stream);

/* dense mat-vecs on column-major device matrices for the DenseCondensedKKTSystem wrappers (jtprod!/mul!/solve_kkt!,
 * src/IPM/factorization.jl:190-229,326-344; the reference calls cuBLAS gemv/symv, lib/MadNLPGPU/.../cuda.jl:54-84):
 *   gemv_n: y = alpha*A*x + beta*y (A rows x cols, ld = lda)   gemv_t: y = alpha*A'*x + beta*y
 *   symv_lower: y = alpha*sym(A)*x + beta*y reading only the lower triangle (the reference's _symv!('L', ...)) */
int b2d_gemv_n(int32_t rows, int32_t cols, int32_t lda, const double* A_d, const double* x_d, double* y_d, double alpha, double beta, void* stream);
int b2d_gemv_t(int32_t rows, int32_t cols, int32_t lda, const double* A_d, const double* x_d, double* y_d, double alpha, double beta, void* stream);
int b2d_symv_lower(int32_t n, int32_t lda, const double* A_d, const double* x_d, double* y_d, double alpha, double beta, void* stream);

/* solve_kkt!(::DenseCondensedKKTSystem, w) (src/IPM/factorization.jl:190-229) and mul!(w, ::AbstractDenseKKTSystem, x, alpha, beta)
 * (:303-324) around b2d_solve.  `b2d_kkt` holds ind_ineq (host, 0-based, ns entries), the derived ind_eq and their inverse map on
 * the device.  jac: m x n column-major (ld m); hess: n x n (lower triangle read, ld n); pd_buffer: n + n_eq; buffer: m;
 * w, x: UnreducedKKTVector buffers [x (n) s (ns) | y (m) | zl | zu].
 *   pre : reduce_rhs!; buffer = 0; buffer[ind_ineq] = D .* (wz + ws ./ Ss); xx = jac' * buffer + wx; xy = wy
 *   (caller: b2d_solve(pd_buffer))
 *   post: wx = xx; dual(w) = jac * wx; wy = xy; wz .*= D; dual(w) .-= buffer; ws = (ws + wz) ./ Ss; finish_aug_solve! */
typedef struct b2_bounds b2_bounds;   /* created by b2_bounds_create, below */
typedef struct b2d_kkt b2d_kkt;
int b2d_kkt_create(int32_t n, int32_t m, int32_t ns, const int64_t* ind_ineq_h, b2d_kkt** out);
int b2d_kkt_destroy(b2d_kkt* k);
int b2d_kkt_solve_pre(b2d_kkt* k, b2_bounds* b, const double* jac_d, const double* pr_diag_d, const double* diag_buffer_d,
                      const double* l_diag_d, const double* u_diag_d, double* buffer_d, double* pd_buffer_d, double* w_d, void* stream);
int b2d_kkt_solve_post(b2d_kkt* k, b2_bounds* b, const double* jac_d, const double* pr_diag_d, const double* diag_buffer_d,
                       const double* l_lower_d, const double* u_lower_d, const double* l_diag_d, const double* u_diag_d,
                       const double* buffer_d, const double* pd_buffer_d, double* w_d, void* stream);
int b2d_kkt_mul(b2d_kkt* k, b2_bounds* b, const double* hess_d, const double* jac_d, const double* reg_d, const double* du_diag_d,
                const double* l_lower_d, const double* u_lower_d, const double* l_diag_d, const double* u_diag_d,
                double alpha, double beta, const double* x_d, double* w_d, void* stream);

/* ------------------------------------------------------------------ IPM vector kernels */
/* Index sets ind_lb / ind_ub over the primal vector (x,s) (src/Callbacks/nlpmodels.jl:369-406), uploaded once
 * together with their inverse maps so that every kernel below is a single race-free pass over n_tot. */
typedef struct b2_bounds b2_bounds;
int b2_bounds_create(int64_t n_tot, int64_t nlb, int64_t nub, const int64_t* ind_lb_h, const int64_t* ind_ub_h,
                     b2_bounds** out);
int b2_bounds_destroy(b2_bounds* b);

/* pr_diag = reg; pr_diag[ind_lb] -= l_lower./l_diag; pr_diag[ind_ub] -= u_lower./u_diag  (IPM/kernels.jl:22-27) */
int b2_set_aug_diagonal(b2_bounds* b, const double* reg_d, const double* l_lower_d, const double* l_diag_d,
                        const double* u_lower_d, const double* u_diag_d, double* pr_diag_d, void* stream);
/* reg += dw; pr_diag += dw; du_diag -= dc   (KKTsystem.jl:222-226) */
int b2_regularize_diagonal(int64_t n_tot, int64_t m, double dw, double dc, double* reg_d, double* pr_diag_d,
                           double* du_diag_d, void* stream);
/* reduce_rhs! / finish_aug_solve!  (IPM/kernels.jl:182-204) on an UnreducedKKTVector buffer
 * w = [xp(n_tot) | y(m) | zl(nlb) | zu(nub)]  (KKT/rhs.jl:101-117) */
int b2_reduce_rhs(b2_bounds* b, int64_t m, const double* l_diag_d, const double* u_diag_d, double* w_d, void* stream);
int b2_finish_aug_solve(b2_bounds* b, int64_t m, const double* l_lower_d, const double* u_lower_d,
                        const double* l_diag_d, const double* u_diag_d, double* w_d, void* stream);

/* CSC sparse mat-vec helpers:  y = alpha*A*x + beta*y  /  y = alpha*A'*x + beta*y  and the symmetric-lower
 * product y = alpha*(L + L' - diag(L))*x + beta*y; gather (row-parallel) forms built once per pattern --
 * replaces the cuSPARSE SpMV calls of lib/MadNLPGPU/src/KKT/gpu_sparse.jl:14-65. */
typedef struct b2_spmv_plan b2_spmv_plan;
int b2_spmv_plan_create(int32_t nrow, int32_t ncol, const int32_t* colptr_h, const int32_t* rowval_h, b2_spmv_plan** out);
int b2_spmv_plan_destroy(b2_spmv_plan* p);
int b2_spmv_n(b2_spmv_plan* p, const double* nz_d, const double* x_d, double* y_d, double alpha, double beta, void* stream);
int b2_spmv_t(b2_spmv_plan* p, const double* nz_d, const double* x_d, double* y_d, double alpha, double beta, void* stream);
int b2_spmv_symlower(b2_spmv_plan* p, const double* nz_d, const double* x_d, double* y_d, double alpha, double beta, void* stream);

/* _kktmul!  (IPM/kernels.jl:161-180) on UnreducedKKTVector buffers w, x */
int b2_kktmul(b2_bounds* b, int64_t m, const double* reg_d, const double* du_diag_d,
              const double* l_lower_d, const double* u_lower_d, const double* l_diag_d, const double* u_diag_d,
              double alpha, double beta, const double* x_d, double* w_d, void* stream);

/* solve_kkt!(::SparseCondensedKKTSystem) pre/post stages around b2_solve (IPM/factorization.jl:143-167), n = nvar, m = ncon:
 *   pre : reduce_rhs!; buffer = D.*(wz + ws./Ss); wx += Jt*buffer
 *   post: buffer2 = Jt'*wx; wz = -buffer + D.*buffer2; ws = (ws+wz)./Ss; finish_aug_solve! */
int b2_condensed_solve_pre(b2_bounds* b, b2_spmv_plan* jt, int64_t n, int64_t m,
                           const double* jt_nz_d, const double* pr_diag_d, const double* diag_buffer_d,
                           const double* l_diag_d, const double* u_diag_d, double* buffer_d, double* w_d, void* stream);
int b2_condensed_solve_post(b2_bounds* b, b2_spmv_plan* jt, int64_t n, int64_t m,
                            const double* jt_nz_d, const double* pr_diag_d, const double* diag_buffer_d,
                            const double* l_lower_d, const double* u_lower_d, const double* l_diag_d, const double* u_diag_d,
                            const double* buffer_d, double* w_d, void* stream);
/* mul!(w, ::SparseCondensedKKTSystem, x, alpha, beta)  (IPM/factorization.jl:303-324) incl. _kktmul! */
int b2_condensed_kkt_mul(b2_bounds* b, b2_spmv_plan* hess, b2_spmv_plan* jt, int64_t n, int64_t m,
                         const double* hess_nz_d, const double* jt_nz_d,
                         const double* reg_d, const double* du_diag_d, const double* l_lower_d, const double* u_lower_d,
                         const double* l_diag_d, const double* u_diag_d, double alpha, double beta,
                         const double* x_d, double* w_d, void* stream);
/* the same product that also accumulates ||w||_inf of its result into *norm_inf_d (device; the caller zeroes it -- 
 * b2_richardson_update does); the residual norm of a Richardson step then costs no extra pass */
int b2_condensed_kkt_mul_norm(b2_bounds* b, b2_spmv_plan* hess, b2_spmv_plan* jt, int64_t n, int64_t m,
                         const double* hess_nz_d, const double* jt_nz_d,
                         const double* reg_d, const double* du_diag_d, const double* l_lower_d, const double* u_lower_d,
                         const double* l_diag_d, const double* u_diag_d, double alpha, double beta,
                         const double* x_d, double* w_d, double* norm_inf_d, void* stream);

/* infinity norm of a device vector into a device scalar (no host sync) */
/* start of solve_refine! (src/LinearSolvers/backsolve.jl:36-44) in one pass: *norm_b_d = ||b||_inf ; x = 0 ; w = b */
int b2_richardson_begin(int64_t n, const double* b_d, double* w_d, double* x_d, double* norm_b_d, void* stream);
/* vector part of one Richardson step (src/LinearSolvers/backsolve.jl:45-48) in one pass: x += w ; w = b ;
 * norms_d[0] = 0 (accumulator for b2_condensed_kkt_mul_norm) ; norms_d[1] = ||x||_inf */
int b2_richardson_update(int64_t n, const double* b_d, double* w_d, double* x_d, double* norms_d, void* stream);
int b2_norm_inf(int64_t n, const double* x_d, double* out_d, void* stream);
/* y += a*x ; y = x ; x = v */
int b2_axpy(int64_t n, double a, const double* x_d, double* y_d, void* stream);
int b2_copy(int64_t n, const double* x_d, double* y_d, void* stream);
/* count <= 16 independent copies dst[k][0:n[k]) = src[k][0:n[k]) in one launch (host arrays of device pointers): how the
 * outputs of the model callbacks (eval_jac_wrapper!/eval_lag_hess_wrapper!, src/IPM/callbacks.jl) and the iterate's
 * diagonals reach the KKT buffers when they are produced elsewhere on the device */
int b2_copy_many(int32_t count, const double* const* src_d, double* const* dst_d, const int64_t* n, void* stream);
int b2_fill(int64_t n, double v, double* x_d, void* stream);

/* ------------------------------------------------------------------ IPM reductions (SURVEY 8f rows 2, 4)
 * The scalars the filter line-search reads every iteration, one single-pass kernel each; same names and argument meaning
 * as src/IPM/kernels.jl (x, xl, xu, f, zl, zu, jacl, dx: length n_tot with +-Inf for absent bounds; zl/zu FULL length,
 * the *_r views of the reference are taken through ind_lb / ind_ub of `b`; dzl/dzu, l: compressed lengths nlb/nub, m).
 * The result is ONE device double at out_d (fetch several with one D2H copy).  Deterministic (fixed reduction tree),
 * NaN-propagating min/max like Julia.  A b2_bounds object serialises its reductions: use it from one stream at a time. */
int b2_get_alpha_max(b2_bounds* b, const double* x_d, const double* xl_d, const double* xu_d, const double* dx_d, double tau,
                     double* out_d, void* stream);                                   /* kernels.jl:356-371 */
int b2_get_alpha_z(b2_bounds* b, const double* zl_d, const double* zu_d, const double* dzl_d, const double* dzu_d, double tau,
                   double* out_d, void* stream);                                     /* :373-388 */
int b2_get_varphi(b2_bounds* b, double obj_val, const double* x_d, const double* xl_d, const double* xu_d, double mu, double* out_d,
                  void* stream);                                                     /* :263-283 */
int b2_get_varphi_d(b2_bounds* b, const double* f_d, const double* x_d, const double* xl_d, const double* xu_d, const double* dx_d,
                    double mu, double* out_d, void* stream);                         /* :341-354 */
int b2_get_inf_du(b2_bounds* b, const double* f_d, const double* zl_d, const double* zu_d, const double* jacl_d, double sd,
                  double* out_d, void* stream);                                      /* :285-291 */
int b2_get_inf_compl(b2_bounds* b, const double* x_d, const double* xl_d, const double* xu_d, const double* zl_d, const double* zu_d,
                     double mu, double sc, double* out_d, void* stream);             /* :293-303 */
int b2_get_average_complementarity(b2_bounds* b, const double* x_d, const double* xl_d, const double* xu_d, const double* zl_d,
                                   const double* zu_d, double* out_d, void* stream); /* :305-314 */
int b2_get_min_complementarity(b2_bounds* b, const double* x_d, const double* xl_d, const double* xu_d, const double* zl_d,
                               const double* zu_d, double* out_d, void* stream);     /* :322-333 */
int b2_get_rel_search_norm(b2_bounds* b, int64_t n, const double* x_d, const double* dx_d, double* out_d, void* stream);   /* :675-681 */
int b2_get_sd(b2_bounds* b, int64_t m, const double* l_d, const double* zl_d, const double* zu_d, double s_max, double* out_d,
              void* stream);                                                         /* :684-689 */
int b2_get_sc(b2_bounds* b, const double* zl_d, const double* zu_d, double s_max, double* out_d, void* stream);            /* :690-695 */
/* set_aug_rhs! (:113-130): p = [ -f + zl - zu - jacl | -c | (xl_r - x_lr) zl_r + mu | (xu_r - x_ur) zu_r - mu ] */
int b2_set_aug_rhs(b2_bounds* b, int64_t m, const double* x_d, const double* xl_d, const double* xu_d, const double* f_d,
                   const double* zl_d, const double* zu_d, const double* jacl_d, const double* c_d, double mu, double* p_d, void* stream);


#ifdef __cplusplus
}
#endif
#endif /* B200KKT_H */
