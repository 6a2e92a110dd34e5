// Bunch-Kaufman pivoting of the dense solver (b2_options.pivoting = B2_PIVOT_BUNCH_KAUFMAN), supernode-bounded as in PARDISO
// (Schenk & Gaertner 2006): the pivot search of block column k only looks at the rows of its own 128 x 128 diagonal block, and the
// symmetric interchanges stay inside that block.  Rows outside the block never move during the factorisation.
//
// A 2 x 2 pivot D_b is stored through its eigen-decomposition D_b = Q diag(lam1, lam2) Q' (Q a Jacobi rotation; a Bunch-Kaufman
// 2 x 2 block has a negative determinant, so one lam is positive and one negative):
//   L11      unit lower (zero between the two columns of a pair), as LAPACK stores it; Linv = L11^{-1} as for static pivoting
//   diagonal / dvec  Lambda
//   L21'     = L21 Q_bd  (Q_bd block diagonal: Q on each pair, 1 elsewhere)
// so L21' Lambda L21'^T = L21 D L21^T and every trailing-update kernel reads its d from the diagonal unchanged.  With
// Q = [[c, s], [-s, c]] stored as rot[p] = c, rot[p + 1] = s (p the first column of the pair): u Q = (c u0 - s u1, s u0 + c u1).
//
//   k_bk_diag128    one CTA: bounded Bunch-Kaufman of the diagonal block in shared memory, write-back, Linv (diag128_invert_store)
//   k_big_trsm<true> (bigfactor_kernels.cuh)  reads column perm[c] of A21 and rotates each row before dividing by Lambda
//   k_bk_swap_left  after the last block: each block's permutation applied to its rows in the columns left of it
// The global permutation P is the product of the block permutations: row ob + i of P A P' is row perm[ob + i] of A.
#pragma once
#include "bigfactor_kernels.cuh"

namespace b2 {

constexpr double BK_ALPHA = 0.64038820320220756;   // (1 + sqrt(17)) / 8: bounds the element growth of one 1 x 1 / 2 x 2 step

struct BkSmem {
    Diag128Smem d;                        // d.Lc: the block with BOTH triangles, Lc[j * DB_LDS + i] = (i, j); d.dd: Lambda
    double rot[DB];
    int32_t perm[DB];                     // block-local: row i of the permuted block is row perm[i] of the original one
    int8_t kind[DB];
    int dec[4];                           // decision for the current pivot: swap s1 <-> s2 (s1 < 0: none), step (1 / 2), kind
};

// Symmetric 2 x 2 Schur decomposition [[a, b], [b, c]] = Q diag(l1, l2) Q', Q = [[cs, sn], [-sn, cs]] (Golub & Van Loan, sym.schur2)
__device__ __forceinline__ void bk_schur2(double a, double b, double c, double& cs, double& sn, double& l1, double& l2) {
    const double tau = (c - a) / (2.0 * b);
    const double t = ((tau >= 0.0) ? 1.0 : -1.0) / (fabs(tau) + hypot(1.0, tau));
    cs = 1.0 / sqrt(1.0 + t * t);
    sn = t * cs;
    l1 = a - t * b;
    l2 = c + t * b;
}

// largest magnitude and its (smallest) index over the warp
__device__ __forceinline__ void bk_warp_argmax(double& v, int& idx) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, v, o);
        const int oi = __shfl_xor_sync(0xffffffffu, idx, o);
        if (ov > v || (ov == v && oi < idx)) { v = ov; idx = oi; }
    }
}

__global__ void __launch_bounds__(256, 1) k_bk_diag128(FactorArgs a, const int32_t* __restrict__ list, int kb,
                                                       double* __restrict__ Linv, const int64_t* __restrict__ linv_off) {
    const int s = list[blockIdx.x];
    const FrontDesc d = a.desc[s];
    if (kb >= d.w) return;
    trace_enter(a, 8 * (kb / DB) + TR_BK);
    extern __shared__ __align__(16) unsigned char dsm_raw[];
    BkSmem& sm = *reinterpret_cast<BkSmem*>(dsm_raw);
    double* M = sm.d.Lc;
    const int f = d.f, nb = min(DB, d.w - kb);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    double* Lp = a.L + d.lp_off;
    // ---- load the lower triangle (coalesced), zero elsewhere, then mirror it into the upper one
    for (int e = tid; e < DB * DB; e += 256) {
        const int i = e & (DB - 1), j = e >> 7;
        M[j * DB_LDS + i] = (i < nb && j <= i) ? Lp[(size_t)(kb + j) * f + kb + i] : 0.0;
    }
    if (tid < DB) sm.perm[tid] = tid;
    __syncthreads();
    for (int e = tid; e < DB * DB; e += 256) {
        const int i = e & (DB - 1), j = e >> 7;
        if (i < j && j < nb) M[j * DB_LDS + i] = M[i * DB_LDS + j];
    }
    __syncthreads();
    // ---- right-looking elimination.  The trailing block is kept fully symmetric; the multipliers l(i, p) of an eliminated column
    //      go to ROW p (M(p, i), i > p), which no later step reads or updates, so that one barrier separates pivot steps.
    int nneg = 0, npert = 0;                                        // (thread 0)
    for (int p = 0; p < nb;) {
        if (warp == 0) {
            const double* col = M + p * DB_LDS;
            double cmax = -1.0;
            int r = DB;
            for (int i = p + 1 + lane; i < nb; i += 32) {
                const double v = fabs(col[i]);
                if (v > cmax) { cmax = v; r = i; }
            }
            bk_warp_argmax(cmax, r);
            const double akk = fabs(col[p]);
            int s1 = -1, s2 = -1, step = 1, kd = B2_PIVOT_KIND_1X1;
            if (!(akk >= a.eps) && !(cmax >= a.eps)) kd = B2_PIVOT_KIND_PERTURBED;    // numerically zero column
            else if (!(akk >= BK_ALPHA * cmax)) {
                const double* cr = M + r * DB_LDS;                        // column r = row r (symmetric)
                double smax = 0.0;
                int dummy = 0;
                for (int i = p + lane; i < nb; i += 32)
                    if (i != r) smax = fmax(smax, fabs(cr[i]));
                bk_warp_argmax(smax, dummy);
                if (akk * smax >= BK_ALPHA * cmax * cmax) {
                } else if (fabs(cr[r]) >= BK_ALPHA * smax) {
                    s1 = p; s2 = r;
                } else {
                    step = 2; kd = B2_PIVOT_KIND_2X2_FIRST;
                    if (r != p + 1) { s1 = p + 1; s2 = r; }
                }
            }
            if (lane == 0) { sm.dec[0] = s1; sm.dec[1] = s2; sm.dec[2] = step; sm.dec[3] = kd; }
        }
        __syncthreads();
        const int s1 = sm.dec[0], s2 = sm.dec[1], step = sm.dec[2], kd = sm.dec[3];
        if (s1 >= 0) {                                              // symmetric interchange s1 <-> s2 (rows of L included)
            if (tid < nb && tid != s1 && tid != s2) {
                double* c = M + tid * DB_LDS;
                const double x = c[s1]; c[s1] = c[s2]; c[s2] = x;
                const double y = M[s1 * DB_LDS + tid]; M[s1 * DB_LDS + tid] = M[s2 * DB_LDS + tid]; M[s2 * DB_LDS + tid] = y;
            } else if (tid == s1) {
                const double x = M[s1 * DB_LDS + s1]; M[s1 * DB_LDS + s1] = M[s2 * DB_LDS + s2]; M[s2 * DB_LDS + s2] = x;
                const double y = M[s1 * DB_LDS + s2]; M[s1 * DB_LDS + s2] = M[s2 * DB_LDS + s1]; M[s2 * DB_LDS + s1] = y;
                const int t = sm.perm[s1]; sm.perm[s1] = sm.perm[s2]; sm.perm[s2] = t;
            }
            __syncthreads();
        }
        const double* w1 = M + p * DB_LDS;
        if (step == 1) {
            const double a11 = w1[p];
            const double dp = (kd == B2_PIVOT_KIND_PERTURBED) ? ((a11 < 0.0) ? -a.eps : a.eps) : a11;
            const double rd = 1.0 / dp;
            const int j0 = p + 1;
            double wi[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) wi[u] = (j0 + lane + 32 * u < nb) ? w1[j0 + lane + 32 * u] : 0.0;
            for (int j = j0 + warp; j < nb; j += 8) {
                const double wj = w1[j];
                double* c = M + j * DB_LDS;
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int i = j0 + lane + 32 * u;
                    if (i < nb) c[i] = fma(-(wi[u] * wj), rd, c[i]);
                }
            }
            if (tid >= j0 && tid < nb) M[tid * DB_LDS + p] = w1[tid] * rd;
            if (tid == 0) {
                sm.d.dd[p] = dp; sm.kind[p] = (int8_t)kd; sm.rot[p] = 0.0;
                if (kd == B2_PIVOT_KIND_PERTURBED) ++npert;
                else if (dp < 0.0) ++nneg;
            }
        } else {
            const double* w2 = M + (p + 1) * DB_LDS;
            const double a11 = w1[p], a21 = w1[p + 1], a22 = w2[p + 1];
            const double det = a11 * a22 - a21 * a21;                 // < 0 (Bunch-Kaufman 2 x 2 condition)
            const double e11 = a22 / det, e12 = -a21 / det, e22 = a11 / det;
            const int j0 = p + 2;
            double u1[4], u2[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = j0 + lane + 32 * u;
                u1[u] = (i < nb) ? w1[i] : 0.0;
                u2[u] = (i < nb) ? w2[i] : 0.0;
            }
            for (int j = j0 + warp; j < nb; j += 8) {
                const double v1 = w1[j], v2 = w2[j];
                double* c = M + j * DB_LDS;
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int i = j0 + lane + 32 * u;
                    if (i < nb) c[i] -= e11 * (u1[u] * v1) + e12 * (u1[u] * v2 + u2[u] * v1) + e22 * (u2[u] * v2);
                }
            }
            if (tid >= j0 && tid < nb) {
                M[tid * DB_LDS + p] = e11 * w1[tid] + e12 * w2[tid];
                M[tid * DB_LDS + p + 1] = e12 * w1[tid] + e22 * w2[tid];
            }
            if (tid == 0) {
                double cs, sn, l1, l2;
                bk_schur2(a11, a21, a22, cs, sn, l1, l2);
                M[(p + 1) * DB_LDS + p] = 0.0;                           // l(p + 1, p) of a pair
                sm.d.dd[p] = l1; sm.d.dd[p + 1] = l2;
                sm.rot[p] = cs; sm.rot[p + 1] = sn;
                sm.kind[p] = (int8_t)B2_PIVOT_KIND_2X2_FIRST; sm.kind[p + 1] = (int8_t)B2_PIVOT_KIND_2X2_SECOND;
                nneg += (l1 < 0.0) + (l2 < 0.0);
            }
        }
        __syncthreads();
        p += step;
    }
    if (tid == 0) {
        if (nneg) atomicAdd(a.counters + 0, nneg);
        if (npert) atomicAdd(a.counters + 1, npert);
    }
    // ---- multipliers to the lower triangle (the layout diag128_invert_store expects), then write back L11 and Lambda
    for (int e = tid; e < DB * DB; e += 256) {
        const int i = e & (DB - 1), j = e >> 7;
        if (j < i && i < nb) M[j * DB_LDS + i] = M[i * DB_LDS + j];
    }
    __syncthreads();
    for (int e = tid; e < DB * DB; e += 256) {
        const int i = e & (DB - 1), j = e >> 7;
        if (i < nb && j < i) Lp[(size_t)(kb + j) * f + kb + i] = M[j * DB_LDS + i];
    }
    if (tid < nb) {
        const double lam = sm.d.dd[tid];
        Lp[(size_t)(kb + tid) * f + kb + tid] = lam;
        a.dvec[d.col0 + kb + tid] = lam;
        a.perm[d.col0 + kb + tid] = d.col0 + kb + sm.perm[tid];
        a.pkind[d.col0 + kb + tid] = sm.kind[tid];
        a.rot[d.col0 + kb + tid] = sm.rot[tid];
    }
    __syncthreads();
    for (int e = tid; e < DB * DB; e += 256) {
        const int i = e & (DB - 1), j = e >> 7;
        if (i <= j) M[j * DB_LDS + i] = 0.0;
    }
    diag128_invert_store(sm.d, tid, nb, Linv + linv_off[s] + (size_t)(kb / DB) * DB * DB);
    trace_exit(a, 8 * (kb / DB) + TR_BK);
}

// Row kb + i of every column left of block k (c < kb) becomes row perm[kb + i]: the block permutations applied to the finished
// L21' blocks.  Grid (column c, block k - 1), one thread per row of the block; nothing of the factorisation reads these rows after
// k_bk_diag128(k), only the solves do.
__global__ void __launch_bounds__(DB) k_bk_swap_left(int N, double* __restrict__ L, const int32_t* __restrict__ perm) {
    const int kb = (blockIdx.y + 1) * DB, c = blockIdx.x;
    if (c >= kb) return;
    const int nb = min(DB, N - kb), i = threadIdx.x;
    double* col = L + (size_t)c * N;
    const double v = (i < nb) ? col[perm[kb + i]] : 0.0;
    __syncthreads();
    if (i < nb) col[kb + i] = v;
}

}  // namespace b2
