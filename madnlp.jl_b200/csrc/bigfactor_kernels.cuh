// Blocked right-looking LDL^T of the HBM-resident fronts (order > small_front_max) and of the dense solver, 128 pivot
// columns per outer step, three launches per step:
//
//   k_big_diag128   one CTA per front: the 128 x 128 diagonal block is factorised entirely in shared memory
//                   (4 sub-blocks of 32: register LDL^T by one warp, sub-panel substitution, in-block trailing update),
//                   written back (unit-lower L11, D), and its unit-lower INVERSE is formed in place and stored to the
//                   Linv buffer -- the same blocks the multi-CTA triangular solves use (bigsolve_kernels.cuh).
//   k_big_trsm      rows below the block:  L21 = A21 * L11^{-T} * D^{-1}  as a DMMA GEMM against Linv (64 rows per CTA,
//                   operands streamed by cp.async), in place.
//   k_big_update_pipe (front_kernels.cuh)  trailing update with all 128 pivots at once.
//
// so a front of order N costs 3*N/128 dependent launches instead of 13*N/128, and the diagonal-block inversion is no
// longer a separate pass.  Pivoting is static (front_kernels.cuh): |d| < eps is replaced by sign(d)*eps and counted.  The dense
// solver's opt-in Bunch-Kaufman mode replaces k_big_diag128 by k_bk_diag128 (bkpivot_kernels.cuh) and runs k_big_trsm<true>.
#pragma once
#include "front_kernels.cuh"

namespace b2 {

constexpr int DB = 128;                   // outer block (== BS of the solve kernels)

// Shared-memory / warp-shuffle issue is the scarce resource of a single SM here (measured on B200,
// tools/microbench/fp64_pipes.cu: one LDS.64 or SHFL.64 per ~4.6-9 clk per scheduler vs one DFMA per ~2 clk), so the
// block lives in REGISTERS: 256 threads as a 16 x 16 grid, thread (ty, tx) owns the 8 x 8 entries (ty + 16a, tx + 16b)
// -- cyclic, so the shrinking trailing matrix stays balanced.  The matrix is kept fully symmetric, which makes the pivot
// column also the pivot row: per pivot the 16 owner threads publish it (one barrier), and every thread then needs just
// 8 + 8 values (conflict-free: lanes read consecutive or identical addresses) for up to 64 FMAs.  Entries of already-eliminated rows/columns in a
// thread's boundary sub-block keep receiving (meaningless) updates; they are never read again.
// Pivot-to-pivot synchronisation is an mbarrier per buffer instead of __syncthreads: the 16 threads that own the NEXT
// pivot column update it first, publish it and arrive; everybody else arrives as soon as the current column has been
// read, so the rest of the rank-1 update overlaps the owners' critical path (wait -> rcp -> column -> publish).
constexpr int DB_LDS = DB + 4;            // leading dimension of the block in shared memory: 132 = 4 (mod 16) doubles, so that the DMMA
                                          // fragment loads of the blocked inversion (8 rows x 4 k, or 4 k x 8 columns) take the minimum of
                                          // two wavefronts; the transposed reads of the symmetric fill stay cheap
struct Diag128Smem {
    double Lc[DB * DB_LDS];               // stage[j*DB_LDS + i] on entry; then Lc[k*DB_LDS + i] = l(i,k) for i > k, 0 for i <= k
    double ubuf[2][DB];                   // pivot column (unscaled), double-buffered
    double xbuf[2][DB];                   // row k of the inverse
    double dd[DB];
    double tb[32 * 36];                   // phase I: one 32 x 32 product of the blocked inversion (column-major, ld 36)
    unsigned long long bar[4];            // [0..1] phase F (2..3 unused)
};
__device__ __forceinline__ void mbar_init(unsigned long long* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"((unsigned)__cvta_generic_to_shared(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, int parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "MBAR_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra MBAR_DONE;\n"
        "bra MBAR_WAIT;\n"
        "MBAR_DONE:\n"
        "}\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(parity) : "memory");
}

// Phase I of the diagonal-block kernel as a function (also the body of k_big_inv128): on entry sm.Lc[k*DB_LDS + i] = l(i,k) for i > k and
// 0 for i <= k; on exit the unit-lower inverse is in sm.Lc and has been stored to `out` (column-major, ld DB, zero outside nb x nb).
__device__ __forceinline__ void diag128_invert_store(Diag128Smem& sm, const int tid, const int nb, double* __restrict__ out) {
    // ---- phase I: X = L11^{-1}, BLOCKED (4 x 4 blocks of 32), in place in sm.Lc (L11 has been written back to global memory):
    //      (1) the four unit-lower diagonal blocks are inverted by one warp each -- lane j runs the forward substitution of column j
    //          in registers, every l(i,k) is a shared-memory broadcast;
    //      (2) X_ij = -X_ii * (sum_{k=j}^{i-1} L_ik X_kj) for i > j, block row by block row and j ascending (so that L_ij may be
    //          overwritten by X_ij), each 32^3 product on the fp64 tensor pipe (8 warps x 2 tiles of m8n8k4 DMMA).
    //      The round-1 version applied the 127 elementary row operations one by one (one mbarrier hand-off each, ~340 clk per step,
    //      22 us of the 60 us this kernel sits on the factorisation's critical path); this is ~16 dependent steps.
    __syncthreads();                                               // (the caller's reads of sm.Lc -- write-back of L11 -- are complete)
    {
        const int warp = tid >> 5, lane = tid & 31;
        double* Lc = sm.Lc;
        if (warp < 4) {
            const int o = 32 * warp;
            double x[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) x[i] = (i == lane) ? 1.0 : 0.0;
#pragma unroll
            for (int i = 1; i < 32; ++i) {
                double acc = 0.0;
#pragma unroll
                for (int k = 0; k < i; ++k) acc = fma(Lc[(o + k) * DB_LDS + o + i], x[k], acc);      // x[k] = 0 for k < lane: harmless
                x[i] = (i > lane) ? -acc : x[i];
            }
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 32; ++i) Lc[(o + lane) * DB_LDS + o + i] = (i >= lane) ? x[i] : 0.0; // column `lane` of X_bb incl. the unit diagonal
        }
        __syncthreads();
        const int g = lane >> 2, q = lane & 3;
        const int tr = warp & 3, tc0 = (warp >> 2) * 2;          // this warp's two 8 x 8 output tiles: tile row tr, tile columns tc0, tc0 + 1
        for (int bi = 1; bi < 4; ++bi) {
            for (int bj = 0; bj < bi; ++bj) {
                double c[2][2];
                // stage 1: T = sum_{k = bj}^{bi-1} L(bi, k) X(k, bj)
                c[0][0] = c[0][1] = c[1][0] = c[1][1] = 0.0;
                for (int bk = bj; bk < bi; ++bk) {
#pragma unroll
                    for (int k0 = 0; k0 < 32; k0 += 4) {
                        const double af = Lc[(32 * bk + k0 + q) * DB_LDS + 32 * bi + 8 * tr + g];            // L(bi,bk)(row 8tr+g, k0+q)
#pragma unroll
                        for (int y = 0; y < 2; ++y) {
                            const double bf = Lc[(32 * bj + 8 * (tc0 + y) + g) * DB_LDS + 32 * bk + k0 + q];  // X(bk,bj)(k0+q, col)
                            asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                                         : "+d"(c[y][0]), "+d"(c[y][1]) : "d"(af), "d"(bf));
                        }
                    }
                }
#pragma unroll
                for (int y = 0; y < 2; ++y)
#pragma unroll
                    for (int e = 0; e < 2; ++e) sm.tb[(8 * (tc0 + y) + 2 * q + e) * 36 + 8 * tr + g] = c[y][e];
                __syncthreads();
                // stage 2: X(bi, bj) = -X(bi, bi) * T      (overwrites L(bi, bj): no later product needs it)
                c[0][0] = c[0][1] = c[1][0] = c[1][1] = 0.0;
#pragma unroll
                for (int k0 = 0; k0 < 32; k0 += 4) {
                    const double af = Lc[(32 * bi + k0 + q) * DB_LDS + 32 * bi + 8 * tr + g];                 // X(bi,bi)(row, k0+q)
#pragma unroll
                    for (int y = 0; y < 2; ++y) {
                        const double bf = sm.tb[(8 * (tc0 + y) + g) * 36 + k0 + q];                       // T(k0+q, col)
                        asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                                     : "+d"(c[y][0]), "+d"(c[y][1]) : "d"(af), "d"(bf));
                    }
                }
                __syncthreads();                                   // every warp has read L(bi, bj) (stage 1) and T (stage 2)
#pragma unroll
                for (int y = 0; y < 2; ++y)
#pragma unroll
                    for (int e = 0; e < 2; ++e) Lc[(32 * bj + 8 * (tc0 + y) + 2 * q + e) * DB_LDS + 32 * bi + 8 * tr + g] = -c[y][e];
                __syncthreads();
            }
        }
    }
    __syncthreads();
    // ---- store the inverse, column-major with ld DB, zero outside the nb x nb unit-lower block
    for (int e = tid; e < DB * DB; e += 256) {
        const int i = e & (DB - 1), j = e >> 7;
        double v = 0.0;
        if (i < nb && j < nb && i >= j) v = (i == j) ? 1.0 : sm.Lc[j * DB_LDS + i];
        out[(size_t)j * DB + i] = v;
    }
}

__global__ void __launch_bounds__(256, 1) k_big_diag128(FactorArgs a, const int32_t* __restrict__ list, int kb,
                                                        double* __restrict__ Linv, const int64_t* __restrict__ linv_off, int with_inv) {
    pdl_sync();                                                    // (no-op unless launched with the PDL attribute: dense chain)
    const int s = list[blockIdx.x];
    const FrontDesc d = a.desc[s];
    if (kb >= d.w) return;
    trace_enter(a, 8 * (kb / DB) + TR_DIAG);
    extern __shared__ __align__(16) unsigned char dsm_raw[];
    Diag128Smem& sm = *reinterpret_cast<Diag128Smem*>(dsm_raw);
    const int f = d.f, nb = min(DB, d.w - kb);
    const int tid = threadIdx.x, ty = tid & 15, tx = tid >> 4;
    double* Lp = a.L + d.lp_off;
#ifdef B2_DIAG_PROF
    long long tprof[8]; int np = 0;
#define DPROF() do { __syncthreads(); tprof[np++] = clock64(); } while (0)
#else
#define DPROF() do {} while (0)
#endif
    DPROF();
    if (tid < 4) mbar_init(&sm.bar[tid], 256);
    // ---- stage the lower triangle (coalesced: i fastest), then pick the symmetric 8 x 8 register block out of it
    double* stage = sm.Lc;                                         // stage[j*DB_LDS + i], i >= j
    for (int e = tid; e < DB * DB; e += 256) {                     // all 64 copies of a thread in flight at once
        const int i = e & (DB - 1), j = e >> 7;
        if (j <= i) cp_async8_zfill(stage + j * DB_LDS + i, Lp + (size_t)(kb + j) * f + kb + min(i, nb - 1), i < nb);
    }
    cp_async_commit_group();
    cp_async_wait_group_n<0>();
    __syncthreads();
    if (nb < DB) {                                                 // identity padding
        if (tid < DB && tid >= nb) stage[tid * DB_LDS + tid] = 1.0;
        __syncthreads();
    }
    double A[8][8];
#pragma unroll
    for (int ia = 0; ia < 8; ++ia)
#pragma unroll
        for (int ib = 0; ib < 8; ++ib) {
            const int i = ty + 16 * ia, j = tx + 16 * ib;
            A[ia][ib] = (ia >= ib) ? stage[min(i, j) * DB_LDS + max(i, j)] : 0.0;    // block-lower part only (see phase F)
        }
    __syncthreads();
    int nneg = 0, npert = 0;
    DPROF();
    // ---- phase F: unblocked right-looking LDL^T.  Only the register blocks on or below the block diagonal (ia >= ib: 36 of the 64)
    //      are kept up to date -- the diagonal blocks stay fully symmetric, so every pivot column is still read out of one b-index.
    if (tx == 0) {
#pragma unroll
        for (int ia = 0; ia < 8; ++ia) sm.ubuf[0][ty + 16 * ia] = A[ia][0];
    }
    mbar_arrive(&sm.bar[0]);
#pragma unroll
    for (int kq = 0; kq < 8; ++kq) {
        for (int kk = 0; kk < 16; ++kk) {
            const int k = 16 * kq + kk;
            if (k >= nb) break;
            const double* ub = sm.ubuf[k & 1];
            mbar_wait(&sm.bar[k & 1], (k >> 1) & 1);
            double dk = ub[k];
            double ur[8], uc[8];
#pragma unroll
            for (int ia = 0; ia < 8; ++ia) ur[ia] = (ia >= kq) ? ub[ty + 16 * ia] : 0.0;
#pragma unroll
            for (int ib = 0; ib < 8; ++ib) uc[ib] = (ib >= kq) ? ub[tx + 16 * ib] : 0.0;
            const bool have_next = k + 1 < nb;
            const bool own_next = tx == ((kk + 1) & 15);
            if (have_next && !own_next) mbar_arrive(&sm.bar[(k + 1) & 1]);     // (this column has been read)
            if (!(fabs(dk) >= a.eps)) { dk = (dk < 0.0) ? -a.eps : a.eps; ++npert; }
            else if (dk < 0.0) ++nneg;
            const double rk = fast_rcp_d(dk);
            double li[8];
#pragma unroll
            for (int ia = 0; ia < 8; ++ia) li[ia] = -ur[ia] * rk;
            // the two candidate next-pivot columns first (b-index kq, or kq+1 when kk == 15)
#pragma unroll
            for (int ib = kq; ib < min(kq + 2, 8); ++ib)
#pragma unroll
                for (int ia = 0; ia < 8; ++ia)
                    if (ia >= kq && ia >= ib) A[ia][ib] = fma(li[ia], uc[ib], A[ia][ib]);
            if (have_next && own_next) {
                double* un = sm.ubuf[(k + 1) & 1];
#pragma unroll
                for (int ia = 0; ia < 8; ++ia) un[ty + 16 * ia] = (kk == 15) ? A[ia][min(kq + 1, 7)] : A[ia][kq];
                mbar_arrive(&sm.bar[(k + 1) & 1]);
            }
            if (tx == kk) {
                double* lc = sm.Lc + k * DB_LDS + ty;
#pragma unroll
                for (int ia = 0; ia < 8; ++ia) lc[16 * ia] = (ty + 16 * ia > k) ? -li[ia] : 0.0;
                if (ty == kk) sm.dd[k] = dk;
            }
#pragma unroll
            for (int ib = kq + 2; ib < 8; ++ib)
#pragma unroll
                for (int ia = 0; ia < 8; ++ia)
                    if (ia >= kq && ia >= ib) A[ia][ib] = fma(li[ia], uc[ib], A[ia][ib]);
        }
    }
    if (tid == 0) {
        if (nneg) atomicAdd(a.counters + 0, nneg);
        if (npert) atomicAdd(a.counters + 1, npert);
    }
    __syncthreads();
    DPROF();
    // ---- write back L11 (strict lower, unit diagonal implied) and D
    for (int e = tid; e < DB * DB; e += 256) {
        const int i = e & (DB - 1), j = e >> 7;
        if (i < nb && j < i) Lp[(size_t)(kb + j) * f + kb + i] = sm.Lc[j * DB_LDS + i];
    }
    if (tid < nb) {
        Lp[(size_t)(kb + tid) * f + kb + tid] = sm.dd[tid];
        a.dvec[d.col0 + kb + tid] = sm.dd[tid];
    }
    DPROF();
    if (!with_inv) { trace_exit(a, 8 * (kb / DB) + TR_DIAG); return; }   // dense chain: the inverse is formed off the critical path (k_big_inv128)
    diag128_invert_store(sm, tid, nb, Linv + linv_off[s] + (size_t)(kb / DB) * DB * DB);
    trace_exit(a, 8 * (kb / DB) + TR_DIAG);
    DPROF();
#ifdef B2_DIAG_PROF
    DPROF();
    if (tid == 0 && blockIdx.x == 0 && (kb == 0 || kb == 1280))
        printf("diag128 kb=%d nb=%d: load %lld  F %lld  writeback %lld  I+store %lld  clk\n", kb, nb, tprof[1] - tprof[0], tprof[2] - tprof[1],
               tprof[3] - tprof[2], tprof[4] - tprof[3]);
#endif
#undef DPROF
}

// L21 = A21 * Linv^T * D^{-1} for the rows below the diagonal block, in place.  GEMM view (transposed so that the
// 128-wide side is the pivot-column index):  Ut(c, i) = sum_{k <= c} Linv(c, k) * A21(i, k);  tile 128 (c) x 64 (rows i).
// PIV (Bunch-Kaufman, bkpivot_kernels.cuh): column c of the permuted A21 is column perm[kb + c] of the stored one, and each row
// u = Ut(:, i) is rotated by the block's pair rotations before the division by Lambda:  L21' = A21 P' L11^{-T} Q_bd Lambda^{-1}.
// In place is safe: a CTA has staged every column of its 64-row strip before its epilogue writes any of them.
constexpr int TR_ROWS = GU_N;            // 64 rows of the front per CTA
template <bool PIV>
__global__ void __launch_bounds__(256, 2) k_big_trsm(FactorArgs a, const int32_t* __restrict__ list, int kb,
                                                     const double* __restrict__ Linv, const int64_t* __restrict__ linv_off, int bx0) {
    const int s = list[blockIdx.y];
    const FrontDesc d = a.desc[s];
    if (kb >= d.w) return;
    const int f = d.f, nb = min(DB, d.w - kb);
    const int r0 = kb + nb + (blockIdx.x + bx0) * TR_ROWS;             // bx0: first 64-row block handled by this launch
    if (r0 >= f) return;
    trace_enter(a, 8 * (kb / DB) + TR_TRSM);
    extern __shared__ __align__(16) double gu_sm[];
    double* As = gu_sm;                                               // [stage][k][GU_LDA]  Linv(c, k)
    double* Bs = gu_sm + GU_STAGES * GU_K * GU_LDA;                   // [stage][k][GU_LDB]  A21(i, k)
    double* dinv = Bs + GU_STAGES * GU_K * GU_LDB;
    double* Lp = a.L + d.lp_off;
    const double* Li = Linv + linv_off[s] + (size_t)(kb / DB) * DB * DB;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, q = lane & 3;
    const int wi = (warp & 3) * 32, wj = (warp >> 2) * 32;
    if (tid < DB) dinv[tid] = (tid < nb) ? 1.0 / Lp[(size_t)(kb + tid) * f + kb + tid] : 0.0;
    const int nchunk = (nb + GU_K - 1) / GU_K;
    const int la_c = tid & (GU_M - 1), la_k = tid >> 7;
    const int lb_i = tid & (GU_N - 1), lb_k = tid >> 6;
    const bool b_ok = r0 + lb_i < f;
    const double* b_src = Lp + (size_t)kb * f + (b_ok ? r0 + lb_i : 0);
    auto issue = [&](int ch) {
        const int st = ch % GU_STAGES;
        double* Ad = As + (size_t)st * GU_K * GU_LDA + la_c;
        double* Bd = Bs + (size_t)st * GU_K * GU_LDB + lb_i;
#pragma unroll
        for (int p = 0; p < GU_K / 2; ++p) {
            const int k = ch * GU_K + la_k + 2 * p;                   // k < 128 always; the buffer is zero-padded
            cp_async8_zfill(Ad + (la_k + 2 * p) * GU_LDA, Li + (size_t)k * DB + la_c, true);
        }
#pragma unroll
        for (int p = 0; p < GU_K / 4; ++p) {
            const int k = ch * GU_K + lb_k + 4 * p;
            const bool ok = b_ok && k < nb;
            const int kc = PIV ? (ok ? a.perm[d.col0 + kb + k] - d.col0 - kb : 0) : (ok ? k : 0);
            cp_async8_zfill(Bd + (lb_k + 4 * p) * GU_LDB, b_src + (size_t)kc * f, ok);
        }
    };
#pragma unroll
    for (int sgi = 0; sgi < GU_STAGES - 1; ++sgi) {
        if (sgi < nchunk) issue(sgi);
        cp_async_commit_group();
    }
    double c[4][4][2];
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) c[x][y][0] = c[x][y][1] = 0.0;
    for (int ch = 0; ch < nchunk; ++ch) {
        cp_async_wait_group_n<GU_STAGES - 2>();
        __syncthreads();
        if (ch + GU_STAGES - 1 < nchunk) issue(ch + GU_STAGES - 1);
        cp_async_commit_group();
        if (wi + 31 < ch * GU_K) continue;                            // Linv(c, k) = 0 for k > c: nothing for this warp
        const double* Ab = As + (size_t)(ch % GU_STAGES) * GU_K * GU_LDA;
        const double* Bb = Bs + (size_t)(ch % GU_STAGES) * GU_K * GU_LDB;
#pragma unroll
        for (int k0 = 0; k0 < GU_K; k0 += 4) {
            double af[4], bf[4];
#pragma unroll
            for (int x = 0; x < 4; ++x) af[x] = Ab[(k0 + q) * GU_LDA + wi + 8 * x + g];
#pragma unroll
            for (int y = 0; y < 4; ++y) bf[y] = Bb[(k0 + q) * GU_LDB + wj + 8 * y + g];
#pragma unroll
            for (int x = 0; x < 4; ++x)
#pragma unroll
                for (int y = 0; y < 4; ++y)
                    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                                 : "+d"(c[x][y][0]), "+d"(c[x][y][1])
                                 : "d"(af[x]), "d"(bf[y]));
        }
    }
    // epilogue: Ut -> shared memory as Cs[i][c], then coalesced stores of L21(i, c) = Ut(c, i) / d_c  (i fastest)
    cp_async_wait_group_n<0>();
    __syncthreads();
    double* Cs = gu_sm;                                               // [TR_ROWS][GU_LDC]
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y)
#pragma unroll
            for (int e = 0; e < 2; ++e) Cs[(wj + 8 * y + 2 * q + e) * GU_LDC + wi + 8 * x + g] = c[x][y][e];
    __syncthreads();
    const int i = tid & (TR_ROWS - 1);
    if (r0 + i < f) {
        for (int cc = tid >> 6; cc < nb; cc += 4) {
            double u = Cs[i * GU_LDC + cc];
            if (PIV) {                                                // (u Q)_c over a pair (p, p + 1), Q = [[cs, sn], [-sn, cs]]
                const int kd = a.pkind[d.col0 + kb + cc];
                if (kd == B2_PIVOT_KIND_2X2_FIRST) {
                    const double cs = a.rot[d.col0 + kb + cc], sn = a.rot[d.col0 + kb + cc + 1];
                    u = cs * u - sn * Cs[i * GU_LDC + cc + 1];
                } else if (kd == B2_PIVOT_KIND_2X2_SECOND) {
                    const double cs = a.rot[d.col0 + kb + cc - 1], sn = a.rot[d.col0 + kb + cc];
                    u = sn * Cs[i * GU_LDC + cc - 1] + cs * u;
                }
            }
            Lp[(size_t)(kb + cc) * f + r0 + i] = u * dinv[cc];
        }
    }
    trace_exit(a, 8 * (kb / DB) + TR_TRSM);
}

// ----------------------------------------------------------------------------------------------------------
// Near-diagonal step of the dense look-ahead schedule (sparse_ldl.cu: enqueue_dense_factor_lookahead).  Between two diagonal-block
// kernels the critical path only needs (1) the 128 x 128 block of L right below the diagonal block and (2) the update of the NEXT
// diagonal block with it.  The general kernels above do these as parts of whole-panel launches whose latency is one 128 x 64 x 128
// tile on one SM (12 + 8 us); here the same 2 x 2.1 Mflop are cut into pieces small enough that latency, not per-SM tensor rate,
// is what remains (~2 x 3 us), and the rest of the panel moves to a side branch that runs beside the next diagonal block.
//
//   k_near_trsm  16 CTAs x 8 rows:  L(i, c) = (sum_{k <= c} A(i, k) Linv(c, k)) / d_c   for the rows i of block k+1, in place.
//                Whole operands land in shared memory in one cp.async round trip (8 x 128 of A, the lower part of Linv); warp w owns
//                the 8-column tiles w and 15 - w (balanced: 8 (w+1) + 8 (16-w) = 136 k-steps of 4).
//   k_near_syrk  10 CTAs, one 32 x 32 tile of the lower triangle each:  C(i, j) -= sum_k L(i, k) d_k L(j, k),  K = 128.
// Both require full blocks (kb + 2*DB <= f); the caller falls back to the general kernels otherwise.
// ----------------------------------------------------------------------------------------------------------
constexpr int NT_ROWS = 8;                       // rows per CTA of k_near_trsm
constexpr int NT_LDA = 12;                       // A strip: As[k*12 + i]  (12 q + g covers every 16-bank residue exactly twice)
constexpr int NT_LDB = DB + 4;                   // Linv:    Bs[k*132 + c]
constexpr size_t NT_SMEM = (size_t)(DB * NT_LDA + DB * NT_LDB + DB) * sizeof(double);
__device__ __forceinline__ void cp_async16_l2(void* smem_dst, const void* gsrc) {
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(gsrc) : "memory");
}
__global__ void __launch_bounds__(256, 1) k_near_trsm(FactorArgs a, const int32_t* __restrict__ list, int kb,
                                                      const double* __restrict__ Linv, const int64_t* __restrict__ linv_off) {
    pdl_sync();
    const int s = list[0];
    const FrontDesc d = a.desc[s];
    const int f = d.f;
    const int r0 = kb + DB + blockIdx.x * NT_ROWS;
    trace_enter(a, 8 * (kb / DB) + TR_NEAR1);
    extern __shared__ __align__(16) double nt_sm[];
    double* As = nt_sm;                           // [128][NT_LDA]
    double* Bs = As + DB * NT_LDA;                // [128][NT_LDB]
    double* dinv = Bs + DB * NT_LDB;              // [128]
    double* Lp = a.L + d.lp_off;
    const double* Li = Linv + linv_off[s] + (size_t)(kb / DB) * DB * DB;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, q = lane & 3;
    // A strip: 128 k x 8 rows (64 contiguous bytes per k)
    for (int e = tid; e < DB * NT_ROWS; e += 256) {
        const int i = e & (NT_ROWS - 1), k = e >> 3;
        cp_async8_zfill(As + k * NT_LDA + i, Lp + (size_t)(kb + k) * f + r0 + i, true);
    }
    // Linv(c, k) at Li[k*DB + c]: row k is needed for the 16-column groups that contain or follow k (pairs of columns, 16 bytes)
    for (int e = tid; e < DB * (DB / 2); e += 256) {
        const int p = e & (DB / 2 - 1), k = e >> 6;
        if (k < 16 * (p / 8 + 1)) cp_async16_l2(Bs + k * NT_LDB + 2 * p, Li + (size_t)k * DB + 2 * p);
    }
    cp_async_commit_group();
    if (tid < DB) dinv[tid] = 1.0 / a.dvec[d.col0 + kb + tid];
    cp_async_wait_group_n<0>();
    __syncthreads();
    double c[2][2];
    const int t0 = warp, t1 = 15 - warp;                               // this warp's two 8-column tiles
#pragma unroll
    for (int y = 0; y < 2; ++y) {
        const int t = y ? t1 : t0;
        const int kend = 8 * (t + 1);                                  // Linv(c, k) = 0 for k > c
        double c0 = 0.0, c1 = 0.0;
        for (int k0 = 0; k0 < kend; k0 += 4) {
            const double af = As[(k0 + q) * NT_LDA + g];
            const double bf = Bs[(k0 + q) * NT_LDB + 8 * t + g];
            asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n" : "+d"(c0), "+d"(c1) : "d"(af), "d"(bf));
        }
        c[y][0] = c0; c[y][1] = c1;
    }
    // lane holds U(i = g, c = 8 t + 2 q + e); every thread has finished with the global A strip (it was read into shared memory
    // before the barrier), so the in-place store is safe
#pragma unroll
    for (int y = 0; y < 2; ++y) {
        const int t = y ? t1 : t0;
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int cc = 8 * t + 2 * q + e;
            Lp[(size_t)(kb + cc) * f + r0 + g] = c[y][e] * dinv[cc];
        }
    }
    trace_exit(a, 8 * (kb / DB) + TR_NEAR1);
}

constexpr int NS_T = 32;                         // tile order of k_near_syrk
constexpr int NS_LD = NS_T + 4;                  // 36 = 4 (mod 16)
constexpr size_t NS_SMEM = (size_t)(2 * DB * NS_LD + DB) * sizeof(double);
__global__ void __launch_bounds__(256, 2) k_near_syrk(FactorArgs a, const int32_t* __restrict__ list, int kb) {
    pdl_sync();
    const int s = list[0];
    const FrontDesc d = a.desc[s];
    const int f = d.f;
    // blockIdx.x -> (ib, jb), jb <= ib, of the 4 x 4 tile grid
    int ib = 0, rem = blockIdx.x;
    while (rem > ib) { rem -= ib + 1; ++ib; }
    const int jb = rem;
    const int base = kb + DB;                                          // first row / column of the next diagonal block
    trace_enter(a, 8 * (kb / DB) + TR_NEAR2);
    extern __shared__ __align__(16) double ns_sm[];
    double* As = ns_sm;                           // [128][NS_LD]  L(base + 32 ib + i, kb + k)
    double* Bs = As + DB * NS_LD;                 // [128][NS_LD]  L(base + 32 jb + j, kb + k)
    double* dneg = Bs + DB * NS_LD;
    double* Lp = a.L + d.lp_off;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, q = lane & 3;
    for (int e = tid; e < DB * NS_T; e += 256) {
        const int i = e & (NS_T - 1), k = e >> 5;
        cp_async8_zfill(As + k * NS_LD + i, Lp + (size_t)(kb + k) * f + base + NS_T * ib + i, true);
        cp_async8_zfill(Bs + k * NS_LD + i, Lp + (size_t)(kb + k) * f + base + NS_T * jb + i, true);
    }
    cp_async_commit_group();
    if (tid < DB) dneg[tid] = -a.dvec[d.col0 + kb + tid];
    cp_async_wait_group_n<0>();
    __syncthreads();
    const int mb = (warp & 1) * 16, nb = (warp >> 1) * 8;              // warp tile: 16 rows (two m8 fragments) x 8 columns
    double c[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
    double cold[2][2];                                                 // the C entries this lane updates: loads in flight under the MMA loop
#pragma unroll
    for (int x = 0; x < 2; ++x)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int i = base + NS_T * ib + mb + 8 * x + g, j = base + NS_T * jb + nb + 2 * q + e;
            cold[x][e] = (i >= j) ? Lp[(size_t)j * f + i] : 0.0;
        }
#pragma unroll 8
    for (int k0 = 0; k0 < DB; k0 += 4) {
        const double sc = dneg[k0 + q];
        const double bf = Bs[(k0 + q) * NS_LD + nb + g];
#pragma unroll
        for (int x = 0; x < 2; ++x) {
            const double af = As[(k0 + q) * NS_LD + mb + 8 * x + g] * sc;
            asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                         : "+d"(c[x][0]), "+d"(c[x][1]) : "d"(af), "d"(bf));
        }
    }
#pragma unroll
    for (int x = 0; x < 2; ++x)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int i = base + NS_T * ib + mb + 8 * x + g, j = base + NS_T * jb + nb + 2 * q + e;
            if (i >= j) Lp[(size_t)j * f + i] = cold[x][e] + c[x][e];
        }
    trace_exit(a, 8 * (kb / DB) + TR_NEAR2);
}

// The inverse of a finished diagonal block as its own kernel (one CTA): the dense chain leaves it to the side branch, where it runs
// beside the next diagonal block instead of in front of the near-diagonal step (16k + 5k of the diagonal kernel's 81k cycles).
__global__ void __launch_bounds__(256, 1) k_big_inv128(FactorArgs a, const int32_t* __restrict__ list, int kb,
                                                       double* __restrict__ Linv, const int64_t* __restrict__ linv_off) {
    const int s = list[blockIdx.x];
    const FrontDesc d = a.desc[s];
    if (kb >= d.w) return;
    extern __shared__ __align__(16) unsigned char dsm_raw[];
    Diag128Smem& sm = *reinterpret_cast<Diag128Smem*>(dsm_raw);
    const int f = d.f, nb = min(DB, d.w - kb), tid = threadIdx.x;
    const double* Lp = a.L + d.lp_off;
    for (int e = tid; e < DB * DB; e += 256) {
        const int i = e & (DB - 1), j = e >> 7;
        const bool in = i < nb && j < nb && i > j;
        cp_async8_zfill(sm.Lc + j * DB_LDS + i, Lp + (size_t)(kb + (in ? j : 0)) * f + kb + (in ? i : 0), in);
    }
    cp_async_commit_group();
    cp_async_wait_group_n<0>();
    __syncthreads();
    trace_enter(a, 8 * (kb / DB) + TR_INV);
    diag128_invert_store(sm, tid, nb, Linv + linv_off[s] + (size_t)(kb / DB) * DB * DB);
    trace_exit(a, 8 * (kb / DB) + TR_INV);
}

// Near-diagonal trsm WITHOUT the inverse: the 128 rows right below a finished diagonal block by forward substitution against L11
// itself, one warp per row (16 CTAs x 8 rows).  Lane l holds the row's entries c = l + 32 j (cyclic, so the shrinking active part
// stays spread over the lanes); step k broadcasts x_k by shuffle and every lane applies it to its entries c > k with L11(c, k) read
// from shared memory (consecutive lanes, consecutive addresses).  Dependent chain per step: SHFL + DFMA; 128 steps.
constexpr size_t NV_SMEM = (size_t)DB * NT_LDB * sizeof(double);
__global__ void __launch_bounds__(256, 1) k_near_trsv(FactorArgs a, const int32_t* __restrict__ list, int kb) {
    pdl_sync();
    const int s = list[0];
    const FrontDesc d = a.desc[s];
    const int f = d.f;
    extern __shared__ __align__(16) double nv_sm[];
    double* Ls = nv_sm;                            // Ls[k*NT_LDB + c] = L11(c, k), c > k
    double* Lp = a.L + d.lp_off;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int row = kb + DB + blockIdx.x * NT_ROWS + warp;
    trace_enter(a, 8 * (kb / DB) + TR_NEAR1);
    for (int e = tid; e < DB * DB; e += 256) {
        const int c = e & (DB - 1), k = e >> 7;
        if (c > k) cp_async8_zfill(Ls + k * NT_LDB + c, Lp + (size_t)(kb + k) * f + kb + c, true);
    }
    cp_async_commit_group();
    double x[4], dinv[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        x[j] = Lp[(size_t)(kb + lane + 32 * j) * f + row];
        dinv[j] = 1.0 / a.dvec[d.col0 + kb + lane + 32 * j];
    }
    cp_async_wait_group_n<0>();
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 4; ++j) {
#pragma unroll 8
        for (int o = 0; o < 32; ++o) {
            const int k = 32 * j + o;
            const double xk = __shfl_sync(0xffffffffu, x[j], o);
            const double* lk = Ls + k * NT_LDB + lane;
            if (lane > o) x[j] = fma(-xk, lk[32 * j], x[j]);
#pragma unroll
            for (int jj = j + 1; jj < 4; ++jj) x[jj] = fma(-xk, lk[32 * jj], x[jj]);
        }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) Lp[(size_t)(kb + lane + 32 * j) * f + row] = x[j] * dinv[j];
    trace_exit(a, 8 * (kb / DB) + TR_NEAR1);
}

}  // namespace b2
