// Device kernels of the supernodal multifrontal LDL^T (numeric phase).
//
// Data model (see analysis.hpp): one dense front per supernode, order f = w + r.
//   factor panel   L + lp_off : f x w column-major (ld = f).  On exit the strict lower part holds the unit-lower
//                               factor (L11 over L21), the diagonal holds D, the strict upper part of the w x w block
//                               holds U = D*L' (scratch).
//   update block   ws + cb_off: r x r column-major (ld = r), lower triangle = Schur complement passed to the parent.
// Fronts are processed level by level (children strictly below parents); inside a level every front is
// independent.  Extend-add is a PULL by the parent over its children in ascending child id, so the summation
// order -- and therefore every bit of the factor -- is deterministic.
//
// Three execution classes per level:
//   S/M  whole front resident in shared memory, one CTA per front (k_front_smem)   -- f <= small_front_max
//   B    front in HBM, blocked right-looking LDL^T across many CTAs (k_big_*)      -- tensor-pipe (DMMA) update
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace b2 {

struct FrontDesc {
    int32_t col0, w, f, nchild;
    int32_t child_off, amap_cnt;
    int64_t rows_off, lp_off, cb_off, rel_off, amap_off;
};
static_assert(sizeof(FrontDesc) == 64, "FrontDesc must be 64 bytes");

struct FactorArgs {
    const FrontDesc* desc;
    const int32_t* child_idx;
    const int32_t* rel;
    const int32_t* amap_src;
    const int32_t* amap_dst;
    const double* A;      // caller's CSC values (aliased)
    double* L;            // factor panels
    double* Lt;           // row-major copies of the warp-class panels (backward solve), same offsets
    double* ws;           // update blocks
    double* dvec;         // D, permuted order
    int32_t* counters;    // [0] = #negative pivots, [1] = #perturbed pivots
    double eps;
    unsigned long long* trace = nullptr;   // debug (B2_DENSE_TRACE): [slot][2] = first entry / last exit of a launch, %globaltimer ns
    unsigned long long* ftrace = nullptr;  // debug (B2_SPARSE_TRACE): [supernode][3] = team starts / children assembled / front finished
    // Bunch-Kaufman pivoting of the dense solver (bkpivot_kernels.cuh); all nullptr = static pivoting.  Per pivot (front order):
    // perm[kb + i] = row of A that became row kb + i (global index), pkind = B2_PIVOT_KIND_*, rot = (cos, sin) over a 2 x 2 pair
    int32_t* perm = nullptr;
    int8_t* pkind = nullptr;
    double* rot = nullptr;
};

// Timeline stamps of the dense look-ahead schedule (b2d_debug_trace): slot = 8 * block column + kernel kind
enum { TR_DIAG = 0, TR_NEAR1 = 1, TR_NEAR2 = 2, TR_TRSM = 3, TR_COL = 4, TR_BULK = 5, TR_INV = 6, TR_BK = 7 };
__device__ __forceinline__ unsigned long long global_ns() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
__device__ __forceinline__ void trace_enter(const FactorArgs& a, int slot) {
    if (a.trace && threadIdx.x == 0) atomicMin(a.trace + 2 * slot, global_ns());
}
__device__ __forceinline__ void trace_exit(const FactorArgs& a, int slot) {
    if (a.trace) { __syncthreads(); if (threadIdx.x == 0) atomicMax(a.trace + 2 * slot + 1, global_ns()); }
}

// ----------------------------------------------------------------------------------------------------------
// S/M class: fused assemble + factor + store with the whole front in shared memory.
// ----------------------------------------------------------------------------------------------------------
template <int NT>
__global__ void __launch_bounds__(NT) k_front_smem(FactorArgs a, const int32_t* __restrict__ list) {
    extern __shared__ double F[];
    const int tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;
    constexpr int NW = NT / 32;
    const int s = list[blockIdx.x];
    const FrontDesc d = a.desc[s];
    const int f = d.f, w = d.w, r = f - w;
    const int ff = f * f;

    for (int i = tid; i < ff; i += NT) F[i] = 0.0;
    __syncthreads();
    // original matrix entries (each lands in a distinct slot of the panel part)
    {
        const int32_t* src = a.amap_src + d.amap_off;
        const int32_t* dst = a.amap_dst + d.amap_off;
        for (int t = tid; t < d.amap_cnt; t += NT) F[dst[t]] = __ldg(a.A + src[t]);
    }
    __syncthreads();
    // extend-add of the children's update blocks, in ascending child order
    for (int c = 0; c < d.nchild; ++c) {
        const int cs = a.child_idx[d.child_off + c];
        const FrontDesc dc = a.desc[cs];
        const int rc = dc.f - dc.w;
        const double* CB = a.ws + dc.cb_off;
        const int32_t* rl = a.rel + dc.rel_off;
        for (int j = warp; j < rc; j += NW) {
            const int pj = rl[j] * f;
            const double* col = CB + (size_t)j * rc;
            for (int i = j + lane; i < rc; i += 32) F[rl[i] + pj] += col[i];
        }
        __syncthreads();
    }

    // ---- factor the w pivot columns (right-looking inside the panel)
    int nneg = 0, npert = 0;
    for (int k = 0; k < w; ++k) {
        __syncthreads();                        // updates of the previous pivot are complete
        double dk = F[k + k * f];
        bool pert = false;
        if (!(fabs(dk) >= a.eps)) {            // also catches NaN
            dk = (dk < 0.0) ? -a.eps : a.eps;
            pert = true;
            if (tid == 0) ++npert;
        } else if (dk < 0.0 && tid == 0) ++nneg;
        const double dinv = 1.0 / dk;
        for (int i = k + 1 + tid; i < f; i += NT) {
            const double u = F[i + k * f];
            F[k + i * f] = u;                   // U(k,i) = D*L' kept in the (free) upper triangle
            F[i + k * f] = u * dinv;
        }
        __syncthreads();                        // column k scaled, row k of U written
        if (pert && tid == 0) F[k + k * f] = dk;
        // update the remaining panel columns j in (k, w); the update block is done once below
        for (int j = k + 1 + warp; j < w; j += NW) {
            const double ukj = F[k + j * f];
            for (int i = j + lane; i < f; i += 32) F[i + j * f] -= F[i + k * f] * ukj;
        }
    }
    __syncthreads();
    // ---- Schur complement: C(i,j) -= sum_k L(i,k) * U(k,j),  i >= j >= w, 4x4 register tiles
    if (r > 0 && w > 0) {
        const int nt = (r + 3) >> 2;
        const int ntiles = nt * (nt + 1) / 2;
        for (int t = tid; t < ntiles; t += NT) {
            // lower-triangular tile index t -> (ti, tj), ti >= tj
            int ti = (int)((sqrtf(8.0f * (float)t + 1.0f) - 1.0f) * 0.5f);
            while (ti * (ti + 1) / 2 > t) --ti;
            while ((ti + 1) * (ti + 2) / 2 <= t) ++ti;
            const int tj = t - ti * (ti + 1) / 2;
            const int i0 = w + 4 * ti, j0 = w + 4 * tj;
            double acc[4][4];
#pragma unroll
            for (int x = 0; x < 4; ++x)
#pragma unroll
                for (int y = 0; y < 4; ++y) acc[x][y] = 0.0;
            for (int k = 0; k < w; ++k) {
                double av[4], bv[4];
#pragma unroll
                for (int x = 0; x < 4; ++x) av[x] = (i0 + x < f) ? F[i0 + x + k * f] : 0.0;
#pragma unroll
                for (int y = 0; y < 4; ++y) bv[y] = (j0 + y < f) ? F[k + (j0 + y) * f] : 0.0;
#pragma unroll
                for (int x = 0; x < 4; ++x)
#pragma unroll
                    for (int y = 0; y < 4; ++y) acc[x][y] = fma(av[x], bv[y], acc[x][y]);
            }
#pragma unroll
            for (int y = 0; y < 4; ++y)
#pragma unroll
                for (int x = 0; x < 4; ++x) {
                    const int i = i0 + x, j = j0 + y;
                    if (i < f && j < f && i >= j) F[i + j * f] -= acc[x][y];
                }
        }
    }
    __syncthreads();
    // ---- store: panel (first w columns, contiguous), D, update block
    {
        double* Lp = a.L + d.lp_off;
        const int pw = f * w;
        for (int i = tid; i < pw; i += NT) Lp[i] = F[i];
        for (int k = tid; k < w; k += NT) a.dvec[d.col0 + k] = F[k + k * f];
        double* CB = a.ws + d.cb_off;
        for (int j = warp; j < r; j += NW) {
            const double* src = F + (w + j) * f + w;
            double* dst = CB + (size_t)j * r;
            for (int i = j + lane; i < r; i += 32) dst[i] = src[i];
        }
    }
    if (tid == 0) {
        if (nneg) atomicAdd(a.counters + 0, nneg);
        if (npert) atomicAdd(a.counters + 1, npert);
    }
}

// ----------------------------------------------------------------------------------------------------------
// B class: fronts that do not fit in shared memory live in HBM:  panel at L+lp_off (ld f), update block at
// ws+cb_off (ld r).  Element (i,j), i>=j, of the front is addressed by front_ptr().
// ----------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double* front_ptr(const FactorArgs& a, const FrontDesc& d, int i, int j) {
    const int w = d.w;
    return (j < w) ? a.L + d.lp_off + (size_t)j * d.f + i
                   : a.ws + d.cb_off + (size_t)(j - w) * (d.f - w) + (i - w);
}

// zero panel + update block of every big front in `list` (grid.y = front)
__global__ void k_big_zero(FactorArgs a, const int32_t* __restrict__ list) {
    const FrontDesc d = a.desc[list[blockIdx.y]];
    const size_t np = (size_t)d.f * d.w, r = d.f - d.w, nc = r * r;
    double* Lp = a.L + d.lp_off;
    double* CB = a.ws + d.cb_off;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < np + nc; i += (size_t)gridDim.x * blockDim.x) {
        if (i < np) Lp[i] = 0.0; else CB[i - np] = 0.0;
    }
}

__global__ void k_big_scatter_A(FactorArgs a, const int32_t* __restrict__ list) {
    const FrontDesc d = a.desc[list[blockIdx.y]];
    const int32_t* src = a.amap_src + d.amap_off;
    const int32_t* dst = a.amap_dst + d.amap_off;
    double* Lp = a.L + d.lp_off;
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < d.amap_cnt; t += gridDim.x * blockDim.x)
        Lp[dst[t]] = __ldg(a.A + src[t]);
}

// extend-add of the `rank`-th child of every big front in `list` (plain +=: one contribution per element per launch)
__global__ void k_big_extend_add(FactorArgs a, const int32_t* __restrict__ list, int rank) {
    const FrontDesc d = a.desc[list[blockIdx.y]];
    if (rank >= d.nchild) return;
    const FrontDesc dc = a.desc[a.child_idx[d.child_off + rank]];
    const int rc = dc.f - dc.w;
    const double* CB = a.ws + dc.cb_off;
    const int32_t* rl = a.rel + dc.rel_off;
    const int lane = threadIdx.x & 31;
    const int wglob = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    const int r = d.f - d.w;
    for (int j = wglob; j < rc; j += nwarps) {
        const int pj = rl[j];
        const double* __restrict__ col = CB + (size_t)j * rc;
        // destination column of the parent front (panel or update block), indexed by the parent-local row
        double* dst = (pj < d.w) ? a.L + d.lp_off + (size_t)pj * d.f : a.ws + d.cb_off + (size_t)(pj - d.w) * r - d.w;
        for (int i = j + lane; i < rc; i += 128) {          // 4 independent read-modify-writes in flight per lane
            int ri[4]; double v[4], t[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int ii = i + 32 * u;
                const bool ok = ii < rc;
                ri[u] = ok ? rl[ii] : -1;
                v[u] = ok ? col[ii] : 0.0;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) t[u] = (ri[u] >= 0) ? dst[ri[u]] : 0.0;
#pragma unroll
            for (int u = 0; u < 4; ++u) if (ri[u] >= 0) dst[ri[u]] = t[u] + v[u];
        }
    }
}

__device__ __forceinline__ double fast_rcp_d(double x) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    r = fma(r, fma(-x, r, 1.0), r);
    r = fma(r, fma(-x, r, 1.0), r);
    return r;
}

// ----------------------------------------------------------------------------------------------------------
// Trailing update of the blocked factorisation (> 95 % of the flops of a big front; see bigfactor_kernels.cuh):
//   C(i,j) -= sum_{k in [kb0, kb0+kcount)} L(i,k) d_k L(j,k),  i >= j, jlo <= j < jhi
// (jlo = kb0 + min(jlo_rel, kcount) when clip_jlo, else kb0 + jlo_rel; jhi = min(f, kb0 + jhi_rel))
// 128 x 64 tiles, 8 warps as 4 x 2 (32 x 32 per warp = 4 x 4 m8n8k4 DMMA fragments).  Both operands are raw panel
// columns of L streamed by cp.async through a GU_STAGES-deep ring of K = 16 slices (no register staging, loads stay in
// flight under the tensor pipe); the -d_k scaling is applied to the A fragments in registers (4 DMUL per 16 DMMA), and
// the epilogue adds the (negative) accumulators to C.
// ----------------------------------------------------------------------------------------------------------
constexpr int GU_M = 128, GU_N = 64, GU_K = 16, GU_STAGES = 4;
constexpr int GU_LDA = GU_M + 4, GU_LDB = GU_N + 4, GU_LDC = GU_M + 2;
constexpr size_t GU_SMEM = (size_t)(GU_STAGES * GU_K * (GU_LDA + GU_LDB) + 128) * sizeof(double);

__device__ __forceinline__ void cp_async8_zfill(void* smem_dst, const void* gsrc, bool valid) {
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
    const int sz = valid ? 8 : 0;
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(sa), "l"(gsrc), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_commit_group() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait_group_n() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// one 128 x 64 tile (bx, by) of the update; `gu_sm` is the CTA's dynamic shared memory (GU_SMEM bytes).  Returns without work for
// tiles above the diagonal / outside the column range.  All threads of the CTA must call it together.
template <bool NAMED>
__device__ __forceinline__ void gu_sync() {           // NAMED: only the 256 consumer threads of a 288-thread CTA (barrier id 1)
    if (NAMED) asm volatile("bar.sync 1, 256;" ::: "memory");
    else __syncthreads();
}
template <bool NAMED = false>
__device__ __forceinline__ void big_update_tile(const FactorArgs& a, const FrontDesc& d, int kb0, int kmax, int jlo_rel, int jhi_rel, int clip_jlo,
                                                int bx, int by, double* gu_sm) {
    if (kb0 >= d.w) return;
    const int f = d.f;
    const int kcount = min(kmax, d.w - kb0);
    const int jlo = kb0 + (clip_jlo ? min(jlo_rel, kcount) : jlo_rel);
    const int jhi = min(f, kb0 + jhi_rel);
    const int i0 = jlo + bx * GU_M, j0 = jlo + by * GU_N;
    if (j0 > i0 + GU_M - 1 || i0 >= f || j0 >= jhi) return;          // tile above the diagonal / outside the front
    double* As = gu_sm;                                               // [stage][k][GU_LDA]
    double* Bs = gu_sm + GU_STAGES * GU_K * GU_LDA;                   // [stage][k][GU_LDB]
    double* dneg = Bs + GU_STAGES * GU_K * GU_LDB;                    // -d_k, k < kcount (<= 128)
    const double* Lp = a.L + d.lp_off;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, q = lane & 3;
    const int wi = (warp & 3) * 32, wj = (warp >> 2) * 32;
    if (tid < 128) dneg[tid] = (tid < kcount) ? -Lp[(size_t)(kb0 + tid) * f + kb0 + tid] : 0.0;
    const int nchunk = (kcount + GU_K - 1) / GU_K;
    const int la_i = tid & (GU_M - 1), la_k = tid >> 7;               // A loader: 2 k-rows per pass, 8 passes
    const int lb_j = tid & (GU_N - 1), lb_k = tid >> 6;               // B loader: 4 k-rows per pass, 4 passes
    const bool a_ok = i0 + la_i < f, b_ok = j0 + lb_j < f;
    const double* a_src = Lp + (size_t)kb0 * f + (a_ok ? i0 + la_i : 0);
    const double* b_src = Lp + (size_t)kb0 * f + (b_ok ? j0 + lb_j : 0);
    auto issue = [&](int ch) {
        const int st = ch % GU_STAGES;
        double* Ad = As + (size_t)st * GU_K * GU_LDA + la_i;
        double* Bd = Bs + (size_t)st * GU_K * GU_LDB + lb_j;
#pragma unroll
        for (int p = 0; p < GU_K / 2; ++p) {
            const int k = ch * GU_K + la_k + 2 * p;
            const bool ok = a_ok && k < kcount;
            cp_async8_zfill(Ad + (la_k + 2 * p) * GU_LDA, a_src + (size_t)(ok ? k : 0) * f, ok);
        }
#pragma unroll
        for (int p = 0; p < GU_K / 4; ++p) {
            const int k = ch * GU_K + lb_k + 4 * p;
            const bool ok = b_ok && k < kcount;
            cp_async8_zfill(Bd + (lb_k + 4 * p) * GU_LDB, b_src + (size_t)(ok ? k : 0) * f, ok);
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
        gu_sync<NAMED>();                                              // slice ch landed; slice ch-1 fully consumed
        if (ch + GU_STAGES - 1 < nchunk) issue(ch + GU_STAGES - 1);
        cp_async_commit_group();
        const double* Ab = As + (size_t)(ch % GU_STAGES) * GU_K * GU_LDA;
        const double* Bb = Bs + (size_t)(ch % GU_STAGES) * GU_K * GU_LDB;
#pragma unroll
        for (int k0 = 0; k0 < GU_K; k0 += 4) {
            const double sc = dneg[ch * GU_K + k0 + q];
            double af[4], bf[4];
#pragma unroll
            for (int x = 0; x < 4; ++x) af[x] = Ab[(k0 + q) * GU_LDA + wi + 8 * x + g] * sc;
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
    // epilogue: accumulators -> shared memory (column-major tile), then a coalesced read-modify-write of C with all of
    // a thread's loads in flight at once (the fragment layout would make it 32 dependent 8-byte round trips per thread)
    cp_async_wait_group_n<0>();
    gu_sync<NAMED>();
    double* Cs = gu_sm;                                               // [GU_N][GU_LDC]
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y)
#pragma unroll
            for (int e = 0; e < 2; ++e) Cs[(wj + 8 * y + 2 * q + e) * GU_LDC + wi + 8 * x + g] = c[x][y][e];
    gu_sync<NAMED>();
    const int r = f - d.w;
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        double t[4][4];
        double* colp[4];
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) {
            const int jj = warp * 8 + half * 4 + cc, j = j0 + jj;
            colp[cc] = (j < d.w) ? a.L + d.lp_off + (size_t)j * f : a.ws + d.cb_off + (size_t)(j - d.w) * r - d.w;
#pragma unroll
            for (int rr = 0; rr < 4; ++rr) {
                const int i = i0 + lane + 32 * rr;
                t[cc][rr] = (j < jhi && i < f && i >= j) ? colp[cc][i] : 0.0;
            }
        }
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) {
            const int jj = warp * 8 + half * 4 + cc, j = j0 + jj;
#pragma unroll
            for (int rr = 0; rr < 4; ++rr) {
                const int i = i0 + lane + 32 * rr;
                if (j < jhi && i < f && i >= j) colp[cc][i] = t[cc][rr] + Cs[jj * GU_LDC + lane + 32 * rr];
            }
        }
    }
}


__global__ void __launch_bounds__(256, 2) k_big_update_pipe(FactorArgs a, const int32_t* __restrict__ list, int kb0, int kmax, int jlo_rel,
                                                            int jhi_rel, int clip_jlo) {
    extern __shared__ __align__(16) double gu_sm[];
    const FrontDesc d = a.desc[list[blockIdx.z]];
    big_update_tile(a, d, kb0, kmax, jlo_rel, jhi_rel, clip_jlo, blockIdx.x, blockIdx.y, gu_sm);
}

// the same tiles from row block `bx0` on (side branch of the dense look-ahead schedule: the first row block is done by k_near_syrk)
__global__ void __launch_bounds__(256, 2) k_big_update_rows(FactorArgs a, const int32_t* __restrict__ list, int kb0, int kmax, int jlo_rel,
                                                            int jhi_rel, int clip_jlo, int bx0) {
    extern __shared__ __align__(16) double gu_sm[];
    const FrontDesc d = a.desc[list[blockIdx.z]];
    trace_enter(a, 8 * (kb0 / 128) + TR_COL);
    big_update_tile(a, d, kb0, kmax, jlo_rel, jhi_rel, clip_jlo, blockIdx.x + bx0, blockIdx.y, gu_sm);
    trace_exit(a, 8 * (kb0 / 128) + TR_COL);
}

// The same update as a PERSISTENT kernel with a dynamic tile queue, for the look-ahead schedule of the dense factorisation:
// CTAs that land on the first `n_reserved` SMs exit at once, so those SMs stay free for the next panel's diagonal-block kernel
// (one CTA that needs a whole SM) while this kernel works through the trailing update on all the others.  Tiles are handed out
// by an atomic counter (`*tile_counter`, zeroed by the host before the launch), so it does not matter which CTAs left.
__device__ __forceinline__ unsigned smid() { unsigned r; asm volatile("mov.u32 %0, %%smid;" : "=r"(r)); return r; }
__global__ void __launch_bounds__(256, 2) k_big_update_dyn(FactorArgs a, const int32_t* __restrict__ list, int kb0, int kmax, int jlo_rel,
                                                           int jhi_rel, int clip_jlo, int nbx, int nby, int* tile_counter, int n_reserved) {
    extern __shared__ __align__(16) double gu_sm[];
    __shared__ int t_sh;
    if ((int)smid() < n_reserved) return;
    const FrontDesc d = a.desc[list[0]];
    const int ntile = nbx * nby;
    trace_enter(a, 8 * (kb0 / 128) + TR_BULK);
    for (;;) {
        __syncthreads();                                 // (the previous tile's epilogue has finished with shared memory)
        if (threadIdx.x == 0) t_sh = atomicAdd(tile_counter, 1);
        __syncthreads();
        const int t = t_sh;
        if (t >= ntile) { trace_exit(a, 8 * (kb0 / 128) + TR_BULK); return; }
        big_update_tile(a, d, kb0, kmax, jlo_rel, jhi_rel, clip_jlo, t % nbx, t / nbx, gu_sm);
    }
}

// ----------------------------------------------------------------------------------------------------------
// The same 128 x 64 tile with operands staged by the TMA unit: 1-D bulk copies (cp.async.bulk.shared::cluster.global, one per
// K-row of each operand: 1 KB of A, 512 B of B) issued by a ninth, producer warp into the same 4-stage ring, completion counted in
// bytes on one mbarrier per stage ("full"); the eight consumer warps release a stage through a second mbarrier ("empty", one
// arrival per warp) instead of a CTA-wide barrier per K-slice, so no warp ever waits for its siblings inside the K loop and no
// consumer thread issues copies (12 cp.async per thread and slice before).  Bulk copies move multiples of 16 bytes between
// 16-byte aligned addresses, but a K-row of a front starts at element lp_off + k f + i0 of the factor array -- odd for every
// other row when f is odd.  Such a row is copied from the element BEFORE it (one extra pair at the end when needed), so its data
// sits one slot to the right in the shared-memory row (LDA has the room); since K-slices hold 16 rows and a lane always reads
// rows k = q (mod 4), that shift is a per-lane constant folded into the operand base pointers.  Requirement, checked per tile:
// whole K-slices (kcount % 16 == 0); other tiles run the cp.async version on the consumer threads.  `it` counts the K-slices this CTA has pushed through the
// ring since the barriers were initialised (stage = it % 4, phase parity = (it / 4) & 1); it is uniform over the CTA.
// ----------------------------------------------------------------------------------------------------------
constexpr int GU_NT_BULK = 288;
constexpr size_t GU_SMEM_BULK = GU_SMEM + 2 * GU_STAGES * sizeof(unsigned long long);
__device__ __forceinline__ unsigned gu_s32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void gu_mbar_init(unsigned long long* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(gu_s32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void gu_mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(gu_s32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void gu_mbar_arrive(unsigned long long* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(gu_s32(bar)) : "memory");
}
__device__ __forceinline__ void gu_mbar_wait(unsigned long long* bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "GU_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra GU_DONE;\n"
        "bra GU_WAIT;\n"
        "GU_DONE:\n"
        "}\n" ::"r"(gu_s32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void gu_bulk_g2s(void* smem_dst, const void* gsrc, unsigned bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(gu_s32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(gu_s32(bar)) : "memory");
}

// All 288 threads of the CTA call this together; the caller separates consecutive tiles by a CTA-wide barrier.
__device__ __forceinline__ void big_update_tile_bulk(const FactorArgs& a, const FrontDesc& d, int kb0, int kmax, int jlo_rel, int jhi_rel,
                                                     int clip_jlo, int bx, int by, double* gu_sm, unsigned& it) {
    if (kb0 >= d.w) return;
    const int f = d.f;
    const int kcount = min(kmax, d.w - kb0);
    const int jlo = kb0 + (clip_jlo ? min(jlo_rel, kcount) : jlo_rel);
    const int jhi = min(f, kb0 + jhi_rel);
    const int i0 = jlo + bx * GU_M, j0 = jlo + by * GU_N;
    if (j0 > i0 + GU_M - 1 || i0 >= f || j0 >= jhi) return;          // tile above the diagonal / outside the front
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const double* Lp = a.L + d.lp_off;
    const bool bulk_ok = (kcount & (GU_K - 1)) == 0 && (reinterpret_cast<size_t>(a.L) & 15) == 0;
    if (!bulk_ok) {                                                   // (uniform over the CTA)
        if (warp < 8) big_update_tile<true>(a, d, kb0, kmax, jlo_rel, jhi_rel, clip_jlo, bx, by, gu_sm);
        return;
    }
    double* As = gu_sm;                                               // [stage][k][GU_LDA]
    double* Bs = gu_sm + GU_STAGES * GU_K * GU_LDA;                   // [stage][k][GU_LDB]
    double* dneg = Bs + GU_STAGES * GU_K * GU_LDB;                    // -d_k
    unsigned long long* full = reinterpret_cast<unsigned long long*>(dneg + 128);
    unsigned long long* empty = full + GU_STAGES;
    const int nchunk = kcount / GU_K;
    const unsigned it0 = it;
    it += nchunk;
    if (warp == 8) {
        // ---- producer warp: lane l < 16 moves K-row l of both operands of a slice
        const int na = min(GU_M, f - i0), nb_ = min(GU_N, f - j0);
        for (int ch = 0; ch < nchunk; ++ch) {
            const unsigned g = it0 + ch, st = g % GU_STAGES;
            if (g >= GU_STAGES) gu_mbar_wait(&empty[st], ((g / GU_STAGES) - 1) & 1);   // every consumer warp has left the stage's previous slice
            // row `lane` of the slice: absolute element index of its first entry, rounded down to a 16-byte boundary
            const size_t eA = (size_t)d.lp_off + (size_t)(kb0 + ch * GU_K + (lane & (GU_K - 1))) * f + i0;
            const size_t eB = eA - i0 + j0;
            const unsigned pA = (unsigned)(eA & 1), pB = (unsigned)(eB & 1);
            const unsigned bytesA = 8u * ((na + pA + 1u) & ~1u), bytesB = 8u * ((nb_ + pB + 1u) & ~1u);
            const unsigned total = __reduce_add_sync(0xffffffffu, lane < GU_K ? bytesA + bytesB : 0u);
            if (lane == 0) gu_mbar_expect_tx(&full[st], total);
            __syncwarp();
            if (lane < GU_K) {
                gu_bulk_g2s(As + ((size_t)st * GU_K + lane) * GU_LDA, a.L + (eA - pA), bytesA, &full[st]);
                gu_bulk_g2s(Bs + ((size_t)st * GU_K + lane) * GU_LDB, a.L + (eB - pB), bytesB, &full[st]);
            }
        }
        return;
    }
    // ---- consumers
    const int g = lane >> 2, q = lane & 3;
    const int wi = (warp & 3) * 32, wj = (warp >> 2) * 32;
    if (tid < 128) dneg[tid] = (tid < kcount) ? -Lp[(size_t)(kb0 + tid) * f + kb0 + tid] : 0.0;
    gu_sync<true>();
    // this lane reads rows k = q (mod 4) only: their alignment shift (see the producer) is a constant of the lane
    const int shA = (int)(((size_t)d.lp_off + (size_t)(kb0 + q) * f + i0) & 1), shB = (int)(((size_t)d.lp_off + (size_t)(kb0 + q) * f + j0) & 1);
    double c[4][4][2];
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) c[x][y][0] = c[x][y][1] = 0.0;
    for (int ch = 0; ch < nchunk; ++ch) {
        const unsigned gi = it0 + ch, st = gi % GU_STAGES;
        gu_mbar_wait(&full[st], (gi / GU_STAGES) & 1);
        const double* Ab = As + (size_t)st * GU_K * GU_LDA + shA;
        const double* Bb = Bs + (size_t)st * GU_K * GU_LDB + shB;
#pragma unroll
        for (int k0 = 0; k0 < GU_K; k0 += 4) {
            const double sc = dneg[ch * GU_K + k0 + q];
            double af[4], bf[4];
#pragma unroll
            for (int x = 0; x < 4; ++x) af[x] = Ab[(k0 + q) * GU_LDA + wi + 8 * x + g] * sc;
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
        __syncwarp();
        if (lane == 0) gu_mbar_arrive(&empty[st]);
    }
    // epilogue (as in big_update_tile): every consumer has passed its last `full` wait, so all copies have landed; the producer
    // cannot touch the ring again before the caller's CTA-wide barrier
    gu_sync<true>();
    double* Cs = gu_sm;                                               // [GU_N][GU_LDC]
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y)
#pragma unroll
            for (int e = 0; e < 2; ++e) Cs[(wj + 8 * y + 2 * q + e) * GU_LDC + wi + 8 * x + g] = c[x][y][e];
    gu_sync<true>();
    const int r = f - d.w;
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        double t[4][4];
        double* colp[4];
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) {
            const int jj = warp * 8 + half * 4 + cc, j = j0 + jj;
            colp[cc] = (j < d.w) ? a.L + d.lp_off + (size_t)j * f : a.ws + d.cb_off + (size_t)(j - d.w) * r - d.w;
#pragma unroll
            for (int rr = 0; rr < 4; ++rr) {
                const int i = i0 + lane + 32 * rr;
                t[cc][rr] = (j < jhi && i < f && i >= j) ? colp[cc][i] : 0.0;
            }
        }
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) {
            const int jj = warp * 8 + half * 4 + cc, j = j0 + jj;
#pragma unroll
            for (int rr = 0; rr < 4; ++rr) {
                const int i = i0 + lane + 32 * rr;
                if (j < jhi && i < f && i >= j) colp[cc][i] = t[cc][rr] + Cs[jj * GU_LDC + lane + 32 * rr];
            }
        }
    }
}

__device__ __forceinline__ void gu_bulk_setup(double* gu_sm) {
    unsigned long long* full = reinterpret_cast<unsigned long long*>(gu_sm + GU_STAGES * GU_K * (GU_LDA + GU_LDB) + 128);
    if (threadIdx.x < GU_STAGES) {
        gu_mbar_init(&full[threadIdx.x], 1);
        gu_mbar_init(&full[GU_STAGES + threadIdx.x], 8);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();
}

// k_big_update_pipe / k_big_update_dyn with bulk-copy operand staging (288 threads: 8 consumer warps + 1 producer warp)
__global__ void __launch_bounds__(GU_NT_BULK, 2) k_big_update_pipe_bulk(FactorArgs a, const int32_t* __restrict__ list, int kb0, int kmax,
                                                                       int jlo_rel, int jhi_rel, int clip_jlo) {
    extern __shared__ __align__(16) double gu_sm[];
    const FrontDesc d = a.desc[list[blockIdx.z]];
    {   // CTAs of tiles above the diagonal / outside the front (about half of the rectangular grid) leave before any set-up
        if (kb0 >= d.w) return;
        const int kcount = min(kmax, d.w - kb0);
        const int jlo = kb0 + (clip_jlo ? min(jlo_rel, kcount) : jlo_rel);
        const int i0 = jlo + blockIdx.x * GU_M, j0 = jlo + blockIdx.y * GU_N;
        if (j0 > i0 + GU_M - 1 || i0 >= d.f || j0 >= min(d.f, kb0 + jhi_rel)) return;
    }
    gu_bulk_setup(gu_sm);
    unsigned it = 0;
    big_update_tile_bulk(a, d, kb0, kmax, jlo_rel, jhi_rel, clip_jlo, blockIdx.x, blockIdx.y, gu_sm, it);
}
__global__ void __launch_bounds__(GU_NT_BULK, 2) k_big_update_dyn_bulk(FactorArgs a, const int32_t* __restrict__ list, int kb0, int kmax,
                                                                      int jlo_rel, int jhi_rel, int clip_jlo, int nbx, int nby, int* tile_counter,
                                                                      int n_reserved) {
    extern __shared__ __align__(16) double gu_sm[];
    __shared__ int t_sh;
    if ((int)smid() < n_reserved) return;
    gu_bulk_setup(gu_sm);
    const FrontDesc d = a.desc[list[0]];
    const int ntile = nbx * nby;
    unsigned it = 0;
    trace_enter(a, 8 * (kb0 / 128) + TR_BULK);
    for (;;) {
        __syncthreads();                                 // (the previous tile's epilogue has finished with shared memory)
        if (threadIdx.x == 0) t_sh = atomicAdd(tile_counter, 1);
        __syncthreads();
        const int t = t_sh;
        if (t >= ntile) { trace_exit(a, 8 * (kb0 / 128) + TR_BULK); return; }
        big_update_tile_bulk(a, d, kb0, kmax, jlo_rel, jhi_rel, clip_jlo, t % nbx, t / nbx, gu_sm, it);
    }
}

}  // namespace b2
