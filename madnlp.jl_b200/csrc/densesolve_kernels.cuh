// Dense triangular solves  x <- (L D L')^{-1} x  in ONE launch: a dataflow over the 128-wide block rows of the factor.
//
// The launch-per-block sweeps (bigsolve_kernels.cuh) cost 2 * N/128 dependent launches (64 at N = 4096: 0.59 ms for a job whose
// HBM time is 20 us).  Here CTA k OWNS block row k of the forward sweep and block column k of the backward sweep:
//
//   forward :  t_k = b_k - sum_{c<k} L(k,c) y_c   accumulated as the y_c become available,  y_k = Linv_k t_k
//   diagonal:  z_k = y_k ./ d_k
//   backward:  s_k = z_k - sum_{c>k} L(c,k)' x_c  accumulated as the x_c become available,  x_k = Linv_k' s_k
//
// Hand-off between CTAs goes through two small global vectors (ybuf, xbuf) whose entries start as a SENTINEL bit pattern
// (all ones: a NaN no arithmetic produces) -- a consumer polls the 128 values themselves, so a block costs ONE L2 round trip
// on the critical path instead of flag + data, and needs no fence (8-byte stores are single-copy atomic).  The factor block a
// CTA needs next is loaded into registers BEFORE it polls, so the chain per block is: poll -> 16 FMAs + shared-memory reduction
// (off-diagonal block) -> 16 FMAs + reduction (inverted diagonal block) -> 128 stores.  Every CTA of the grid must be
// resident (grid = N/128 <= number of SMs, 1024 threads each); polls are bounded and report through `err`.
// Deterministic: fixed summation order, no atomics.
#pragma once
#include "bigsolve_kernels.cuh"

namespace b2 {

constexpr unsigned long long DS_SENTINEL = 0xFFFFFFFFFFFFFFFFull;
constexpr int DS_NT = 1024;

__device__ __forceinline__ double ds_poll(const double* p, int* err) {
    unsigned long long v = DS_SENTINEL;
    unsigned it = 0;
    do {
        asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
        if (v != DS_SENTINEL) break;
    } while (++it < (1u << 22));
    if (v == DS_SENTINEL) { atomicExch(err, 1); return 0.0; }
    return __longlong_as_double((long long)v);
}

// L: N x N column-major factor (unit lower, D on the diagonal), Linv: inverted 128 x 128 diagonal blocks (ld 128),
// dvec: D, x: right-hand side in / solution out, ybuf/xbuf: [nblk*128] hand-off vectors preset to the sentinel.
// Registers hold ONE 128 x 128 block of L (16 doubles per thread, 1024 threads); its load is issued BEFORE the poll of the
// vector it multiplies, so on the critical path (the newest y_c / x_c) the block is already there.  The CTA's own inverted
// diagonal block sits in shared memory (cp.async at kernel start, padded rows: both the plain and the transposed apply are
// bank-conflict free).
// PIV: the factor of a Bunch-Kaufman factorisation (bkpivot_kernels.cuh), P A P' = L_bd Lambda L_bd' with L21' = L21 Q_bd.  Block k
// loads b through perm, publishes y~_k = Q_k' y_k (what the stored L' multiplies), divides by Lambda, rotates the accumulated
// z~_k - sum L'^T x_c by Q_k before Linv_k', and stores x through perm.  Everything stays inside the CTA that owns block k.
constexpr int DS_LDI = BS + 1;
constexpr size_t DS_SMEM = (size_t)(BS * DS_LDI + 2 * BS + 2 * 8 * BS + BS) * sizeof(double);

template <bool PIV>
__global__ void __launch_bounds__(DS_NT, 1) k_dense_solve_flow(int N, const double* __restrict__ L, const double* __restrict__ Linv,
                                                              const double* __restrict__ dvec, double* __restrict__ x,
                                                              double* ybuf, double* xbuf, int* err, const int32_t* __restrict__ perm,
                                                              const int8_t* __restrict__ pkind, const double* __restrict__ rot) {
    extern __shared__ __align__(16) double ds_sm[];
    double* Ls = ds_sm;                                   // [BS][DS_LDI]: Ls[c*DS_LDI + r] = Linv_k(r, c)
    double (*vec)[BS] = (double (*)[BS])(Ls + BS * DS_LDI);                  // [2][BS] the block vector being applied
    double (*part)[8][BS] = (double (*)[8][BS])(Ls + BS * DS_LDI + 2 * BS);  // [2][8][BS] partial sums of the 8 groups
    double* tk = Ls + BS * DS_LDI + 2 * BS + 2 * 8 * BS;                     // [BS]
    const int k = blockIdx.x, kb = k * BS;
    const int nblk = gridDim.x;
    const int nb = min(BS, N - kb);
    const int tid = threadIdx.x, r = tid & (BS - 1), g = tid >> 7;           // r: row (fwd) / column (bwd) inside the block
    {
        const double* Li = Linv + (size_t)k * BS * BS;
        for (int e = tid; e < BS * BS; e += DS_NT) cp_async8(Ls + (e >> 7) * DS_LDI + (e & (BS - 1)), Li + e);
        asm volatile("cp.async.commit_group;" ::: "memory");
    }
    // ---------------- forward
    const int xr = (PIV && r < nb) ? perm[kb + r] : kb + r;                  // row of x behind row kb + r of the (permuted) system
    double t = (g == 0 && r < nb) ? x[xr] : 0.0;                             // group 0 carries the accumulator
    double v[16];
    for (int c = 0; c < k; ++c) {
        {                                                                     // L(kb + r, c*BS + g*16 + q), issued before the poll
            const double* p = L + (size_t)(c * BS + g * 16) * N + kb + min(r, nb - 1);
#pragma unroll
            for (int q = 0; q < 16; ++q) v[q] = (r < nb) ? p[(size_t)q * N] : 0.0;
        }
        const int b = c & 1;
        if (tid < BS) vec[b][tid] = ds_poll(ybuf + (size_t)c * BS + tid, err);
        __syncthreads();
        double acc = 0.0;
#pragma unroll
        for (int q = 0; q < 16; ++q) acc = fma(v[q], vec[b][g * 16 + q], acc);
        part[b][g][r] = acc;
        __syncthreads();
        if (g == 0) {
            double sum = 0.0;
#pragma unroll
            for (int u = 0; u < 8; ++u) sum += part[b][u][r];
            t -= sum;
        }
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    if (g == 0) tk[r] = t;
    __syncthreads();
    {                                                                         // y_k = Linv_k t_k   (Linv(r, c) = 0 for c > r)
        double acc = 0.0;
#pragma unroll
        for (int q = 0; q < 16; ++q) { const int c = g * 16 + q; acc = fma((c <= r) ? Ls[c * DS_LDI + r] : 0.0, tk[c], acc); }
        part[0][g][r] = acc;
    }
    __syncthreads();
    double yk = 0.0;
    if (g == 0) {
#pragma unroll
        for (int u = 0; u < 8; ++u) yk += part[0][u][r];
        if (r >= nb) yk = 0.0;
    }
    // pair rotation of block k at row r: kd = B2_PIVOT_KIND_*, (cs, sn) of its pair
    int kd = B2_PIVOT_KIND_1X1;
    double cs = 1.0, sn = 0.0;
    if (PIV) {
        if (g == 0 && r < nb) {
            kd = pkind[kb + r];
            if (kd == B2_PIVOT_KIND_2X2_FIRST) { cs = rot[kb + r]; sn = rot[kb + r + 1]; }
            else if (kd == B2_PIVOT_KIND_2X2_SECOND) { cs = rot[kb + r - 1]; sn = rot[kb + r]; }
            tk[r] = yk;
        }
        __syncthreads();
        if (kd == B2_PIVOT_KIND_2X2_FIRST) yk = cs * yk - sn * tk[r + 1];         // y~ = Q' y
        else if (kd == B2_PIVOT_KIND_2X2_SECOND) yk = sn * tk[r - 1] + cs * yk;
    }
    if (g == 0) ybuf[(size_t)k * BS + r] = yk;                                // publish y_k (consumers: the block rows below)
    // ---------------- diagonal + backward
    // s_k(j) -= sum_i L(cb + i, kb + j) x_c(i): a warp owns 4 columns j, its lanes stride the rows i (each load instruction reads
    // 32 consecutive rows of one column: coalesced), column sums meet through shuffles; `sacc` lives in the threads tid < BS
    double s = (g == 0 && r < nb) ? yk / dvec[kb + r] : 0.0;
    const int warp = tid >> 5, lane = tid & 31;
    for (int c = nblk - 1; c > k; --c) {
        const int cb = c * BS, ncb = min(BS, N - cb);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int j = warp * 4 + q;
            const double* p = L + (size_t)(kb + min(j, nb - 1)) * N + cb;
#pragma unroll
            for (int u = 0; u < 4; ++u) v[q * 4 + u] = (j < nb && lane + 32 * u < ncb) ? p[lane + 32 * u] : 0.0;
        }
        const int b = c & 1;
        if (tid < BS) vec[b][tid] = ds_poll(xbuf + (size_t)c * BS + tid, err);
        __syncthreads();
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            double acc = 0.0;
#pragma unroll
            for (int u = 0; u < 4; ++u) acc = fma(v[q * 4 + u], vec[b][lane + 32 * u], acc);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
            if (lane == 0) part[b][0][warp * 4 + q] = acc;
        }
        __syncthreads();
        if (g == 0) s -= part[b][0][r];
    }
    __syncthreads();
    if (g == 0) tk[r] = s;
    __syncthreads();
    const double* sv = tk;
    if (PIV) {                                                                // s = Q s~  (vec is free: the last poll has been consumed)
        if (g == 0) {
            double sr = s;
            if (kd == B2_PIVOT_KIND_2X2_FIRST) sr = cs * s + sn * tk[r + 1];
            else if (kd == B2_PIVOT_KIND_2X2_SECOND) sr = cs * s - sn * tk[r - 1];
            vec[0][r] = sr;
        }
        __syncthreads();
        sv = vec[0];
    }
    {                                                                         // x_k = Linv_k' s_k : sum_{i >= r} Linv(i, r) s_i
        double acc = 0.0;
#pragma unroll
        for (int q = 0; q < 16; ++q) { const int i = g * 16 + q; acc = fma((i >= r) ? Ls[r * DS_LDI + i] : 0.0, sv[i], acc); }
        part[1][g][r] = acc;
    }
    __syncthreads();
    if (g == 0) {
        double xk = 0.0;
#pragma unroll
        for (int u = 0; u < 8; ++u) xk += part[1][u][r];
        if (r >= nb) xk = 0.0;
        xbuf[(size_t)k * BS + r] = xk;                                        // publish x_k (consumers: the block columns before)
        if (r < nb) x[xr] = xk;
    }
}

}  // namespace b2
