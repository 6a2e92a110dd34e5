// b2_* sparse LDL^T solver: host driver (analysis -> device schedule -> CUDA-graph replay).
// C-ABI declared in include/b200kkt.h; replaces the AbstractLinearSolver back-end role of CUDSSSolver
// (lib/MadNLPGPU/ext/MadNLPGPUCUDAExt/cudss.jl:88-214) / Ma97Solver (lib/MadNLPHSL/src/ma97.jl:29-115).
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <stdexcept>
#include <array>
#include <vector>

#include "analysis.hpp"
#include "common.cuh"
#include "front_kernels.cuh"
#include "bigfactor_kernels.cuh"
#include "bkpivot_kernels.cuh"
#include "solve_kernels.cuh"
#include "warp_kernels.cuh"
#include "bigsolve_kernels.cuh"
#include "densesolve_kernels.cuh"

using namespace b2;

namespace {

struct WarpLaunch {          // one launch of the team-per-front kernels (offsets into d_sched)
    int n_cta = 0, cta_ptr_off = 0, stage_off_off = 0, stage_cnt_off = 0;
    int nw = 1;              // warps per team: 1 (order <= 32) or 2 (order <= 64)
    int maxf = 0;            // largest front in the launch (sizes the shared-memory assembly area)
};
struct LevelSched {
    WarpLaunch W, W2;                               // fronts of order <= 32 / <= 64
    int offM = 0, nM = 0, maxfM = 0;                // shared-memory CTA class
    int offB = 0, nB = 0, maxfB = 0, maxwB = 0, maxchildB = 0, maxamapB = 0, maxrB = 0;   // HBM-resident class
    // the first nLA fronts of the B list are factorised ONE AT A TIME with the three-branch look-ahead schedule (enqueue_front_lookahead);
    // la[i] = {w, f, offset of its tile counters}; maxfBr / maxwBr: maxima over the remaining (batched) fronts
    int nLA = 0, maxfBr = 0, maxwBr = 0;
    std::vector<std::array<int, 3>> la;
    int offC = 0, nC = 0, maxfC = 0, maxwC = 0;     // M and B fronts together, for the multi-CTA solve kernels
};
struct Phase {
    WarpLaunch fused;                               // bottom subtrees, one CTA each (n_cta == 0: none)
    WarpLaunch topfused;                            // the sparse top of the tree (levels with <= 4 fronts): ONE CTA, one stage per level
    std::vector<LevelSched> lev;
    // single-launch dependency-driven schedule (used instead of fused + levels when every front is team-class)
    int offAllC = 0, nAllC = 0, maxwAllC = 0;       // every M/B front of the phase (diagonal-block inversion)
    int dep_ngroup = 0, dep_type_off = 0, dep_ptr_off = 0, dep_tasks_off = 0, dep_maxf1 = 0, dep_maxf2 = 0;
    // hybrid sweeps (dep_schedule bit 2): the fused bottom subtrees by their staged kernel, every front above them as ONE flag-driven
    // launch (groups in level order of the upper tree); flags of the fused fronts are preset from d_flags_tpl
    int dep2_ngroup = 0, dep2_type_off = 0, dep2_ptr_off = 0, dep2_tasks_off = 0;
    cudaGraphExec_t g_factor = nullptr, g_fwd = nullptr, g_bwd = nullptr;
    int64_t n_factor_launches = 0, n_solve_launches = 0;
    int64_t n_fused_fronts = 0;
};

constexpr int W_MAX = 64;        // team-per-front classes: f <= 32 (one warp), f <= 64 (two warps)

}  // namespace

struct b2_solver {
    Symbolic S;
    b2_options opt;
    bool symbolic_only = false;
    const double* nzval_d = nullptr;
    int device = 0;
    // device copies of the symbolic structure
    DevBuf<FrontDesc> d_desc;
    DevBuf<int32_t> d_rows, d_child_idx, d_rel, d_amap_src, d_amap_dst, d_perm, d_sched;
    DevBuf<int64_t> d_cbv_off;
    DevBuf<uint8_t> d_mask_p;
    DevBuf<ChildRec> d_childrec;
    // numeric storage
    DevBuf<double> d_L, d_Lt, d_ws, d_dvec, d_xp, d_cbv;
    DevBuf<int32_t> d_counters;
    DevBuf<double> d_Linv, d_side;
    DevBuf<int64_t> d_linv_off;
    DevBuf<int32_t> d_flags, d_parent;   // dependency flags [3][nsuper], supernode parents
    DevBuf<int32_t> d_flags_tpl;         // [nsuper] 1 for fronts of the fused bottom subtrees (hybrid sweeps), else 0
    int32_t* h_counters = nullptr;   // pinned
    std::vector<int64_t> cbv_off;
    int64_t exch_cbv = 0;
    Phase phase[2];                  // 0 = local (owned subtrees), 1 = shared top tree
    cudaStream_t cap_stream = nullptr;
    cudaStream_t la_bulk = nullptr, la_side = nullptr;   // side branches of the look-ahead schedule of the largest fronts
    std::vector<cudaEvent_t> ev_pool;
    size_t ev_next = 0;
    DevBuf<unsigned long long> d_ftrace;                 // B2_SPARSE_TRACE=1: per-front stamps of the team-class factor kernels (b2_debug_trace)
    DevBuf<int32_t> d_tilecnt;                           // dynamic-tile counters, one per 128-column block of every look-ahead front
    bool factorized = false;
    int64_t last_perturbed = 0;
    std::vector<uint8_t> owned_mask;  // original numbering

    ~b2_solver() {
        for (auto& p : phase) {
            if (p.g_factor) cudaGraphExecDestroy(p.g_factor);
            if (p.g_fwd) cudaGraphExecDestroy(p.g_fwd);
            if (p.g_bwd) cudaGraphExecDestroy(p.g_bwd);
        }
        if (cap_stream) cudaStreamDestroy(cap_stream);
        if (la_bulk) cudaStreamDestroy(la_bulk);
        if (la_side) cudaStreamDestroy(la_side);
        for (auto e : ev_pool) cudaEventDestroy(e);
        if (h_counters) cudaFreeHost(h_counters);
    }
};

namespace {

// one outer step of every big front in `lb`: diagonal block (factor + inverse), rows below, trailing update
inline bool lookahead_bulk() {
    static const bool on = [] { const char* e = getenv("B2_UPDATE_BULK"); return !e || atoi(e) != 0; }();
    return on;
}
// (a.perm set: Bunch-Kaufman diagonal block and the pivoted trsm; the trailing update is the same)
void launch_big_step(const FactorArgs& a, const int32_t* lb, int nfronts, int ob, int maxf, double* Linv, const int64_t* linv_off,
                     cudaStream_t st, int64_t* nl) {
    static bool attr = false;
    if (!attr) {
        cudaFuncSetAttribute(k_big_diag128, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Diag128Smem));
        cudaFuncSetAttribute(k_bk_diag128, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(BkSmem));
        cudaFuncSetAttribute(k_big_trsm<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GU_SMEM);
        cudaFuncSetAttribute(k_big_trsm<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GU_SMEM);
        cudaFuncSetAttribute(k_big_update_pipe, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GU_SMEM);
        attr = true;
    }
    const bool piv = a.perm != nullptr;
    if (piv) k_bk_diag128<<<nfronts, 256, sizeof(BkSmem), st>>>(a, lb, ob, Linv, linv_off);
    else k_big_diag128<<<nfronts, 256, sizeof(Diag128Smem), st>>>(a, lb, ob, Linv, linv_off, 1);
    if (nl) ++*nl;
    const int rem = maxf - ob - 1;                  // rows below the first pivot of the block (upper bound over the fronts)
    if (rem <= 0) return;
    if (piv) k_big_trsm<true><<<dim3((rem + TR_ROWS - 1) / TR_ROWS, nfronts), 256, GU_SMEM, st>>>(a, lb, ob, Linv, linv_off, 0);
    else k_big_trsm<false><<<dim3((rem + TR_ROWS - 1) / TR_ROWS, nfronts), 256, GU_SMEM, st>>>(a, lb, ob, Linv, linv_off, 0);
    if (lookahead_bulk()) {
        static bool battr = false;
        if (!battr) { cudaFuncSetAttribute(k_big_update_pipe_bulk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GU_SMEM_BULK); battr = true; }
        k_big_update_pipe_bulk<<<dim3((rem + GU_M - 1) / GU_M, (rem + GU_N - 1) / GU_N, nfronts), GU_NT_BULK, GU_SMEM_BULK, st>>>(a, lb, ob, DB, DB, 1 << 30, 1);
    } else
    k_big_update_pipe<<<dim3((rem + GU_M - 1) / GU_M, (rem + GU_N - 1) / GU_N, nfronts), 256, GU_SMEM, st>>>(a, lb, ob, DB, DB, 1 << 30, 1);
    if (nl) *nl += 2;
}

// ----------------------------------------------------------------------------------------------------------
// Look-ahead schedule of ONE HBM-resident front (the dense solver's matrix: f = w = N; a big front of the multifrontal tree: f > w),
// three stream branches joined back into S1 (captured into the caller's graph).  Per block column k of 128 pivots:
//   chain S1:  D(k) diagonal block -> N1(k) the 128 x 128 block of L below it (k_near_trsm) -> N2(k) update of the NEXT diagonal block
//              (k_near_syrk) -> D(k+1) ...                         -- the only kernels on the critical path, each a few SMs wide
//   side  S3:  T(k) trsm of the rows from block k+2 on (after D(k)) -> C(k) rest of block column k+1 (after N1(k), R(k-1))
//   bulk  S2:  R(k) update of the columns >= k+2 incl. the front's update block (persistent, dynamic tiles, leaves the reserved SMs
//              to the chain)
// N1(k+1) waits for C(k), N2(k) and C(k) wait for R(k-1).  While the trailing update is long (first panels) the chain waits for it;
// once it is short the period is D + N1 + N2 instead of D + whole-panel trsm + whole-column update (42 + 12 + 8 us).
// Block columns whose successor is not a full pivot block (tail of the pivots, w not a multiple of 128) take the general path:
// whole-panel trsm and whole-column update on the chain.  B2_DENSE_NEAR=0 forces it everywhere (the two-branch schedule).
// ----------------------------------------------------------------------------------------------------------
__global__ void k_trace_reset(unsigned long long* t, int nslot) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 2 * nslot) t[i] = (i & 1) ? 0ull : ~0ull;
}

struct LookaheadCtx {
    cudaStream_t S2 = nullptr, S3 = nullptr;
    std::vector<cudaEvent_t>* pool = nullptr;        // events, created on demand, handed out in order
    size_t* next = nullptr;
    int32_t* tilecnt = nullptr;                      // one dynamic-tile counter per block column (zeroed by the caller)
    cudaEvent_t ev() {
        if (*next == pool->size()) { cudaEvent_t e; cudaEventCreateWithFlags(&e, cudaEventDisableTiming); pool->push_back(e); }
        return (*pool)[(*next)++];
    }
};

struct LookaheadKnobs { int n_reserved, inv_side, use_near, relax, early_reserved, chain_pdl, bulk, depth2; };
const LookaheadKnobs& lookahead_knobs() {
    static LookaheadKnobs K = [] {
        LookaheadKnobs k;
        auto geti = [](const char* name, int dflt) { const char* e = getenv(name); return e ? atoi(e) : dflt; };
        // B2_DENSE_INV_SIDE=1: the diagonal-block kernel stops after writing L11 / D back; the near-diagonal trsm substitutes against L11
        // (k_near_trsv) and the inverse (needed by the whole-panel trsm and by the solves) is formed by k_big_inv128 on the side branch
        k.inv_side = geti("B2_DENSE_INV_SIDE", 0) != 0;
        k.n_reserved = std::max(1, geti("B2_DENSE_RESERVED_SMS", k.inv_side ? 2 : 1));   // SMs the trailing update leaves to the chain
        k.use_near = geti("B2_DENSE_NEAR", 1) != 0;
        // B2_DENSE_RELAX (default 1): R(k) waits for the panel's trsm only (not for the block-column update C(k), which it does not touch), and
        // while the trailing update is long it leaves `early_reserved` SMs to the side branch so that T(k+1) / C(k+1) finish beside it
        k.relax = geti("B2_DENSE_RELAX", 1) != 0;
        k.early_reserved = std::max(1, geti("B2_DENSE_EARLY_RESERVED", 4));
        // chain kernels launched programmatically dependent on their stream predecessor (each of them starts with pdl_sync())
        k.chain_pdl = geti("B2_DENSE_PDL", 0) != 0;
        // trailing updates with TMA bulk-copy operand staging + mbarrier ring + producer warp (front_kernels.cuh: big_update_tile_bulk)
        k.bulk = geti("B2_UPDATE_BULK", 1) != 0;
        // B2_DENSE_DEPTH2=1: the side branch updates TWO block columns (k+1, k+2) and the bulk update starts at k+3, so the next diagonal
        // block only waits for the bulk update of two panels back: the chain of panel k+1 (and its panel trsm) runs a whole bulk period
        // ahead and R(k+1) can follow R(k) without a gap while the trailing update is long
        k.depth2 = geti("B2_DENSE_DEPTH2", 0) != 0;
        return k;
    }();
    return K;
}

void lookahead_attrs() {
    static bool attr = false;
    if (attr) return;
    cudaFuncSetAttribute(k_big_diag128, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Diag128Smem));
    cudaFuncSetAttribute(k_big_trsm<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GU_SMEM);
    cudaFuncSetAttribute(k_big_trsm<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GU_SMEM);
    cudaFuncSetAttribute(k_bk_diag128, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(BkSmem));
    cudaFuncSetAttribute(k_big_update_pipe, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GU_SMEM);
    cudaFuncSetAttribute(k_big_update_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GU_SMEM);
    cudaFuncSetAttribute(k_big_update_dyn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GU_SMEM);
    cudaFuncSetAttribute(k_big_update_dyn_bulk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GU_SMEM_BULK);
    cudaFuncSetAttribute(k_big_update_pipe_bulk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GU_SMEM_BULK);
    cudaFuncSetAttribute(k_near_trsm, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)NT_SMEM);
    cudaFuncSetAttribute(k_near_syrk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)NS_SMEM);
    cudaFuncSetAttribute(k_near_trsv, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)NV_SMEM);
    cudaFuncSetAttribute(k_big_inv128, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Diag128Smem));
    attr = true;
}

// `list1`: device pointer to the front's supernode id; f, w: its order and pivot count.  Returns the number of launches.
// a.perm set (Bunch-Kaufman pivoting of the dense solver): the general path throughout, with the pivoted diagonal block and trsm --
// the near-diagonal kernels have no pivoted variant.
int64_t enqueue_front_lookahead(const FactorArgs& a, const int32_t* list1, int f, int w, double* Linv, const int64_t* linv_off,
                                LookaheadCtx& cx, cudaStream_t S1) {
    const LookaheadKnobs& K = lookahead_knobs();
    lookahead_attrs();
    const int nb = (w + DB - 1) / DB, nsm = sm_count();
    cudaStream_t S2 = cx.S2, S3 = cx.S3;
    int64_t nl = 0;
    auto launch_chain = [&](auto kern, dim3 grid, size_t smem, auto... args) {
        if (K.chain_pdl) launch_pdl(kern, grid, dim3(256), smem, S1, args...);
        else kern<<<grid, 256, smem, S1>>>(args...);
        ++nl;
    };
    cudaEvent_t ev_bulk = nullptr, ev_side = nullptr;            // most recent R(.) / side-branch completion
    cudaEvent_t ev_bulk_prev = nullptr;                          // R(.) before the most recent one (depth-2 look-ahead)
    const int cw = K.depth2 ? 2 * DB : DB;                       // columns the side branch updates per panel
    const bool piv = a.perm != nullptr;
    for (int k = 0; k < nb; ++k) {
        const int ob = k * DB;
        const int nbk = std::min(DB, w - ob);                    // pivots of this block column
        const int j1 = ob + nbk;                                 // first trailing row / column
        const int rem2 = f - (ob + 2 * DB);                      // rows / columns from the block after the next on
        const bool near_step = K.use_near && !piv && ob + 2 * DB <= w;   // the next diagonal block is a full pivot block
        const int with_inv = (near_step && K.inv_side) ? 0 : 1;  // inverse of this block formed on the side branch?
        if (piv) { k_bk_diag128<<<1, 256, sizeof(BkSmem), S1>>>(a, list1, ob, Linv, linv_off); ++nl; }
        else if (K.use_near && k > 0) launch_chain(k_big_diag128, dim3(1), sizeof(Diag128Smem), a, list1, ob, Linv, linv_off, with_inv);
        else { k_big_diag128<<<1, 256, sizeof(Diag128Smem), S1>>>(a, list1, ob, Linv, linv_off, with_inv); ++nl; }
        if (j1 >= f) continue;                                   // no rows below (last block of a dense matrix)
        if (near_step) {
            cudaEvent_t ev_diag = cx.ev(), ev_near = cx.ev();
            cudaEventRecord(ev_diag, S1);
            if (ev_side) cudaStreamWaitEvent(S1, ev_side, 0);                          // C(k-1) wrote the rows N1(k) reads
            if (K.inv_side) launch_chain(k_near_trsv, dim3(DB / NT_ROWS), NV_SMEM, a, list1, ob);
            else launch_chain(k_near_trsm, dim3(DB / NT_ROWS), NT_SMEM, a, list1, ob, (const double*)Linv, linv_off);
            cudaEventRecord(ev_near, S1);
            // R(k-1) also wrote the next diagonal block -- unless the side branch covers two block columns: then R(k-1) starts at
            // block column k+2 and the last bulk writer of this tile is R(k-2)
            if (K.depth2) { if (ev_bulk_prev) cudaStreamWaitEvent(S1, ev_bulk_prev, 0); }
            else if (ev_bulk) cudaStreamWaitEvent(S1, ev_bulk, 0);
            launch_chain(k_near_syrk, dim3(10), NS_SMEM, a, list1, ob);
            if (K.inv_side) {
                cudaStreamWaitEvent(S3, ev_diag, 0);
                k_big_inv128<<<1, 256, sizeof(Diag128Smem), S3>>>(a, list1, ob, Linv, linv_off);
                ++nl;
                if (rem2 <= 0) { ev_side = cx.ev(); cudaEventRecord(ev_side, S3); }
            }
            if (rem2 > 0) {
                if (!K.inv_side) cudaStreamWaitEvent(S3, ev_diag, 0);
                k_big_trsm<false><<<dim3((rem2 + TR_ROWS - 1) / TR_ROWS, 1), 256, GU_SMEM, S3>>>(a, list1, ob, Linv, linv_off, DB / TR_ROWS);
                cudaEvent_t ev_panel = nullptr;
                if (K.relax) { ev_panel = cx.ev(); cudaEventRecord(ev_panel, S3); }    // "panel k's L is complete"
                cudaStreamWaitEvent(S3, ev_near, 0);
                if (ev_bulk) cudaStreamWaitEvent(S3, ev_bulk, 0);                      // R(k-1) also wrote these block columns
                k_big_update_rows<<<dim3((rem2 + GU_M - 1) / GU_M, (cw + GU_N - 1) / GU_N, 1), 256, GU_SMEM, S3>>>(a, list1, ob, DB, DB, DB + cw, 1, 1);
                ev_side = cx.ev();
                cudaEventRecord(ev_side, S3);
                nl += 2;
                const int remb = f - (ob + DB + cw);                                   // columns left to the bulk branch
                if (remb > 0) {
                    cudaStreamWaitEvent(S2, K.relax ? ev_panel : ev_side, 0);
                    const int nbx = (remb + GU_M - 1) / GU_M, nby = (remb + GU_N - 1) / GU_N;
                    const int nres = (K.relax && remb >= 2048) ? std::max(K.n_reserved, K.early_reserved) : K.n_reserved;
                    if (K.bulk) k_big_update_dyn_bulk<<<2 * nsm, GU_NT_BULK, GU_SMEM_BULK, S2>>>(a, list1, ob, DB, DB + cw, 1 << 30, 0, nbx, nby, cx.tilecnt + k, nres);
                    else k_big_update_dyn<<<2 * nsm, 256, GU_SMEM, S2>>>(a, list1, ob, DB, DB + cw, 1 << 30, 0, nbx, nby, cx.tilecnt + k, nres);
                    ev_bulk_prev = ev_bulk;
                    ev_bulk = cx.ev();
                    cudaEventRecord(ev_bulk, S2);
                    ++nl;
                }
            }
            continue;
        }
        // general path: whole-panel trsm and the update of the next 128 columns on the chain, the rest on the bulk branch
        if (ev_side) cudaStreamWaitEvent(S1, ev_side, 0);
        if (piv) k_big_trsm<true><<<dim3((f - j1 + TR_ROWS - 1) / TR_ROWS, 1), 256, GU_SMEM, S1>>>(a, list1, ob, Linv, linv_off, 0);
        else k_big_trsm<false><<<dim3((f - j1 + TR_ROWS - 1) / TR_ROWS, 1), 256, GU_SMEM, S1>>>(a, list1, ob, Linv, linv_off, 0);
        if (ev_bulk) cudaStreamWaitEvent(S1, ev_bulk, 0);                              // R(k-1) also wrote block column k+1
        const int jhi = std::min(f, ob + 2 * DB);
        k_big_update_pipe<<<dim3((f - j1 + GU_M - 1) / GU_M, (jhi - j1 + GU_N - 1) / GU_N, 1), 256, GU_SMEM, S1>>>(a, list1, ob, DB, DB, 2 * DB, 1);
        nl += 2;
        if (rem2 > 0) {
            cudaEvent_t ev_chain = cx.ev();
            cudaEventRecord(ev_chain, S1);
            cudaStreamWaitEvent(S2, ev_chain, 0);
            const int nbx = (rem2 + GU_M - 1) / GU_M, nby = (rem2 + GU_N - 1) / GU_N;
            if (K.bulk) k_big_update_dyn_bulk<<<2 * nsm, GU_NT_BULK, GU_SMEM_BULK, S2>>>(a, list1, ob, DB, 2 * DB, 1 << 30, 0, nbx, nby, cx.tilecnt + k, K.n_reserved);
                else k_big_update_dyn<<<2 * nsm, 256, GU_SMEM, S2>>>(a, list1, ob, DB, 2 * DB, 1 << 30, 0, nbx, nby, cx.tilecnt + k, K.n_reserved);
            ev_bulk = cx.ev();
            cudaEventRecord(ev_bulk, S2);
            ++nl;
        }
    }
    if (ev_bulk) cudaStreamWaitEvent(S1, ev_bulk, 0);                                  // join
    if (ev_side) cudaStreamWaitEvent(S1, ev_side, 0);
    return nl;
}

FactorArgs factor_args(b2_solver* s) {
    FactorArgs a;
    a.desc = s->d_desc.p; a.child_idx = s->d_child_idx.p; a.rel = s->d_rel.p;
    a.amap_src = s->d_amap_src.p; a.amap_dst = s->d_amap_dst.p;
    a.A = s->nzval_d; a.L = s->d_L.p; a.Lt = s->d_Lt.p; a.ws = s->d_ws.p; a.dvec = s->d_dvec.p;
    a.counters = s->d_counters.p; a.eps = s->opt.pivot_eps;
    a.ftrace = s->d_ftrace.p;
    return a;
}
SolveArgs solve_args(b2_solver* s) {
    SolveArgs a;
    a.desc = s->d_desc.p; a.rows = s->d_rows.p; a.child_idx = s->d_child_idx.p; a.rel = s->d_rel.p;
    a.cbv_off = s->d_cbv_off.p; a.L = s->d_L.p; a.Lt = s->d_Lt.p; a.dvec = s->d_dvec.p; a.xp = s->d_xp.p; a.cbv = s->d_cbv.p;
    return a;
}

BigSolveArgs big_solve_args(b2_solver* s) {
    BigSolveArgs b;
    b.s = solve_args(s);
    b.Linv = s->d_Linv.p;
    b.linv_off = s->d_linv_off.p;
    b.side = s->d_side.p;
    return b;
}

inline size_t smem_front(int f) { return (size_t)f * f * sizeof(double); }

WarpSched warp_sched(b2_solver* s, const WarpLaunch& L) {
    WarpSched w;
    w.cta_ptr = s->d_sched.p + L.cta_ptr_off;
    w.stage_off = s->d_sched.p + L.stage_off_off;
    w.stage_cnt = s->d_sched.p + L.stage_cnt_off;
    w.list = s->d_sched.p;
    return w;
}

// issue the numeric factorisation of one phase on `st`; returns number of launches
int64_t enqueue_factor(b2_solver* s, int ph, cudaStream_t st) {
    FactorArgs a = factor_args(s);
    a.counters += 2 * ph;   // [0,1] owned subtrees, [2,3] shared top tree
    const int32_t* sched = s->d_sched.p;
    int64_t nl = 0;
    const Phase& P = s->phase[ph];
    auto warp_launch = [&](const WarpLaunch& L) {
        if (L.nw == 1) {
            const size_t sm = (size_t)FW_WARPS * TeamSmem<1>::doubles(L.maxf) * sizeof(double);
            k_factor_warp<1><<<L.n_cta, FW_WARPS * 32, sm, st>>>(a, s->d_childrec.p, warp_sched(s, L), L.maxf);
        } else {
            const size_t sm = (size_t)TeamSmem<2>::doubles(L.maxf) * sizeof(double);
            k_factor_warp<2><<<L.n_cta, 64, sm, st>>>(a, s->d_childrec.p, warp_sched(s, L), L.maxf);
        }
        ++nl;
    };
    if (P.dep_ngroup && (s->opt.dep_schedule & 1)) {
        DepSched ds;
        ds.grp_type = sched + P.dep_type_off; ds.grp_ptr = sched + P.dep_ptr_off; ds.tasks = sched + P.dep_tasks_off; ds.ngroup = P.dep_ngroup;
        // (the group ticket in slot 3*nsuper re-arms itself: the CTA that takes the last group resets it)
        cudaMemsetAsync(s->d_flags.p, 0, (size_t)s->S.nsuper * sizeof(int32_t), st);
        const size_t sm = sizeof(double) * std::max<size_t>((size_t)FW_WARPS * TeamSmem<1>::doubles(P.dep_maxf1), (size_t)TeamSmem<2>::doubles(P.dep_maxf2));
        k_factor_dep<<<P.dep_ngroup, 128, sm, st>>>(a, s->d_childrec.p, ds, P.dep_maxf1, P.dep_maxf2, s->d_flags.p, s->d_counters.p + 4,
                                                    s->d_flags.p + (size_t)3 * s->S.nsuper);
        return 2;
    }
    if (P.fused.n_cta) warp_launch(P.fused);
    s->ev_next = 0;
    if (s->d_tilecnt.p) cudaMemsetAsync(s->d_tilecnt.p, 0, s->d_tilecnt.bytes(), st);
    for (const LevelSched& lv : P.lev) {
        if (lv.W.n_cta) warp_launch(lv.W);
        if (lv.W2.n_cta) warp_launch(lv.W2);
        if (lv.nM) {
            k_front_smem<512><<<lv.nM, 512, smem_front(lv.maxfM), st>>>(a, sched + lv.offM);
            ++nl;
        }
        if (lv.nB) {
            const int32_t* lb = sched + lv.offB;
            const int nsm = sm_count();
            // (latency-bound streaming kernels: enough warps to cover the DRAM round trips -- 32 / 64 resident warps per SM)
            k_big_zero<<<dim3(std::max(1, 16 * nsm / lv.nB), lv.nB), 256, 0, st>>>(a, lb);
            k_big_scatter_A<<<dim3(std::max(1, std::min(nsm, (lv.maxamapB + 255) / 256)), lv.nB), 256, 0, st>>>(a, lb);
            nl += 2;
            for (int c = 0; c < lv.maxchildB; ++c) {
                k_big_extend_add<<<dim3(std::max(1, std::min(8 * nsm / lv.nB + 1, (lv.maxrB * 32 + 255) / 256)), lv.nB), 256, 0, st>>>(a, lb, c);
                ++nl;
            }
            // the largest fronts one at a time, each with the whole GPU: diagonal blocks / near-diagonal steps of panel k+1 run beside
            // the trailing update of panel k (three stream branches, joined back into `st`)
            for (int i = 0; i < lv.nLA; ++i) {
                LookaheadCtx cx;
                cx.S2 = s->la_bulk; cx.S3 = s->la_side; cx.pool = &s->ev_pool; cx.next = &s->ev_next; cx.tilecnt = s->d_tilecnt.p + lv.la[i][2];
                nl += enqueue_front_lookahead(a, lb + i, lv.la[i][1], lv.la[i][0], s->d_Linv.p, s->d_linv_off.p, cx, st);
            }
            // the others batched level-wide, three launches per 128 pivot columns
            if (lv.nB > lv.nLA)
                for (int ob = 0; ob < lv.maxwBr; ob += DB)
                    launch_big_step(a, lb + lv.nLA, lv.nB - lv.nLA, ob, lv.maxfBr, s->d_Linv.p, s->d_linv_off.p, st, &nl);
        }
    }
    if (P.topfused.n_cta) warp_launch(P.topfused);
    if (P.nAllC) {
        k_big_inv<<<dim3((P.maxwAllC + BS - 1) / BS, P.nAllC), BS, (size_t)BS * (BS + 1) * sizeof(double), st>>>(
            s->d_desc.p, sched + P.offAllC, s->d_L.p, s->d_Linv.p, s->d_linv_off.p);
        ++nl;
    }
    return nl;
}

int64_t enqueue_solve(b2_solver* s, int ph, bool forward, cudaStream_t st) {
    SolveArgs a = solve_args(s);
    const int32_t* sched = s->d_sched.p;
    int64_t nl = 0;
    const Phase& P = s->phase[ph];
    // level kernels are launched programmatically dependent on their predecessor (see warp_kernels.cuh: pdl_wait)
    const bool pdl = pdl_enabled();
    cudaLaunchAttribute pattr[1];
    pattr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    pattr[0].val.programmaticStreamSerializationAllowed = 1;
    auto cfg_of = [&](int grid, int block, size_t sm) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(grid); cfg.blockDim = dim3(block); cfg.dynamicSmemBytes = sm; cfg.stream = st;
        cfg.attrs = pattr; cfg.numAttrs = pdl ? 1 : 0;
        return cfg;
    };
    auto warp_launch = [&](const WarpLaunch& L, bool fused = false) {
        const ChildRec* cr = s->d_childrec.p;
        const WarpSched wsched = warp_sched(s, L);
        if (L.nw == 1 && fused) {     // bottom subtrees: more one-warp teams per CTA, fewer sequential rounds per stage
            cudaLaunchConfig_t cfg = cfg_of(L.n_cta, SOLVE_FUSED_TEAMS * 32, (size_t)SOLVE_FUSED_TEAMS * SolveSmem<1>::doubles * sizeof(double));
            if (forward) cudaLaunchKernelEx(&cfg, k_fwd_warp2<1, SOLVE_FUSED_TEAMS>, a, cr, wsched);
            else cudaLaunchKernelEx(&cfg, k_bwd_warp2<1, SOLVE_FUSED_TEAMS>, a, wsched);
        } else if (L.nw == 1) {
            cudaLaunchConfig_t cfg = cfg_of(L.n_cta, FW_WARPS * 32, (size_t)FW_WARPS * SolveSmem<1>::doubles * sizeof(double));
            if (forward) cudaLaunchKernelEx(&cfg, k_fwd_warp2<1>, a, cr, wsched);
            else cudaLaunchKernelEx(&cfg, k_bwd_warp2<1>, a, wsched);
        } else {
            cudaLaunchConfig_t cfg = cfg_of(L.n_cta, 64, (size_t)SolveSmem<2>::doubles * sizeof(double));
            if (forward) cudaLaunchKernelEx(&cfg, k_fwd_warp2<2>, a, cr, wsched);
            else cudaLaunchKernelEx(&cfg, k_bwd_warp2<2>, a, wsched);
        }
        ++nl;
    };
    if (P.dep_ngroup && (s->opt.dep_schedule & 2)) {
        DepSched ds;
        ds.grp_type = sched + P.dep_type_off; ds.grp_ptr = sched + P.dep_ptr_off; ds.tasks = sched + P.dep_tasks_off; ds.ngroup = P.dep_ngroup;
        int* flags = s->d_flags.p + (size_t)(forward ? 1 : 2) * s->S.nsuper;
        int* ticket = s->d_flags.p + (size_t)3 * s->S.nsuper;
        cudaMemsetAsync(flags, 0, (size_t)s->S.nsuper * sizeof(int32_t), st);
        const size_t smd = sizeof(double) * std::max<size_t>((size_t)4 * SolveSmem<1>::doubles, (size_t)SolveSmem<2>::doubles);
        if (forward) k_fwd_dep<<<P.dep_ngroup, 128, smd, st>>>(a, s->d_childrec.p, ds, flags, s->d_counters.p + 4, ticket);
        else k_bwd_dep<<<P.dep_ngroup, 128, smd, st>>>(a, ds, s->d_parent.p, flags, s->d_counters.p + 4, ticket);
        return 2;
    }
    if (P.dep2_ngroup && (s->opt.dep_schedule & 4)) {
        // hybrid: the bottom subtrees in their fused staged kernel, everything above them in one flag-driven launch
        DepSched ds;
        ds.grp_type = sched + P.dep2_type_off; ds.grp_ptr = sched + P.dep2_ptr_off; ds.tasks = sched + P.dep2_tasks_off; ds.ngroup = P.dep2_ngroup;
        int* flags = s->d_flags.p + (size_t)(forward ? 1 : 2) * s->S.nsuper;
        int* ticket = s->d_flags.p + (size_t)3 * s->S.nsuper;
        const size_t smd = sizeof(double) * std::max<size_t>((size_t)4 * SolveSmem<1>::doubles, (size_t)SolveSmem<2>::doubles);
        if (forward) {
            if (P.fused.n_cta) warp_launch(P.fused, true);
            cudaMemcpyAsync(flags, s->d_flags_tpl.p, (size_t)s->S.nsuper * sizeof(int32_t), cudaMemcpyDeviceToDevice, st);   // fused fronts: done
            k_fwd_dep<<<P.dep2_ngroup, 128, smd, st>>>(a, s->d_childrec.p, ds, flags, s->d_counters.p + 4, ticket);
        } else {
            cudaMemsetAsync(flags, 0, (size_t)s->S.nsuper * sizeof(int32_t), st);
            k_bwd_dep<<<P.dep2_ngroup, 128, smd, st>>>(a, ds, s->d_parent.p, flags, s->d_counters.p + 4, ticket);
            if (P.fused.n_cta) warp_launch(P.fused, true);
        }
        return nl + 2;
    }
    if (forward && P.fused.n_cta) warp_launch(P.fused, true);
    if (!forward && P.topfused.n_cta) warp_launch(P.topfused);
    const int nlev = (int)P.lev.size();
    for (int q = 0; q < nlev; ++q) {
        const LevelSched& lv = forward ? P.lev[q] : P.lev[nlev - 1 - q];
        if (lv.W.n_cta) warp_launch(lv.W);
        if (lv.W2.n_cta) warp_launch(lv.W2);
        if (lv.nC) {
            const BigSolveArgs bs = big_solve_args(s);
            const int32_t* lc = sched + lv.offC;
            const int nblk = (lv.maxwC + BS - 1) / BS;
            if (forward) {
                k_bs_fwd_init<<<lv.nC, 1024, 0, st>>>(bs, lc);
                k_bs_head<<<lv.nC, BS_NT, 0, st>>>(bs, lc, 0, 0);
                nl += 2;
                for (int b = 0; b < nblk; ++b) {
                    const int rows = std::max(1, lv.maxfC - b * BS - 1);
                    k_bs_fwd<<<dim3((rows + BSF_ROWS - 1) / BSF_ROWS, lv.nC), BS_NT, 0, st>>>(bs, lc, b);
                    ++nl;
                }
            } else {
                k_bs_bwd_init<<<dim3((lv.maxwC + 7) / 8, lv.nC), 256, 0, st>>>(bs, lc);
                k_bs_head<<<lv.nC, BS_NT, 0, st>>>(bs, lc, -1, 1);
                nl += 2;
                for (int b = nblk - 1; b >= 1; --b) {
                    k_bs_bwd<<<dim3(b, lv.nC), BS_NT, 0, st>>>(bs, lc, b);
                    ++nl;
                }
                k_bs_bwd_finish<<<dim3((lv.maxwC + 255) / 256, lv.nC), 256, 0, st>>>(bs, lc);
                ++nl;
            }
        }
    }
    if (forward && P.topfused.n_cta) warp_launch(P.topfused);
    if (!forward && P.fused.n_cta) warp_launch(P.fused, true);
    return nl;
}

int set_smem_attrs() {
    B2_CUDA(cudaFuncSetAttribute(k_front_smem<512>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    B2_CUDA(cudaFuncSetAttribute(k_factor_warp<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
    B2_CUDA(cudaFuncSetAttribute(k_factor_warp<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
    B2_CUDA(cudaFuncSetAttribute(k_factor_dep, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
    B2_CUDA(cudaFuncSetAttribute(k_fwd_warp2<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    B2_CUDA(cudaFuncSetAttribute(k_bwd_warp2<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    B2_CUDA(cudaFuncSetAttribute((k_fwd_warp2<1, SOLVE_FUSED_TEAMS>), cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    B2_CUDA(cudaFuncSetAttribute((k_bwd_warp2<1, SOLVE_FUSED_TEAMS>), cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    B2_CUDA(cudaFuncSetAttribute(k_fwd_warp2<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    B2_CUDA(cudaFuncSetAttribute(k_bwd_warp2<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    B2_CUDA(cudaFuncSetAttribute(k_fwd_dep, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    B2_CUDA(cudaFuncSetAttribute(k_bwd_dep, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    B2_CUDA(cudaFuncSetAttribute(k_big_inv, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
    return B2_OK;
}

// capture `fn(stream)` into an executable graph
template <typename Fn>
int capture(b2_solver* s, cudaGraphExec_t* out, Fn fn) {
    if (*out) { cudaGraphExecDestroy(*out); *out = nullptr; }
    cudaGraph_t g = nullptr;
    B2_CUDA(cudaStreamBeginCapture(s->cap_stream, cudaStreamCaptureModeThreadLocal));
    fn(s->cap_stream);
    cudaError_t e = cudaStreamEndCapture(s->cap_stream, &g);
    if (e != cudaSuccess) return cuda_fail(e, "cudaStreamEndCapture", __FILE__, __LINE__);
    e = cudaGraphInstantiate(out, g, 0);
    cudaGraphDestroy(g);
    if (e != cudaSuccess) return cuda_fail(e, "cudaGraphInstantiate", __FILE__, __LINE__);
    return B2_OK;
}

void build_schedule(b2_solver* s) {
    // fronts with at least this many pivot columns get the look-ahead schedule (B2_LOOKAHEAD_MIN_W; 0 = off, the default: on the 64^3
    // augmented grid one front at a time with look-ahead measured 52.6 ms against 51.2 ms for the level-batched launches, whose
    // diagonal-block kernels already run side by side across the fronts of a level -- profiles/r02_c5_lookahead.txt)
    int la_min_w = 0, la_tiles = 0;
    if (const char* e = getenv("B2_LOOKAHEAD_MIN_W")) la_min_w = atoi(e);
    const Symbolic& S = s->S;
    const int ns = S.nsuper;
    const int rank = std::max(0, s->opt.part_rank);
    const int smax = s->opt.small_front_max;
    const int wmax = std::min(W_MAX, smax);
    const int w1max = std::min(32, smax);     // one-warp teams; fused subtrees are built from these only
    const int fuse_max = s->opt.fuse_max_fronts;
    std::vector<int32_t> sched;
    auto fdim = [&](int sn, int& w, int& f) {
        w = S.sn_first[sn + 1] - S.sn_first[sn];
        f = (int)(S.rows_ptr[sn + 1] - S.rows_ptr[sn]);
    };
    // a warp launch whose CTA c processes the stage lists given in `ctas[c]`
    auto emit_warp_launch = [&](const std::vector<std::vector<std::vector<int32_t>>>& ctas, int nw) {
        WarpLaunch L;
        L.nw = nw;
        L.n_cta = (int)ctas.size();
        std::vector<int32_t> cta_ptr(1, 0), st_off, st_cnt;
        for (const auto& stages : ctas) {
            for (const auto& fr : stages) {
                st_off.push_back((int32_t)sched.size());
                st_cnt.push_back((int32_t)fr.size());
                for (int32_t sn : fr) {
                    int w, f; fdim(sn, w, f);
                    L.maxf = std::max(L.maxf, f);
                    sched.push_back(sn);
                }
            }
            cta_ptr.push_back((int32_t)st_off.size());
        }
        L.cta_ptr_off = (int)sched.size(); sched.insert(sched.end(), cta_ptr.begin(), cta_ptr.end());
        L.stage_off_off = (int)sched.size(); sched.insert(sched.end(), st_off.begin(), st_off.end());
        L.stage_cnt_off = (int)sched.size(); sched.insert(sched.end(), st_cnt.begin(), st_cnt.end());
        return L;
    };
    for (int ph = 0; ph < 2; ++ph) {
        Phase& P = s->phase[ph];
        P.lev.clear(); P.fused = WarpLaunch(); P.n_fused_fronts = 0; P.dep_ngroup = 0;
        std::vector<char> mine(ns, 0);
        for (int sn = 0; sn < ns; ++sn) mine[sn] = (ph == 0) ? (S.owner[sn] == rank) : (S.owner[sn] == -1);
        // ---- dependency-driven single launch: every front of the phase is team-class and the tree is not sharded
        if (s->opt.dep_schedule && s->opt.n_parts <= 1 && wmax > 32) {
            bool all_team = true;
            int cntm = 0;
            for (int sn = 0; sn < ns && all_team; ++sn) if (mine[sn]) { int w, f; fdim(sn, w, f); all_team = f <= wmax; ++cntm; }
            if (all_team && cntm > 0) {
                std::vector<int32_t> order;
                for (int l = 0; l < S.nlevels; ++l)
                    for (int q = S.level_ptr[l]; q < S.level_ptr[l + 1]; ++q) if (mine[S.level_sn[q]]) order.push_back(S.level_sn[q]);
                std::vector<int32_t> gtype, gptr(1, 0), tasks;
                size_t k = 0;
                while (k < order.size()) {
                    int w, f; fdim(order[k], w, f);
                    if (f > 32) {
                        gtype.push_back(2); tasks.push_back(order[k]); ++k;
                        P.dep_maxf2 = std::max(P.dep_maxf2, f);
                    } else {
                        gtype.push_back(1);
                        int c = 0;
                        while (k < order.size() && c < FW_WARPS) {
                            int w2, f2; fdim(order[k], w2, f2);
                            if (f2 > 32) break;
                            tasks.push_back(order[k]); P.dep_maxf1 = std::max(P.dep_maxf1, f2); ++k; ++c;
                        }
                    }
                    gptr.push_back((int32_t)tasks.size());
                }
                P.dep_ngroup = (int)gtype.size();
                P.dep_type_off = (int)sched.size(); sched.insert(sched.end(), gtype.begin(), gtype.end());
                P.dep_ptr_off = (int)sched.size(); sched.insert(sched.end(), gptr.begin(), gptr.end());
                P.dep_tasks_off = (int)sched.size(); sched.insert(sched.end(), tasks.begin(), tasks.end());
            }
        }
        // ---- bottom subtrees that can run inside one CTA: all fronts warp-class, at most fuse_max fronts
        std::vector<int32_t> cnt(ns, 0);
        std::vector<char> okw(ns, 0);
        for (int sn = 0; sn < ns; ++sn) {          // children have smaller ids
            if (!mine[sn]) continue;
            int w, f; fdim(sn, w, f);
            bool ok = f <= w1max;
            int c = 1;
            for (int q = S.child_ptr[sn]; q < S.child_ptr[sn + 1]; ++q) {
                const int ch = S.child_idx[q];
                if (!mine[ch]) { continue; }       // (cannot happen inside one phase except across the top boundary)
                ok = ok && okw[ch];
                c += cnt[ch];
            }
            cnt[sn] = c;
            okw[sn] = ok && fuse_max > 0 && c <= fuse_max;
        }
        std::vector<int32_t> root_of(ns, -1);
        std::vector<int32_t> roots;
        for (int sn = ns - 1; sn >= 0; --sn) {     // parents first
            if (!mine[sn] || !okw[sn]) continue;
            const int p = S.sn_parent[sn];
            if (p >= 0 && mine[p] && okw[p]) root_of[sn] = root_of[p];
            else { root_of[sn] = sn; roots.push_back(sn); }
        }
        std::reverse(roots.begin(), roots.end());
        if (!roots.empty()) {
            std::vector<int32_t> ridx(ns, -1);
            for (size_t k = 0; k < roots.size(); ++k) ridx[roots[k]] = (int32_t)k;
            std::vector<std::vector<std::vector<int32_t>>> ctas(roots.size());
            for (int sn = 0; sn < ns; ++sn) {
                if (root_of[sn] < 0) continue;
                auto& stages = ctas[ridx[root_of[sn]]];
                const int lv = S.sn_level[sn];
                if ((int)stages.size() <= lv) stages.resize(lv + 1);
                stages[lv].push_back(sn);
                P.n_fused_fronts++;
            }
            for (auto& stages : ctas) {            // drop empty levels (cannot occur: levels are contiguous in a subtree)
                std::vector<std::vector<int32_t>> t;
                for (auto& v : stages) if (!v.empty()) t.push_back(std::move(v));
                stages.swap(t);
            }
            // longest subtrees first: better tail behaviour when there are more subtrees than resident CTAs
            std::stable_sort(ctas.begin(), ctas.end(), [](const auto& a, const auto& b) {
                size_t na = 0, nb = 0;
                for (auto& v : a) na += v.size();
                for (auto& v : b) nb += v.size();
                return na > nb;
            });
            P.fused = emit_warp_launch(ctas, 1);
        }
        // ---- the rest, level by level (levels recomputed above the fused subtrees)
        std::vector<int32_t> ulev(ns, -1);
        int nul = 0;
        for (int sn = 0; sn < ns; ++sn) {
            if (!mine[sn] || root_of[sn] >= 0) continue;
            int lv = 0;
            for (int q = S.child_ptr[sn]; q < S.child_ptr[sn + 1]; ++q) {
                const int ch = S.child_idx[q];
                if (mine[ch] && root_of[ch] < 0) lv = std::max(lv, ulev[ch] + 1);
            }
            ulev[sn] = lv;
            nul = std::max(nul, lv + 1);
        }
        std::vector<int32_t> allC;
        P.maxwAllC = 0;
        std::vector<std::vector<int32_t>> by_level(nul);
        for (int sn = 0; sn < ns; ++sn) if (ulev[sn] >= 0) by_level[ulev[sn]].push_back(sn);
        // ---- hybrid sweeps: one flag-driven launch for the whole upper tree (only when all of it is team-class and unsharded)
        P.dep2_ngroup = 0;
        if ((s->opt.dep_schedule & 4) && s->opt.n_parts <= 1 && wmax > 32 && ph == 0) {
            bool all_team = nul > 0;
            for (int l = 0; l < nul && all_team; ++l)
                for (int sn : by_level[l]) { int w, f; fdim(sn, w, f); if (f > wmax) { all_team = false; break; } }
            if (all_team) {
                std::vector<int32_t> order;
                for (int l = 0; l < nul; ++l) order.insert(order.end(), by_level[l].begin(), by_level[l].end());
                std::vector<int32_t> gtype, gptr(1, 0), tasks;
                size_t k = 0;
                while (k < order.size()) {
                    int w, f; fdim(order[k], w, f);
                    if (f > 32) { gtype.push_back(2); tasks.push_back(order[k]); ++k; }
                    else {
                        gtype.push_back(1);
                        int c = 0;
                        while (k < order.size() && c < FW_WARPS) {
                            int w2, f2; fdim(order[k], w2, f2);
                            if (f2 > 32) break;
                            tasks.push_back(order[k]); ++k; ++c;
                        }
                    }
                    gptr.push_back((int32_t)tasks.size());
                }
                P.dep2_ngroup = (int)gtype.size();
                P.dep2_type_off = (int)sched.size(); sched.insert(sched.end(), gtype.begin(), gtype.end());
                P.dep2_ptr_off = (int)sched.size(); sched.insert(sched.end(), gptr.begin(), gptr.end());
                P.dep2_tasks_off = (int)sched.size(); sched.insert(sched.end(), tasks.begin(), tasks.end());
                std::vector<int32_t> tpl(ns, 0);
                for (int sn = 0; sn < ns; ++sn) if (mine[sn] && root_of[sn] >= 0) tpl[sn] = 1;
                B2_CUDA_THROW(s->d_flags_tpl.upload(tpl.data(), tpl.size()));
            }
        }
        // ---- the top of the tree: trailing levels that hold at most 4 team-class fronts each are chained inside ONE CTA
        //      (stage = level): a launch boundary per level would cost more than the fronts themselves.
        P.topfused = WarpLaunch();
        int ntoplev = 0;
        if (wmax > 32 && s->opt.fuse_max_fronts > 0) {
            while (ntoplev < nul) {
                const auto& lvv = by_level[nul - 1 - ntoplev];
                bool ok = lvv.size() <= 4;
                for (int sn : lvv) { int w, f; fdim(sn, w, f); ok = ok && f <= wmax; }
                if (!ok) break;
                ++ntoplev;
            }
            if (ntoplev >= 2) {
                std::vector<std::vector<std::vector<int32_t>>> ctas(1);
                for (int l = nul - ntoplev; l < nul; ++l) ctas[0].push_back(by_level[l]);
                P.topfused = emit_warp_launch(ctas, 2);
                nul -= ntoplev;
            }
        }
        for (int l = 0; l < nul; ++l) {
            std::vector<int32_t> Wx, W2x, Mx, Bx;
            LevelSched lv;
            for (int sn : by_level[l]) {
                int w, f; fdim(sn, w, f);
                const int nch = S.child_ptr[sn + 1] - S.child_ptr[sn];
                const int nam = (int)(S.amap_ptr[sn + 1] - S.amap_ptr[sn]);
                if (f <= wmax && wmax > 32) W2x.push_back(sn);      // above the fused subtrees fronts are few: two-warp teams
                else if (f <= w1max) Wx.push_back(sn);
                else if (f <= smax) { Mx.push_back(sn); lv.maxfM = std::max(lv.maxfM, f); }
                else {
                    Bx.push_back(sn);
                    lv.maxfB = std::max(lv.maxfB, f); lv.maxwB = std::max(lv.maxwB, w);
                    lv.maxchildB = std::max(lv.maxchildB, nch); lv.maxamapB = std::max(lv.maxamapB, nam);
                    for (int c = S.child_ptr[sn]; c < S.child_ptr[sn + 1]; ++c) {
                        int cw, cf; fdim(S.child_idx[c], cw, cf);
                        lv.maxrB = std::max(lv.maxrB, cf - cw);
                    }
                }
                if (f > wmax) {
                    lv.maxfC = std::max(lv.maxfC, f); lv.maxwC = std::max(lv.maxwC, w);
                    if (f <= smax) { allC.push_back(sn); P.maxwAllC = std::max(P.maxwAllC, w); }   // (B fronts invert in k_big_diag128)
                }
            }
            auto level_launch = [&](const std::vector<int32_t>& X, int nw) {
                std::vector<std::vector<std::vector<int32_t>>> ctas;
                const size_t per = (nw == 1) ? FW_WARPS : 1;
                for (size_t k = 0; k < X.size(); k += per) {
                    std::vector<int32_t> fr(X.begin() + k, X.begin() + std::min(X.size(), k + per));
                    ctas.push_back({fr});
                }
                return emit_warp_launch(ctas, nw);
            };
            if (!Wx.empty()) lv.W = level_launch(Wx, 1);
            if (!W2x.empty()) lv.W2 = level_launch(W2x, 2);
            lv.offM = (int)sched.size(); lv.nM = (int)Mx.size(); sched.insert(sched.end(), Mx.begin(), Mx.end());
            {   // look-ahead fronts first (stable: ascending supernode id inside both groups)
                std::vector<int32_t> la_sn, rest;
                for (int sn : Bx) {
                    int w, f; fdim(sn, w, f);
                    if (la_min_w > 0 && w >= la_min_w && s->la_bulk && s->la_side) {
                        la_sn.push_back(sn);
                        lv.la.push_back({w, f, la_tiles});
                        la_tiles += (w + DB - 1) / DB;
                    } else {
                        rest.push_back(sn);
                        lv.maxfBr = std::max(lv.maxfBr, f); lv.maxwBr = std::max(lv.maxwBr, w);
                    }
                }
                lv.nLA = (int)la_sn.size();
                Bx = la_sn; Bx.insert(Bx.end(), rest.begin(), rest.end());
            }
            lv.offB = (int)sched.size(); lv.nB = (int)Bx.size(); sched.insert(sched.end(), Bx.begin(), Bx.end());
            lv.offC = lv.offM; lv.nC = lv.nM + lv.nB;        // M and B lists are adjacent
            P.lev.push_back(lv);
        }
        P.offAllC = (int)sched.size(); P.nAllC = (int)allC.size(); sched.insert(sched.end(), allC.begin(), allC.end());
    }
    if (sched.empty()) sched.push_back(0);
    B2_CUDA_THROW(s->d_sched.upload(sched.data(), sched.size()));
    if (la_tiles) B2_CUDA_THROW(s->d_tilecnt.alloc((size_t)la_tiles));
}

int create_common(int32_t n, int64_t nnz, const int32_t* colptr_h, const int32_t* rowval_h, const double* nzval_d,
                  const b2_options* opt, const int32_t* user_perm_h, bool symbolic_only, b2_solver** out) {
    if (!out || !colptr_h || !rowval_h || n <= 0) { set_error("b2_create: invalid argument"); return B2_ERR_INVALID; }
    if (colptr_h[n] != nnz) { set_error("b2_create: colptr[n] != nnz"); return B2_ERR_INVALID; }
    if (opt && opt->pivoting != B2_PIVOT_STATIC) { set_error("b2_create: pivoting mode not supported by the sparse solver"); return B2_ERR_INVALID; }
    b2_solver* s = new b2_solver();
    if (opt) s->opt = *opt; else b2_options_default(&s->opt);
    s->symbolic_only = symbolic_only;
    s->nzval_d = nzval_d;
    if (s->opt.small_front_max < 8) s->opt.small_front_max = 8;
    if (s->opt.small_front_max > 168) s->opt.small_front_max = 168;
    try {
        AnalysisOptions ao;
        ao.ordering = s->opt.ordering; ao.nemin = s->opt.nemin; ao.relax_zeros = s->opt.relax_zeros;
        ao.chain_merge_f = s->opt.chain_merge_f;
        ao.n_parts = std::max(1, s->opt.n_parts);
        ao.kkt_n_primal = s->opt.kkt_n_primal;
        analyse(n, colptr_h, rowval_h, ao, user_perm_h, s->S);
    } catch (std::exception& e) {
        set_error(std::string("b2_create: analysis failed: ") + e.what());
        delete s;
        return B2_ERR_SYMBOLIC;
    }
    const Symbolic& S = s->S;
    const int ns = S.nsuper;
    // contribution-vector offsets: blocks crossing into the shared top tree first (exchange region)
    {
        s->cbv_off.assign(ns + 1, 0);
        int64_t off = 0;
        const bool multi = s->opt.n_parts > 1;
        for (int pass = 0; pass < 2; ++pass) {
            for (int sn = 0; sn < ns; ++sn) {
                const int p = S.sn_parent[sn];
                const bool boundary = multi && S.owner[sn] >= 0 && p >= 0 && S.owner[p] == -1;
                if ((pass == 0) != boundary) continue;
                s->cbv_off[sn] = off;
                off += S.rel_ptr[sn + 1] - S.rel_ptr[sn];
            }
            if (pass == 0) s->exch_cbv = off;
        }
        s->cbv_off[ns] = off;
    }
    // rows this rank finalises in the back-substitution (multi-GPU); rank 0 also reports the top tree
    {
        s->owned_mask.assign(n, 1);
        if (s->opt.n_parts > 1) {
            const int rank = s->opt.part_rank;
            for (int sn = 0; sn < ns; ++sn) {
                const bool mine = S.owner[sn] == rank || (S.owner[sn] == -1 && rank == 0);
                for (int j = S.sn_first[sn]; j < S.sn_first[sn + 1]; ++j) s->owned_mask[S.perm[j]] = mine ? 1 : 0;
            }
        }
    }
    if (symbolic_only) { *out = s; return B2_OK; }

    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        set_error("b2_create: no CUDA device (this library has no CPU fallback)");
        delete s;
        return B2_ERR_NO_DEVICE;
    }
    cudaGetDevice(&s->device);
    try {
        std::vector<FrontDesc> desc(ns);
        for (int sn = 0; sn < ns; ++sn) {
            FrontDesc& d = desc[sn];
            d.col0 = S.sn_first[sn];
            d.w = S.sn_first[sn + 1] - S.sn_first[sn];
            d.f = (int)(S.rows_ptr[sn + 1] - S.rows_ptr[sn]);
            d.nchild = S.child_ptr[sn + 1] - S.child_ptr[sn];
            d.child_off = S.child_ptr[sn];
            d.amap_cnt = (int)(S.amap_ptr[sn + 1] - S.amap_ptr[sn]);
            d.rows_off = S.rows_ptr[sn];
            d.lp_off = S.lp_off[sn];
            d.cb_off = S.cb_off[sn];
            d.rel_off = S.rel_ptr[sn];
            d.amap_off = S.amap_ptr[sn];
        }
        std::vector<int32_t> asrc(S.amap_src.size()), adst(S.amap_dst.size());
        for (int sn = 0; sn < ns; ++sn)
            for (int64_t q = S.amap_ptr[sn]; q < S.amap_ptr[sn + 1]; ++q) {
                asrc[q] = (int32_t)S.amap_src[q];
                adst[q] = (int32_t)(S.amap_dst[q] - S.lp_off[sn]);
            }
        std::vector<uint8_t> mask_p(n);
        for (int j = 0; j < n; ++j) mask_p[j] = s->owned_mask[S.perm[j]];
        B2_CUDA_THROW(s->d_desc.upload(desc.data(), desc.size()));
        B2_CUDA_THROW(s->d_rows.upload(S.rows.data(), S.rows.size()));
        B2_CUDA_THROW(s->d_child_idx.upload(S.child_idx.data(), S.child_idx.size()));
        B2_CUDA_THROW(s->d_rel.upload(S.rel.data(), S.rel.size()));
        B2_CUDA_THROW(s->d_amap_src.upload(asrc.data(), asrc.size()));
        B2_CUDA_THROW(s->d_amap_dst.upload(adst.data(), adst.size()));
        B2_CUDA_THROW(s->d_perm.upload(S.perm.data(), S.perm.size()));
        B2_CUDA_THROW(s->d_cbv_off.upload(s->cbv_off.data(), s->cbv_off.size()));
        B2_CUDA_THROW(s->d_mask_p.upload(mask_p.data(), mask_p.size()));
        {
            std::vector<ChildRec> cr(std::max<size_t>(1, S.child_idx.size()));
            for (size_t q = 0; q < S.child_idx.size(); ++q) {
                const int c = S.child_idx[q];
                cr[q].cb_off = S.cb_off[c];
                cr[q].rel_off = S.rel_ptr[c];
                cr[q].cbv_off = s->cbv_off[c];
                cr[q].rc = (int32_t)(S.rel_ptr[c + 1] - S.rel_ptr[c]);
                cr[q].sn = c;
            }
            B2_CUDA_THROW(s->d_childrec.upload(cr.data(), cr.size()));
        }
        if (const char* e = getenv("B2_SPARSE_TRACE")) if (atoi(e)) B2_CUDA_THROW(s->d_ftrace.alloc((size_t)3 * ns));
        B2_CUDA_THROW(s->d_L.alloc((size_t)S.lp_off[ns] + 2));          // (+2: the bulk-copy staging may read one aligned pair past a panel)
        B2_CUDA_THROW(s->d_Lt.alloc((size_t)S.lp_off[ns]));
        {
            const int wmax_ = std::min(W_MAX, s->opt.small_front_max);
            std::vector<int64_t> lo(ns, -1);
            int64_t tot = 0;
            for (int sn = 0; sn < ns; ++sn) {
                const int w = S.sn_first[sn + 1] - S.sn_first[sn];
                const int f = (int)(S.rows_ptr[sn + 1] - S.rows_ptr[sn]);
                if (f > wmax_) { lo[sn] = tot; tot += (int64_t)((w + BS - 1) / BS) * BS * BS; }
            }
            B2_CUDA_THROW(s->d_linv_off.upload(lo.data(), lo.size()));
            B2_CUDA_THROW(s->d_Linv.alloc((size_t)std::max<int64_t>(1, tot)));
            B2_CUDA_THROW(s->d_side.alloc(tot > 0 ? (size_t)n : 1));
        }
        B2_CUDA_THROW(s->d_ws.alloc((size_t)std::max<int64_t>(1, S.cb_off[ns])));
        B2_CUDA_THROW(s->d_dvec.alloc(n));
        B2_CUDA_THROW(s->d_xp.alloc(n));
        B2_CUDA_THROW(s->d_cbv.alloc((size_t)std::max<int64_t>(1, s->cbv_off[ns])));
        B2_CUDA_THROW(s->d_counters.alloc(8));
        B2_CUDA_THROW(cudaMemset(s->d_counters.p, 0, 8 * sizeof(int32_t)));
        B2_CUDA_THROW(s->d_flags.alloc((size_t)3 * ns + 1));
        B2_CUDA_THROW(cudaMemset(s->d_flags.p, 0, s->d_flags.bytes()));
        B2_CUDA_THROW(s->d_parent.upload(S.sn_parent.data(), S.sn_parent.size()));
        B2_CUDA_THROW(cudaMemset(s->d_ws.p, 0, s->d_ws.bytes()));
        B2_CUDA_THROW(cudaMemset(s->d_cbv.p, 0, s->d_cbv.bytes()));
        B2_CUDA_THROW(cudaMallocHost((void**)&s->h_counters, 8 * sizeof(int32_t)));
        B2_CUDA_THROW(cudaStreamCreateWithFlags(&s->cap_stream, cudaStreamNonBlocking));
        B2_CUDA_THROW(cudaStreamCreateWithFlags(&s->la_bulk, cudaStreamNonBlocking));
        B2_CUDA_THROW(cudaStreamCreateWithFlags(&s->la_side, cudaStreamNonBlocking));
        build_schedule(s);
        if (set_smem_attrs() != B2_OK) throw std::runtime_error("attr");
    } catch (std::exception&) {
        delete s;
        return B2_ERR_CUDA;
    }
    *out = s;
    return B2_OK;
}

// a pre-instantiated graph cannot be launched into a stream that is itself being captured (e.g. the caller records a
// whole IPM step into its own CUDA graph): in that case the kernels are enqueued directly and become part of THAT graph
bool stream_is_capturing(cudaStream_t st) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cs) != cudaSuccess) { cudaGetLastError(); return false; }
    return cs == cudaStreamCaptureStatusActive;
}

int run_factor_phase(b2_solver* s, int ph, cudaStream_t st) {
    Phase& P = s->phase[ph];
    if (s->opt.use_cuda_graph && !stream_is_capturing(st)) {
        if (!P.g_factor) {
            int rc = capture(s, &P.g_factor, [&](cudaStream_t cs) { P.n_factor_launches = enqueue_factor(s, ph, cs); });
            if (rc != B2_OK) return rc;
        }
        B2_CUDA(cudaGraphLaunch(P.g_factor, st));
    } else {
        P.n_factor_launches = enqueue_factor(s, ph, st);
        B2_CUDA(cudaGetLastError());
    }
    return B2_OK;
}

int run_solve_phase(b2_solver* s, int ph, bool fwd, cudaStream_t st) {
    Phase& P = s->phase[ph];
    cudaGraphExec_t* g = fwd ? &P.g_fwd : &P.g_bwd;
    if (s->opt.use_cuda_graph && !stream_is_capturing(st)) {
        if (!*g) {
            int64_t nl = 0;
            int rc = capture(s, g, [&](cudaStream_t cs) { nl = enqueue_solve(s, ph, fwd, cs); });
            if (rc != B2_OK) return rc;
            if (fwd) P.n_solve_launches = 2 * nl;
        }
        B2_CUDA(cudaGraphLaunch(*g, st));
    } else {
        int64_t nl = enqueue_solve(s, ph, fwd, st);
        if (fwd) P.n_solve_launches = 2 * nl;
        B2_CUDA(cudaGetLastError());
    }
    return B2_OK;
}

}  // namespace

extern "C" {

int b2_options_default(b2_options* opt) {
    if (!opt) return B2_ERR_INVALID;
    std::memset(opt, 0, sizeof(*opt));
    opt->ordering = B2_ORDER_METIS_ND;
    opt->nemin = 16;
    opt->relax_zeros = 0.25;
    opt->pivot_eps = 1e-13;
    opt->use_cuda_graph = 1;
    opt->small_front_max = 160;
    opt->fuse_max_fronts = 8;      // measured optimum on OPF-10k (profiles/r02_sweep.txt)
    opt->dep_schedule = 1;
    if (const char* e = getenv("B2_DEP_SCHEDULE")) opt->dep_schedule = atoi(e);
    opt->chain_merge_f = 0;      // measured on the OPF-10k tree: 16 -> 11 levels but the merged (two-warp, 14 us) leaves make the
                                 // throughput-bound bottom of the tree 30 us longer: factorize 0.145 -> 0.172 ms (profiles/r02_chain_merge.txt)
    if (const char* e = getenv("B2_CHAIN_MERGE_F")) opt->chain_merge_f = atoi(e);
    opt->n_parts = 1;
    opt->part_rank = 0;
    return B2_OK;
}

int b2_create(int32_t n, int64_t nnz, const int32_t* colptr_h, const int32_t* rowval_h, const double* nzval_d,
              const b2_options* opt, const int32_t* user_perm_h, b2_solver** out) {
    return create_common(n, nnz, colptr_h, rowval_h, nzval_d, opt, user_perm_h, false, out);
}

int b2_create_symbolic_only(int32_t n, int64_t nnz, const int32_t* colptr_h, const int32_t* rowval_h,
                            const b2_options* opt, const int32_t* user_perm_h, b2_solver** out) {
    return create_common(n, nnz, colptr_h, rowval_h, nullptr, opt, user_perm_h, true, out);
}

int b2_destroy(b2_solver* s) {
    delete s;
    return B2_OK;
}

int b2_set_values_ptr(b2_solver* s, const double* nzval_d) {
    if (!s) return B2_ERR_INVALID;
    if (nzval_d != s->nzval_d) {
        s->nzval_d = nzval_d;
        for (auto& p : s->phase)
            if (p.g_factor) { cudaGraphExecDestroy(p.g_factor); p.g_factor = nullptr; }   // pointer is baked into the graph
    }
    return B2_OK;
}

int b2_factorize_local(b2_solver* s, void* stream) {
    if (!s || s->symbolic_only) { set_error("b2_factorize: solver has no device state"); return B2_ERR_INVALID; }
    if (!s->nzval_d) { set_error("b2_factorize: value pointer not set"); return B2_ERR_INVALID; }
    cudaStream_t st = as_stream(stream);
    B2_CUDA(cudaMemsetAsync(s->d_counters.p, 0, 8 * sizeof(int32_t), st));
    if (s->opt.n_parts > 1 && s->S.exch_cb > 0) B2_CUDA(cudaMemsetAsync(s->d_ws.p, 0, (size_t)s->S.exch_cb * sizeof(double), st));
    return run_factor_phase(s, 0, st);
}

int b2_factorize_top(b2_solver* s, void* stream) {
    if (!s || s->symbolic_only) return B2_ERR_INVALID;
    int rc = run_factor_phase(s, 1, as_stream(stream));
    if (rc == B2_OK) s->factorized = true;
    return rc;
}

int b2_factorize(b2_solver* s, void* stream) {
    int rc = b2_factorize_local(s, stream);
    if (rc != B2_OK) return rc;
    if (s->opt.n_parts > 1) { set_error("b2_factorize: multi-part solver needs factorize_local/exchange/factorize_top"); return B2_ERR_INVALID; }
    s->factorized = true;
    return B2_OK;
}

int b2_inertia_enqueue(b2_solver* s, void* stream) {
    if (!s || s->symbolic_only || !s->factorized) { set_error("b2_inertia: not factorized"); return B2_ERR_FACTORIZATION; }
    B2_CUDA(cudaMemcpyAsync(s->h_counters, s->d_counters.p, 8 * sizeof(int32_t), cudaMemcpyDeviceToHost, as_stream(stream)));
    return B2_OK;
}

int b2_inertia_fetch(b2_solver* s, int64_t* num_pos, int64_t* num_zero, int64_t* num_neg) {
    if (!s || s->symbolic_only || !s->factorized) { set_error("b2_inertia: not factorized"); return B2_ERR_FACTORIZATION; }
    if (s->h_counters[4]) { set_error("b2: dependency wait timed out inside the single-launch schedule"); return B2_ERR_FACTORIZATION; }
    // single-part: everything is in the "local" phase.  Multi-part: this is only this rank's view; the host layer
    // all-reduces b2_inertia_parts() instead.
    const int64_t neg = (int64_t)s->h_counters[0] + s->h_counters[2], zero = (int64_t)s->h_counters[1] + s->h_counters[3];
    s->last_perturbed = zero;
    if (num_neg) *num_neg = neg;
    if (num_zero) *num_zero = zero;
    if (num_pos) *num_pos = (int64_t)s->S.n - neg - zero;
    return B2_OK;
}

int b2_inertia(b2_solver* s, int64_t* num_pos, int64_t* num_zero, int64_t* num_neg, void* stream) {
    int rc = b2_inertia_enqueue(s, stream);
    if (rc != B2_OK) return rc;
    B2_CUDA(cudaStreamSynchronize(as_stream(stream)));
    return b2_inertia_fetch(s, num_pos, num_zero, num_neg);
}

int b2_inertia_parts(b2_solver* s, int64_t* local_neg, int64_t* local_zero, int64_t* top_neg, int64_t* top_zero, void* stream) {
    if (!s || s->symbolic_only || !s->factorized) { set_error("b2_inertia_parts: not factorized"); return B2_ERR_FACTORIZATION; }
    cudaStream_t st = as_stream(stream);
    B2_CUDA(cudaMemcpyAsync(s->h_counters, s->d_counters.p, 8 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    B2_CUDA(cudaStreamSynchronize(st));
    if (s->h_counters[4]) { set_error("b2: dependency wait timed out inside the single-launch schedule"); return B2_ERR_FACTORIZATION; }
    if (local_neg) *local_neg = s->h_counters[0];
    if (local_zero) *local_zero = s->h_counters[1];
    if (top_neg) *top_neg = s->h_counters[2];
    if (top_zero) *top_zero = s->h_counters[3];
    return B2_OK;
}

int b2_solve_fwd_local(b2_solver* s, double* x_d, void* stream) {
    if (!s || s->symbolic_only || !x_d) return B2_ERR_INVALID;
    if (!s->factorized) { set_error("b2_solve: not factorized"); return B2_ERR_SOLVE; }
    cudaStream_t st = as_stream(stream);
    const int n = s->S.n;
    const int grid = std::min(4 * sm_count(), (n + 255) / 256);
    launch_pdl(k_perm_in, dim3(grid), dim3(256), 0, st, n, s->d_perm.p, x_d, s->d_xp.p);
    if (s->opt.n_parts > 1 && s->exch_cbv > 0) B2_CUDA(cudaMemsetAsync(s->d_cbv.p, 0, (size_t)s->exch_cbv * sizeof(double), st));
    return run_solve_phase(s, 0, true, st);
}

int b2_solve_top(b2_solver* s, double* x_d, void* stream) {
    if (!s || s->symbolic_only) return B2_ERR_INVALID;
    (void)x_d;
    int rc = run_solve_phase(s, 1, true, as_stream(stream));
    if (rc != B2_OK) return rc;
    return run_solve_phase(s, 1, false, as_stream(stream));
}

int b2_solve_bwd_local(b2_solver* s, double* x_d, void* stream) {
    if (!s || s->symbolic_only || !x_d) return B2_ERR_INVALID;
    cudaStream_t st = as_stream(stream);
    int rc = run_solve_phase(s, 0, false, st);
    if (rc != B2_OK) return rc;
    const int n = s->S.n;
    const int grid = std::min(4 * sm_count(), (n + 255) / 256);
    if (s->opt.n_parts > 1) k_perm_out_masked<<<grid, 256, 0, st>>>(n, s->d_perm.p, s->d_mask_p.p, s->d_xp.p, x_d);
    else launch_pdl(k_perm_out, dim3(grid), dim3(256), 0, st, n, s->d_perm.p, s->d_xp.p, x_d);
    B2_CUDA(cudaGetLastError());
    return B2_OK;
}

int b2_solve(b2_solver* s, double* x_d, int32_t nrhs, void* stream) {
    if (!s || s->symbolic_only || !x_d || nrhs < 1) { set_error("b2_solve: invalid argument"); return B2_ERR_INVALID; }
    if (s->opt.n_parts > 1) { set_error("b2_solve: multi-part solver needs the phased solve"); return B2_ERR_INVALID; }
    for (int c = 0; c < nrhs; ++c) {
        double* x = x_d + (size_t)c * s->S.n;
        int rc = b2_solve_fwd_local(s, x, stream);
        if (rc != B2_OK) return rc;
        rc = b2_solve_bwd_local(s, x, stream);
        if (rc != B2_OK) return rc;
    }
    return B2_OK;
}

int b2_improve(b2_solver* s, int32_t* changed) {
    if (!s) return B2_ERR_INVALID;
    // Static pivoting has one knob: the perturbation threshold.  Raise it (like ma97's u -> u^0.75, ma97.jl:103-111)
    // up to 1e-8; the caller re-factorises.
    int32_t ch = 0;
    if (s->opt.pivot_eps < 1e-8) {
        s->opt.pivot_eps = std::min(1e-8, std::max(s->opt.pivot_eps * 100.0, 1e-13));
        for (auto& p : s->phase)
            if (p.g_factor) { cudaGraphExecDestroy(p.g_factor); p.g_factor = nullptr; }
        ch = 1;
    }
    if (changed) *changed = ch;
    return B2_OK;
}

int b2_get_stats(b2_solver* s, b2_stats* st) {
    if (!s || !st) return B2_ERR_INVALID;
    std::memset(st, 0, sizeof(*st));
    const Symbolic& S = s->S;
    st->n = S.n; st->nnz_a = S.nnz_a; st->nnz_l = S.nnz_l; st->flops = S.flops;
    st->n_supernodes = S.nsuper; st->n_levels = S.nlevels; st->max_front = S.max_front;
    const int smax = s->opt.small_front_max;
    for (int sn = 0; sn < S.nsuper; ++sn) {
        const int f = (int)(S.rows_ptr[sn + 1] - S.rows_ptr[sn]);
        if (f <= smax) st->n_small_fronts++; else st->n_big_fronts++;
    }
    st->factor_bytes = (int64_t)S.lp_off[S.nsuper] * 8;
    st->workspace_bytes = (int64_t)(S.cb_off[S.nsuper] + s->cbv_off[S.nsuper]) * 8;
    st->sep_rows = S.top_rows;
    st->n_factor_launches = s->phase[0].n_factor_launches + s->phase[1].n_factor_launches;
    st->n_solve_launches = s->phase[0].n_solve_launches + s->phase[1].n_solve_launches;
    st->n_perturbed = s->last_perturbed;
    return B2_OK;
}

int b2_get_perm(b2_solver* s, int32_t* perm_h) {
    if (!s || !perm_h) return B2_ERR_INVALID;
    std::memcpy(perm_h, s->S.perm.data(), (size_t)s->S.n * sizeof(int32_t));
    return B2_OK;
}

int b2_exchange_buffer(b2_solver* s, double** buf_d, int64_t* n_factor_doubles, int64_t* n_solve_doubles) {
    if (!s || s->symbolic_only) return B2_ERR_INVALID;
    if (buf_d) *buf_d = s->d_ws.p;
    if (n_factor_doubles) *n_factor_doubles = s->S.exch_cb;
    if (n_solve_doubles) *n_solve_doubles = s->exch_cbv;
    return B2_OK;
}

int b2_exchange_vector(b2_solver* s, double** buf_d, int64_t* n_doubles) {
    if (!s || s->symbolic_only) return B2_ERR_INVALID;
    if (buf_d) *buf_d = s->d_cbv.p;
    if (n_doubles) *n_doubles = s->exch_cbv;
    return B2_OK;
}

int b2_owned_mask(b2_solver* s, uint8_t* owned_h) {
    if (!s || !owned_h) return B2_ERR_INVALID;
    std::memcpy(owned_h, s->owned_mask.data(), s->owned_mask.size());
    return B2_OK;
}

int b2_symbolic_query(b2_solver* s, b2_symbolic_sizes* sz) {
    if (!s || !sz) return B2_ERR_INVALID;
    const Symbolic& S = s->S;
    sz->n = S.n; sz->n_supernodes = S.nsuper; sz->n_rows = (int64_t)S.rows.size();
    sz->n_children = (int64_t)S.child_idx.size(); sz->n_rel = (int64_t)S.rel.size();
    sz->n_amap = (int64_t)S.amap_src.size(); sz->n_levels = S.nlevels;
    sz->lval_size = S.lp_off[S.nsuper]; sz->cb_size = S.cb_off[S.nsuper];
    return B2_OK;
}

int b2_symbolic_export(b2_solver* s, int32_t* perm, int32_t* sn_first, int32_t* sn_parent, int32_t* sn_level,
                       int64_t* rows_ptr, int32_t* rows, int64_t* lp_off, int64_t* cb_off,
                       int64_t* rel_ptr, int32_t* rel, int64_t* amap_ptr, int64_t* amap_src, int64_t* amap_dst) {
    if (!s) return B2_ERR_INVALID;
    const Symbolic& S = s->S;
    auto cp = [](auto* dst, const auto& v) { if (dst) std::memcpy(dst, v.data(), v.size() * sizeof(v[0])); };
    cp(perm, S.perm); cp(sn_first, S.sn_first); cp(sn_parent, S.sn_parent); cp(sn_level, S.sn_level);
    cp(rows_ptr, S.rows_ptr); cp(rows, S.rows); cp(lp_off, S.lp_off); cp(cb_off, S.cb_off);
    cp(rel_ptr, S.rel_ptr); cp(rel, S.rel); cp(amap_ptr, S.amap_ptr); cp(amap_src, S.amap_src); cp(amap_dst, S.amap_dst);
    return B2_OK;
}

int b2_debug_profile_front(b2_solver* s, int32_t sn, int32_t reps, int64_t* stamps_h) {
    if (!s || s->symbolic_only || sn < 0 || sn >= s->S.nsuper || reps < 1 || reps > 64) return B2_ERR_INVALID;
    const int f = (int)(s->S.rows_ptr[sn + 1] - s->S.rows_ptr[sn]);
    if (f > W_MAX) { set_error("b2_debug_profile_front: front is not team-class"); return B2_ERR_INVALID; }
    DevBuf<long long> prof;
    B2_CUDA(prof.alloc(8 * reps));
    FactorArgs a = factor_args(s);
    a.counters += 2;   // scratch counters: do not disturb the inertia of the real factorisation
    if (f <= 32) {
        B2_CUDA(cudaFuncSetAttribute(k_factor_team_profile<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
        k_factor_team_profile<1><<<1, 32, (size_t)TeamSmem<1>::doubles(f) * sizeof(double)>>>(a, s->d_childrec.p, sn, f, prof.p, reps);
    } else {
        B2_CUDA(cudaFuncSetAttribute(k_factor_team_profile<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
        k_factor_team_profile<2><<<1, 64, (size_t)TeamSmem<2>::doubles(f) * sizeof(double)>>>(a, s->d_childrec.p, sn, f, prof.p, reps);
    }
    B2_CUDA(cudaDeviceSynchronize());
    B2_CUDA(cudaMemcpy(stamps_h, prof.p, 8 * reps * sizeof(long long), cudaMemcpyDeviceToHost));
    return B2_OK;
}

int b2_debug_trace(b2_solver* s, uint64_t* stamps_h, int32_t* parent_h, int32_t* w_h, int32_t* f_h, int64_t capacity, int64_t* count) {
    if (!s || !count) { set_error("b2_debug_trace: invalid argument"); return B2_ERR_INVALID; }
    const int64_t ns = s->S.nsuper;
    *count = ns;
    if (capacity < ns) return B2_OK;
    for (int64_t i = 0; i < ns; ++i) {
        if (parent_h) parent_h[i] = s->S.sn_parent[i];
        const int w = s->S.sn_first[i + 1] - s->S.sn_first[i];
        if (w_h) w_h[i] = w;
        if (f_h) f_h[i] = (int32_t)(s->S.rows_ptr[i + 1] - s->S.rows_ptr[i]);
    }
    if (stamps_h && s->d_ftrace.p) {
        B2_CUDA(cudaDeviceSynchronize());
        B2_CUDA(cudaMemcpy(stamps_h, s->d_ftrace.p, s->d_ftrace.bytes(), cudaMemcpyDeviceToHost));
    } else if (stamps_h) {
        std::memset(stamps_h, 0, (size_t)3 * ns * sizeof(uint64_t));
    }
    return B2_OK;
}

int b2_debug_get_factor(b2_solver* s, double* lval_h, double* dvec_h) {
    if (!s || s->symbolic_only) return B2_ERR_INVALID;
    B2_CUDA(cudaDeviceSynchronize());
    if (lval_h) B2_CUDA(cudaMemcpy(lval_h, s->d_L.p, (size_t)s->S.lp_off[s->S.nsuper] * sizeof(double), cudaMemcpyDeviceToHost));
    if (dvec_h) B2_CUDA(cudaMemcpy(dvec_h, s->d_dvec.p, s->d_dvec.bytes(), cudaMemcpyDeviceToHost));
    return B2_OK;
}

int b2_symbolic_exchange(b2_solver* s, int64_t* cbv_off, int64_t* exch_cb, int64_t* exch_cbv) {
    if (!s) return B2_ERR_INVALID;
    if (cbv_off) std::memcpy(cbv_off, s->cbv_off.data(), s->cbv_off.size() * sizeof(int64_t));
    if (exch_cb) *exch_cb = s->S.exch_cb;
    if (exch_cbv) *exch_cbv = s->exch_cbv;
    return B2_OK;
}

int b2_symbolic_owner(b2_solver* s, int32_t* owner) {
    if (!s || !owner) return B2_ERR_INVALID;
    std::memcpy(owner, s->S.owner.data(), s->S.owner.size() * sizeof(int32_t));
    return B2_OK;
}

}  // extern "C"

// =========================================================================================================
// b2d_*: dense LDL^T (DenseCondensedKKTSystem back-end; replaces cusolverDnDsytrf/Xsytrs, cusolver.jl:150-187,
// and dsytrf/dsytrs, src/LinearSolvers/lapack.jl:164-172).  The dense matrix is one "big front" with w = f = N:
// the same blocked right-looking kernels (k_big_diag128 / k_big_trsm / k_big_update_pipe, bigfactor_kernels.cuh).
// =========================================================================================================
struct b2d_solver {
    int32_t N = 0, lda = 0;
    const double* A_d = nullptr;
    b2_options opt;
    DevBuf<double> fact, dvec, linv, side, flow;     // flow: [2][nblk*128] hand-off vectors of the single-launch solve
    DevBuf<int32_t> tilecnt;                         // look-ahead schedule: one dynamic-tile counter per panel step
    DevBuf<unsigned long long> trace;                // B2_DENSE_TRACE=1: [8 * nblk][2] first-entry / last-exit stamps (b2d_debug_trace)
    cudaStream_t aux_stream = nullptr;               // second branch of the look-ahead schedule (trailing updates)
    cudaStream_t side_stream = nullptr;              // third branch: rest of the panel (trsm + next block column) beside the next diagonal block
    std::vector<cudaEvent_t> ev_pool;               // events of the look-ahead schedule (created on demand)
    size_t ev_next = 0;
    DevBuf<int64_t> linv_off;
    DevBuf<FrontDesc> desc;
    DevBuf<int32_t> list, counters;
    DevBuf<int32_t> perm;                            // Bunch-Kaufman pivoting only: FactorArgs::perm / pkind / rot
    DevBuf<int8_t> pkind;
    DevBuf<double> rot;
    int32_t* h_counters = nullptr;
    cudaGraphExec_t g_factor = nullptr;
    cudaStream_t cap_stream = nullptr;
    bool factorized = false;
    ~b2d_solver() {
        if (g_factor) cudaGraphExecDestroy(g_factor);
        for (auto e : ev_pool) cudaEventDestroy(e);
        if (aux_stream) cudaStreamDestroy(aux_stream);
        if (side_stream) cudaStreamDestroy(side_stream);
        if (cap_stream) cudaStreamDestroy(cap_stream);
        if (h_counters) cudaFreeHost(h_counters);
    }
};

namespace {
__global__ void k_copy_lower(int N, int lda, const double* __restrict__ A, double* __restrict__ F) {
    const int j = blockIdx.y;
    for (int i = j + blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x)
        F[(size_t)j * N + i] = A[(size_t)j * lda + i];
}

FactorArgs dense_factor_args(b2d_solver* s) {
    FactorArgs a;
    a.desc = s->desc.p; a.child_idx = nullptr; a.rel = nullptr; a.amap_src = nullptr; a.amap_dst = nullptr;
    a.A = nullptr; a.L = s->fact.p; a.ws = nullptr; a.dvec = s->dvec.p; a.counters = s->counters.p; a.eps = s->opt.pivot_eps;
    a.perm = s->perm.p; a.pkind = s->pkind.p; a.rot = s->rot.p;       // (nullptr unless pivoting)
    return a;
}

void enqueue_dense_factor_lookahead(b2d_solver* s, cudaStream_t S1) {
    FactorArgs a = dense_factor_args(s);
    const int N = s->N, nb = (N + DB - 1) / DB;
    if (s->trace.p) {
        a.trace = s->trace.p;
        k_trace_reset<<<(16 * nb + 255) / 256, 256, 0, S1>>>(s->trace.p, 8 * nb);
    }
    cudaMemsetAsync(s->counters.p, 0, 2 * sizeof(int32_t), S1);
    cudaMemsetAsync(s->tilecnt.p, 0, s->tilecnt.bytes(), S1);
    k_copy_lower<<<dim3(std::max(1, std::min(8, (N + 255) / 256)), N), 256, 0, S1>>>(N, s->lda, s->A_d, s->fact.p);
    LookaheadCtx cx;
    cx.S2 = s->aux_stream; cx.S3 = s->side_stream; cx.pool = &s->ev_pool; s->ev_next = 0; cx.next = &s->ev_next; cx.tilecnt = s->tilecnt.p;
    enqueue_front_lookahead(a, s->list.p, N, N, s->linv.p, s->linv_off.p, cx, S1);
}

void enqueue_dense_factor(b2d_solver* s, cudaStream_t st) {
    static int lookahead = -1;
    if (lookahead < 0) { const char* e = getenv("B2_DENSE_LOOKAHEAD"); lookahead = e ? (atoi(e) != 0) : 1; }
    const int N = s->N;
    if (lookahead && s->aux_stream && s->side_stream && N > 4 * DB) enqueue_dense_factor_lookahead(s, st);
    else {
        FactorArgs a = dense_factor_args(s);
        cudaMemsetAsync(s->counters.p, 0, 2 * sizeof(int32_t), st);     // [2] = sticky error flag of the dataflow solve
        k_copy_lower<<<dim3(std::max(1, std::min(8, (N + 255) / 256)), N), 256, 0, st>>>(N, s->lda, s->A_d, s->fact.p);
        for (int ob = 0; ob < N; ob += DB) launch_big_step(a, s->list.p, 1, ob, N, s->linv.p, s->linv_off.p, st, nullptr);
    }
    // Bunch-Kaufman: every block's interchanges reach the rows of the finished columns left of it
    if (s->perm.p && N > DB) k_bk_swap_left<<<dim3(((N - 1) / DB) * DB, (N - 1) / DB), DB, 0, st>>>(N, s->fact.p, s->perm.p);
}
}  // namespace

extern "C" {

int b2d_create(int32_t N, int32_t lda, const double* A_d, const b2_options* opt, b2d_solver** out) {
    if (!out || N <= 0 || lda < N || !A_d) { set_error("b2d_create: invalid argument"); return B2_ERR_INVALID; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        set_error("b2d_create: no CUDA device (this library has no CPU fallback)");
        return B2_ERR_NO_DEVICE;
    }
    b2_options o;
    if (opt) o = *opt; else b2_options_default(&o);
    if (o.pivoting != B2_PIVOT_STATIC && o.pivoting != B2_PIVOT_BUNCH_KAUFMAN) { set_error("b2d_create: unknown pivoting mode"); return B2_ERR_INVALID; }
    // the pivoted solve is the single-launch dataflow kernel only: one resident CTA per 128-row block
    if (o.pivoting == B2_PIVOT_BUNCH_KAUFMAN && (N + DB - 1) / DB > sm_count()) {
        set_error("b2d_create: Bunch-Kaufman pivoting needs N <= 128 * (number of SMs) = " + std::to_string(DB * sm_count()));
        return B2_ERR_INVALID;
    }
    auto* s = new b2d_solver();
    s->N = N; s->lda = lda; s->A_d = A_d;
    s->opt = o;
    FrontDesc d;
    std::memset(&d, 0, sizeof(d));
    d.col0 = 0; d.w = N; d.f = N;
    int32_t zero = 0;
    int64_t zero64 = 0;
    if (s->side.alloc(N) != cudaSuccess || s->linv.alloc((size_t)((N + BS - 1) / BS) * BS * BS) != cudaSuccess || s->linv_off.upload(&zero64, 1) != cudaSuccess ||
        s->fact.alloc((size_t)N * N + 2) != cudaSuccess || s->dvec.alloc(N) != cudaSuccess ||
        s->flow.alloc((size_t)2 * ((N + BS - 1) / BS) * BS) != cudaSuccess || s->desc.upload(&d, 1) != cudaSuccess ||
        s->list.upload(&zero, 1) != cudaSuccess || s->counters.alloc(4) != cudaSuccess ||
        cudaMallocHost((void**)&s->h_counters, 4 * sizeof(int32_t)) != cudaSuccess ||
        cudaStreamCreateWithFlags(&s->cap_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&s->aux_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&s->side_stream, cudaStreamNonBlocking) != cudaSuccess ||
        s->tilecnt.alloc((size_t)((N + DB - 1) / DB)) != cudaSuccess ||
        (getenv("B2_DENSE_TRACE") && atoi(getenv("B2_DENSE_TRACE")) && s->trace.alloc((size_t)16 * ((N + DB - 1) / DB)) != cudaSuccess) ||
        cudaMemset(s->fact.p, 0, s->fact.bytes()) != cudaSuccess || cudaMemset(s->counters.p, 0, 4 * sizeof(int32_t)) != cudaSuccess ||
        (o.pivoting == B2_PIVOT_BUNCH_KAUFMAN &&
         (s->perm.alloc(N) != cudaSuccess || s->pkind.alloc(N) != cudaSuccess || s->rot.alloc(N) != cudaSuccess))) {
        delete s;
        return cuda_fail(cudaGetLastError(), "b2d_create allocation", __FILE__, __LINE__);
    }
    if (set_smem_attrs() != B2_OK) { delete s; return B2_ERR_CUDA; }
    *out = s;
    return B2_OK;
}

int b2d_destroy(b2d_solver* s) { delete s; return B2_OK; }

int b2d_factorize(b2d_solver* s, void* stream) {
    if (!s) return B2_ERR_INVALID;
    cudaStream_t st = as_stream(stream);
    if (s->opt.use_cuda_graph && !stream_is_capturing(st)) {
        if (!s->g_factor) {
            cudaGraph_t g = nullptr;
            B2_CUDA(cudaStreamBeginCapture(s->cap_stream, cudaStreamCaptureModeThreadLocal));
            enqueue_dense_factor(s, s->cap_stream);
            cudaError_t e = cudaStreamEndCapture(s->cap_stream, &g);
            if (e != cudaSuccess) return cuda_fail(e, "cudaStreamEndCapture", __FILE__, __LINE__);
            e = cudaGraphInstantiate(&s->g_factor, g, 0);
            cudaGraphDestroy(g);
            if (e != cudaSuccess) return cuda_fail(e, "cudaGraphInstantiate", __FILE__, __LINE__);
        }
        B2_CUDA(cudaGraphLaunch(s->g_factor, st));
    } else {
        enqueue_dense_factor(s, st);
        B2_CUDA(cudaGetLastError());
    }
    s->factorized = true;
    return B2_OK;
}

int b2d_debug_trace(b2d_solver* s, uint64_t* stamps_h, int64_t capacity, int64_t* count) {
    if (!s || !count) { set_error("b2d_debug_trace: invalid argument"); return B2_ERR_INVALID; }
    *count = (int64_t)s->trace.n;
    if (!s->trace.p || !stamps_h || capacity < (int64_t)s->trace.n) return B2_OK;      // (count = 0: tracing is off)
    B2_CUDA(cudaDeviceSynchronize());
    B2_CUDA(cudaMemcpy(stamps_h, s->trace.p, s->trace.bytes(), cudaMemcpyDeviceToHost));
    return B2_OK;
}

int b2d_inertia_enqueue(b2d_solver* s, void* stream) {
    if (!s || !s->factorized) { set_error("b2d_inertia: not factorized"); return B2_ERR_FACTORIZATION; }
    B2_CUDA(cudaMemcpyAsync(s->h_counters, s->counters.p, 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, as_stream(stream)));
    return B2_OK;
}

int b2d_inertia_fetch(b2d_solver* s, int64_t* num_pos, int64_t* num_zero, int64_t* num_neg) {
    if (!s || !s->factorized) { set_error("b2d_inertia: not factorized"); return B2_ERR_FACTORIZATION; }
    if (s->h_counters[2]) { set_error("b2d: a hand-off wait timed out inside the single-launch solve"); return B2_ERR_SOLVE; }
    const int64_t neg = s->h_counters[0], zero = s->h_counters[1];
    if (num_neg) *num_neg = neg;
    if (num_zero) *num_zero = zero;
    if (num_pos) *num_pos = (int64_t)s->N - neg - zero;
    return B2_OK;
}

int b2d_inertia(b2d_solver* s, int64_t* num_pos, int64_t* num_zero, int64_t* num_neg, void* stream) {
    int rc = b2d_inertia_enqueue(s, stream);
    if (rc != B2_OK) return rc;
    B2_CUDA(cudaStreamSynchronize(as_stream(stream)));
    return b2d_inertia_fetch(s, num_pos, num_zero, num_neg);
}

int b2d_solve(b2d_solver* s, double* x_d, int32_t nrhs, void* stream) {
    if (!s || !x_d || nrhs < 1) { set_error("b2d_solve: invalid argument"); return B2_ERR_INVALID; }
    if (!s->factorized) { set_error("b2d_solve: not factorized"); return B2_ERR_SOLVE; }
    cudaStream_t st = as_stream(stream);
    const int N = s->N;
    const int nblk = (N + BS - 1) / BS;
    static int flow_ok = -1;            // every CTA of the dataflow kernel must be resident: one per SM
    if (flow_ok < 0) {
        flow_ok = (cudaFuncSetAttribute(k_dense_solve_flow<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)DS_SMEM) == cudaSuccess &&
                   cudaFuncSetAttribute(k_dense_solve_flow<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)DS_SMEM) == cudaSuccess) ? 1 : 0;
        if (const char* e = getenv("B2_DENSE_SOLVE_FLOW")) flow_ok = flow_ok && atoi(e) != 0;
    }
    const bool piv = s->perm.p != nullptr;
    if (piv && !(flow_ok && nblk <= sm_count())) {
        set_error("b2d_solve: the Bunch-Kaufman factor is solved by the single-launch kernel only, which is unavailable");
        return B2_ERR_SOLVE;
    }
    for (int c = 0; c < nrhs; ++c) {
        double* x = x_d + (size_t)c * N;
        if (flow_ok && nblk <= sm_count()) {
            // ONE launch: block row / block column k is owned by CTA k, hand-off through sentinel-initialised vectors
            B2_CUDA(cudaMemsetAsync(s->flow.p, 0xFF, s->flow.bytes(), st));
            if (piv)
                k_dense_solve_flow<true><<<nblk, DS_NT, DS_SMEM, st>>>(N, s->fact.p, s->linv.p, s->dvec.p, x, s->flow.p, s->flow.p + (size_t)nblk * BS,
                                                                      s->counters.p + 2, s->perm.p, s->pkind.p, s->rot.p);
            else
                k_dense_solve_flow<false><<<nblk, DS_NT, DS_SMEM, st>>>(N, s->fact.p, s->linv.p, s->dvec.p, x, s->flow.p, s->flow.p + (size_t)nblk * BS,
                                                                       s->counters.p + 2, nullptr, nullptr, nullptr);
            continue;
        }
        BigSolveArgs bs;
        SolveArgs& a = bs.s;
        a.desc = s->desc.p; a.rows = nullptr; a.child_idx = nullptr; a.rel = nullptr; a.cbv_off = s->linv_off.p;   // single zero offset
        a.L = s->fact.p; a.Lt = nullptr; a.dvec = s->dvec.p; a.xp = x; a.cbv = nullptr;
        bs.Linv = s->linv.p; bs.linv_off = s->linv_off.p; bs.side = s->side.p;
        k_bs_head<<<1, BS_NT, 0, st>>>(bs, s->list.p, 0, 0);
        for (int b = 0; b < nblk; ++b) {
            const int rows = std::max(1, N - b * BS - 1);
            k_bs_fwd<<<dim3((rows + BSF_ROWS - 1) / BSF_ROWS, 1), BS_NT, 0, st>>>(bs, s->list.p, b);
        }
        k_bs_bwd_init<<<dim3((N + 7) / 8, 1), 256, 0, st>>>(bs, s->list.p);
        k_bs_head<<<1, BS_NT, 0, st>>>(bs, s->list.p, -1, 1);
        for (int b = nblk - 1; b >= 1; --b) k_bs_bwd<<<dim3(b, 1), BS_NT, 0, st>>>(bs, s->list.p, b);
        k_bs_bwd_finish<<<dim3((N + 255) / 256, 1), 256, 0, st>>>(bs, s->list.p);
    }
    B2_CUDA(cudaGetLastError());
    return B2_OK;
}

int b2d_pivot_info(b2d_solver* s, int32_t* perm_h, int8_t* kind_h, int64_t* n_2x2, int64_t* n_perturbed) {
    if (!s) { set_error("b2d_pivot_info: invalid argument"); return B2_ERR_INVALID; }
    if (!s->factorized) { set_error("b2d_pivot_info: not factorized"); return B2_ERR_FACTORIZATION; }
    B2_CUDA(cudaDeviceSynchronize());
    const int N = s->N;
    std::vector<int8_t> kind(N, (int8_t)B2_PIVOT_KIND_1X1);
    int64_t n2 = 0, np = 0;
    if (s->perm.p) {
        B2_CUDA(cudaMemcpy(kind.data(), s->pkind.p, N * sizeof(int8_t), cudaMemcpyDeviceToHost));
        if (perm_h) B2_CUDA(cudaMemcpy(perm_h, s->perm.p, N * sizeof(int32_t), cudaMemcpyDeviceToHost));
        for (int8_t k : kind) { n2 += k == B2_PIVOT_KIND_2X2_FIRST; np += k == B2_PIVOT_KIND_PERTURBED; }
    } else {
        int32_t c[2];
        B2_CUDA(cudaMemcpy(c, s->counters.p, sizeof(c), cudaMemcpyDeviceToHost));
        np = c[1];
        if (perm_h) for (int i = 0; i < N; ++i) perm_h[i] = i;
    }
    if (kind_h) std::memcpy(kind_h, kind.data(), N);
    if (n_2x2) *n_2x2 = n2;
    if (n_perturbed) *n_perturbed = np;
    return B2_OK;
}

}  // extern "C"
