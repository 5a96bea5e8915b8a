// direct.cu -- numeric sparse block Cholesky + triangular solves on the device (see direct.h).
//
// One kernel per LM trial does what LinearSolverEigen::solve [EXT g2o] does per trial (numeric LDL^T of
// Hpp + lambda I, two triangular solves; reference plug-in site kitti_surf.cpp:553-557):
//   scatter   L <- permuted (H + lambda I), fill-in blocks zeroed
//   per level (the independent sets of the multiple-minimum-degree order, direct_host.cpp):
//     gather  every block of the level's columns subtracts its ordered list of L_ij L_kj^T products
//     pivot   Cholesky of the level's d x d diagonal blocks, inverse of the triangular factor kept
//     scale   sub-diagonal blocks of the level's columns times L_kk^-T
//   forward / backward substitution level by level (8-lane group per block row, shuffles inside the group)
// Every block has one writer and a fixed summation order: bitwise reproducible.  Small factors (the KITTI-size
// graphs) run in ONE CTA with __syncthreads between phases -- the whole solve is one launch and no
// host round trip; larger ones run as a cooperative grid (one CTA per SM) with grid barriers.
#include <cooperative_groups.h>

#include <algorithm>
#include <climits>
#include <cstring>

#include "direct.h"
#include "problem.h"
#include "reduce.cuh"

namespace cg = cooperative_groups;

namespace s3o {

struct DirectDev {
    int n, nlev, nL;
    const int32_t *perm, *lev_ptr, *cptr, *brow, *bcol, *src, *upd_ptr, *upd_a, *upd_b, *row_ptr, *row_blk, *row_col;
    double *L;       // [nL][D*D]
    double *Linv;    // [n][D*D]   inverse of the lower-triangular pivot factors
    double *y;       // [n][D]     solve workspace, elimination order
    int *fail;
};

struct DirectState {
    DirectPlan plan;
    bool analyzed = false, available = false;
    int32_t *d_perm = nullptr, *d_lev_ptr = nullptr, *d_cptr = nullptr, *d_brow = nullptr, *d_bcol = nullptr, *d_src = nullptr;
    int32_t *d_upd_ptr = nullptr, *d_upd_a = nullptr, *d_upd_b = nullptr, *d_row_ptr = nullptr, *d_row_blk = nullptr, *d_row_col = nullptr;
    double *d_L = nullptr, *d_Linv = nullptr, *d_y = nullptr;
    int *d_fail = nullptr;
    int coop_grid = 0;          // CTAs of the cooperative launch (<= 1: single CTA)
    int wide_levels = 0;        // leading levels wide enough for the whole grid; the rest runs on CTA 0
    bool factored = false;
    // marginal covariances (direct_marginals), allocated on the first call
    int32_t *d_sel_ptr = nullptr, *d_sel_sig = nullptr;
    double *d_Sig = nullptr;    // [nL][D*D] selected inverse, laid out like L
    double *d_E = nullptr, *d_X = nullptr;      // [D][n*D] unit right-hand sides / solutions of one block column
    DevScalars *d_msc = nullptr;                // status of those solves (the LM's DevScalars stay untouched)
    int32_t *d_pick = nullptr, *d_crow = nullptr, *d_cdst = nullptr;
    double *d_out = nullptr;
    int out_cap = 0;            // pairs d_pick / d_crow / d_cdst / d_out hold
    std::vector<int32_t> col_ptr, col_id;       // the requested pairs off the pattern, by block column (marginals_open)
    uint64_t serial = 0;        // plan_and_upload's count: the plan's identity for gather lists kept elsewhere
    // the plan of the marginals under the forced cap, when the linear solver has none of its own (PCG)
    DirectState *marg = nullptr;
};

namespace {

constexpr int kDirectNT = 512;

// loads of data written earlier in the same kernel by other SMs must bypass the (non-coherent) L1
template <bool COOP> __device__ __forceinline__ double ldw(const double *p) { return COOP ? __ldcg(p) : *p; }

// ---- phases (all take the executing thread space: tid in [0, nthreads)) ---------------------------------------
// gather: every block of the level's columns subtracts its ordered list of L[a] L[b]^T products
template <int D, bool COOP>
__device__ __forceinline__ void dk_gather(const DirectDev &P, int lev, int tid, int nthreads) {
    constexpr int DD = D * D;
    const int c0 = P.lev_ptr[lev], c1 = P.lev_ptr[lev + 1];
    const int t0 = P.cptr[c0], t1 = P.cptr[c1];
    for (int item = tid; item < (t1 - t0) * DD; item += nthreads) {
        const int t = t0 + item / DD, e = item % DD;
        const int q0 = P.upd_ptr[t], q1 = P.upd_ptr[t + 1];
        if (q0 == q1) continue;
        const int r = e / D, c = e - r * D;
        double acc = ldw<COOP>(P.L + (size_t)t * DD + e);
        for (int q = q0; q < q1; ++q) {
            const double *La = P.L + (size_t)P.upd_a[q] * DD + r * D;
            const double *Lb = P.L + (size_t)P.upd_b[q] * DD + c * D;
            double s = 0;
#pragma unroll
            for (int m = 0; m < D; ++m) s += ldw<COOP>(La + m) * ldw<COOP>(Lb + m);
            acc -= s;
        }
        P.L[(size_t)t * DD + e] = acc;
    }
}

// lower Cholesky of one d x d pivot block and the inverse of the factor (one thread)
template <int D, bool COOP>
__device__ __forceinline__ void dk_pivot_one(const DirectDev &P, int k) {
    constexpr int DD = D * D;
    double *Ld = P.L + (size_t)P.cptr[k] * DD;
    double *Lik = P.Linv + (size_t)k * DD;
    double A[DD], Li[DD];
#pragma unroll
    for (int i = 0; i < DD; ++i) A[i] = ldw<COOP>(Ld + i);
    bool ok = true;
#pragma unroll
    for (int j = 0; j < D; ++j) {
        double djj = A[j * D + j];
#pragma unroll
        for (int m = 0; m < j; ++m) djj -= A[j * D + m] * A[j * D + m];
        if (!(djj > 0) || !isfinite(djj)) { ok = false; djj = 1; }
        const double ljj = sqrt(djj), inv = 1.0 / ljj;
        A[j * D + j] = ljj;
#pragma unroll
        for (int r = j + 1; r < D; ++r) {
            double v = A[r * D + j];
#pragma unroll
            for (int m = 0; m < j; ++m) v -= A[r * D + m] * A[j * D + m];
            A[r * D + j] = v * inv;
        }
    }
#pragma unroll
    for (int c = 0; c < D; ++c)
#pragma unroll
        for (int r = 0; r < D; ++r) {
            if (r < c) { Li[r * D + c] = 0; continue; }
            double v = (r == c) ? 1.0 : 0.0;
#pragma unroll
            for (int m = c; m < r; ++m) v -= A[r * D + m] * Li[m * D + c];
            Li[r * D + c] = v / A[r * D + r];
        }
#pragma unroll
    for (int r = 0; r < D; ++r)
#pragma unroll
        for (int c = 0; c < D; ++c) {
            Ld[r * D + c] = c <= r ? A[r * D + c] : 0.0;
            Lik[r * D + c] = Li[r * D + c];
        }
    if (!ok) *P.fail = 1;
}

// scale one row of a sub-diagonal block: L_ik[r,:] = A_ik[r,:] L_kk^-T
template <int D, bool COOP>
__device__ __forceinline__ void dk_scale_row(const DirectDev &P, int t, int r, const double *Lik) {
    constexpr int DD = D * D;
    double a[D];
    double *row = P.L + (size_t)t * DD + r * D;
#pragma unroll
    for (int m = 0; m < D; ++m) a[m] = ldw<COOP>(row + m);
#pragma unroll
    for (int c = 0; c < D; ++c) {
        double sacc = 0;
#pragma unroll
        for (int m = 0; m <= c; ++m) sacc += a[m] * ldw<COOP>(Lik + c * D + m);
        row[c] = sacc;
    }
}

// A level with many columns: one thread per pivot (32 pivots per warp instruction), barrier, then one thread per
// block row.  A level with few columns: one warp per column, lane 0 factors, the warp scales -- no barrier between.
template <int D, bool COOP, class Sync>
__device__ __forceinline__ void dk_pivot_scale(const DirectDev &P, int lev, int tid, int nthreads, Sync sync) {
    constexpr int DD = D * D;
    const int c0 = P.lev_ptr[lev], c1 = P.lev_ptr[lev + 1];
    const int nwarps = nthreads >> 5;
    if (c1 - c0 > 2 * nwarps) {
        for (int k = c0 + tid; k < c1; k += nthreads) dk_pivot_one<D, COOP>(P, k);
        sync();
        const int t0 = P.cptr[c0], t1 = P.cptr[c1];
        for (int item = tid; item < (t1 - t0) * D; item += nthreads) {
            const int t = t0 + item / D, r = item % D;
            const int k = P.bcol[t];
            if (P.brow[t] == k) continue;
            dk_scale_row<D, COOP>(P, t, r, P.Linv + (size_t)k * DD);
        }
        return;
    }
    const int warp = tid >> 5, lane = tid & 31;
    for (int k = c0 + warp; k < c1; k += nwarps) {
        if (lane == 0) { dk_pivot_one<D, COOP>(P, k); __threadfence(); }
        __syncwarp();
        const int nsub = P.cptr[k + 1] - P.cptr[k] - 1;
        for (int item = lane; item < nsub * D; item += 32)
            dk_scale_row<D, COOP>(P, P.cptr[k] + 1 + item / D, item % D, P.Linv + (size_t)k * DD);
    }
}

// forward substitution of one level: y_k = L_kk^-1 (b_perm(k) - sum_j L_kj y_j), a GL-lane group per block row
template <int D, bool COOP>
__device__ __forceinline__ void dk_forward(const DirectDev &P, int lev, const double *__restrict__ b, int tid, int nthreads) {
    constexpr int DD = D * D, GL = GroupLanes<D>::value;
    const int group = tid / GL, lane = tid % GL, ngroups = nthreads / GL;
    const int c0 = P.lev_ptr[lev], c1 = P.lev_ptr[lev + 1];
    for (int kb = c0; kb < c1; kb += ngroups) {       // uniform trip count: the shuffles below stay convergent
        const int k = kb + group;
        const bool act = k < c1 && lane < D;
        double acc = 0;
        if (act) {
            acc = b[(size_t)P.perm[k] * D + lane];
            for (int q = P.row_ptr[k]; q < P.row_ptr[k + 1]; ++q) {
                const double *Lt = P.L + (size_t)P.row_blk[q] * DD + lane * D;
                const double *yj = P.y + (size_t)P.row_col[q] * D;
                double s = 0;
#pragma unroll
                for (int m = 0; m < D; ++m) s += ldw<COOP>(Lt + m) * ldw<COOP>(yj + m);
                acc -= s;
            }
        }
        double yl = 0;
#pragma unroll
        for (int m = 0; m < D; ++m) {
            const double am = __shfl_sync(0xffffffffu, acc, m, GL);
            if (act && m <= lane) yl += ldw<COOP>(P.Linv + (size_t)k * DD + lane * D + m) * am;
        }
        if (act) P.y[(size_t)k * D + lane] = yl;
    }
}

// backward substitution of one level: x_k = L_kk^-T (y_k - sum_i L_ik^T x_i), written in Hessian order as well
template <int D, bool COOP>
__device__ __forceinline__ void dk_backward(const DirectDev &P, int lev, double *__restrict__ x, int tid, int nthreads) {
    constexpr int DD = D * D, GL = GroupLanes<D>::value;
    const int group = tid / GL, lane = tid % GL, ngroups = nthreads / GL;
    const int c0 = P.lev_ptr[lev], c1 = P.lev_ptr[lev + 1];
    for (int kb = c0; kb < c1; kb += ngroups) {
        const int k = kb + group;
        const bool act = k < c1 && lane < D;
        double acc = 0;
        if (act) {
            acc = ldw<COOP>(P.y + (size_t)k * D + lane);
            for (int t = P.cptr[k] + 1; t < P.cptr[k + 1]; ++t) {
                const double *Lt = P.L + (size_t)t * DD + lane;
                const double *xi = P.y + (size_t)P.brow[t] * D;
                double s = 0;
#pragma unroll
                for (int m = 0; m < D; ++m) s += ldw<COOP>(Lt + m * D) * ldw<COOP>(xi + m);
                acc -= s;
            }
        }
        double xl = 0;
#pragma unroll
        for (int m = 0; m < D; ++m) {
            const double am = __shfl_sync(0xffffffffu, acc, m, GL);
            if (act && m >= lane) xl += ldw<COOP>(P.Linv + (size_t)k * DD + m * D + lane) * am;
        }
        if (act) {
            P.y[(size_t)k * D + lane] = xl;
            x[(size_t)P.perm[k] * D + lane] = xl;
        }
    }
}

// Schedule.  The first `wide` levels (the rounds that eliminate many columns at once) run on the whole grid with
// grid barriers; the narrow tail -- most of the rounds, each a handful of blocks -- runs on CTA 0 alone with CTA
// barriers while the other CTAs wait at ONE grid barrier.  Per level: [gather(l) + forward(l-1)] | pivot+scale(l);
// the forward substitution of a level only needs that level's pivots, so it rides in the next gather phase.
//   COOP = false: one CTA, wide = 0.
template <int D, bool COOP>
__global__ void __launch_bounds__(kDirectNT) direct_kernel(DirectDev P, const double *__restrict__ H, double lambda,
                                                           const double *__restrict__ b, double *__restrict__ x,
                                                           DevScalars *sc, int do_factor, int wide, const GridBarrier gb) {
    constexpr int DD = D * D;
    unsigned phase = 0;
    const int ltid = threadIdx.x;
    const int gtid = blockIdx.x * kDirectNT + threadIdx.x, gthreads = gridDim.x * kDirectNT;
    auto gsync = [&]() {
        if constexpr (COOP) grid_barrier(gb, phase);
        else __syncthreads();
    };
    if (do_factor) {
        if (gtid == 0) *P.fail = 0;
        // ---- scatter (H + lambda I) into the factor's storage, elimination order
        for (long long item = gtid; item < (long long)P.nL * DD; item += gthreads) {
            const int t = (int)(item / DD), e = (int)(item - (long long)t * DD);
            const int r = e / D, c = e - r * D;
            const int s = P.src[t];
            double v = 0;
            if (s >= 0) {
                const double *Hb = H + (size_t)(s >> 1) * DD;
                v = (s & 1) ? Hb[c * D + r] : Hb[e];
            }
            if (r == c && P.brow[t] == P.bcol[t]) v += lambda;
            P.L[item] = v;
        }
        gsync();
    }
    // ---- wide levels on the whole grid
    for (int lev = 0; lev < wide; ++lev) {
        if (do_factor) dk_gather<D, COOP>(P, lev, gtid, gthreads);
        if (lev > 0) dk_forward<D, COOP>(P, lev - 1, b, gtid, gthreads);
        if (do_factor || lev > 0) gsync();
        if (do_factor) { dk_pivot_scale<D, COOP>(P, lev, gtid, gthreads, gsync); gsync(); }
    }
    // ---- narrow tail on CTA 0 (CTA barriers), then its share of the backward substitution
    if (blockIdx.x == 0) {
        for (int lev = wide; lev < P.nlev; ++lev) {
            if (do_factor) dk_gather<D, COOP>(P, lev, ltid, kDirectNT);
            if (lev > 0) dk_forward<D, COOP>(P, lev - 1, b, ltid, kDirectNT);
            __syncthreads();
            if (do_factor) { dk_pivot_scale<D, COOP>(P, lev, ltid, kDirectNT, [] { __syncthreads(); }); __syncthreads(); }
        }
        if (P.nlev > 0) {
            if (wide == P.nlev) { /* the last level's forward step still runs on the grid below */ }
            else { dk_forward<D, COOP>(P, P.nlev - 1, b, ltid, kDirectNT); __syncthreads(); }
        }
        for (int lev = P.nlev - 1; lev >= wide; --lev) { dk_backward<D, COOP>(P, lev, x, ltid, kDirectNT); __syncthreads(); }
    }
    if (wide > 0) {
        if (wide == P.nlev) { dk_forward<D, COOP>(P, P.nlev - 1, b, gtid, gthreads); }
        gsync();
        for (int lev = wide - 1; lev >= 0; --lev) { dk_backward<D, COOP>(P, lev, x, gtid, gthreads); gsync(); }
    }
    if (gtid == 0) {     // the PCG bookkeeping the LM driver reads: an exact solve, 0 iterations
        const int failed = *reinterpret_cast<volatile int *>(P.fail);
        sc->done = failed ? 3 : 1;
        sc->iters = 0;
        sc->rr = 0;
        sc->rr0 = 1;
    }
}

// ---- selected inverse (Takahashi recurrences): Sigma = H^-1 on the pattern of L, from the factor --------------
// Sigma L = L^-T (upper triangular) gives, column j of L with sub-diagonal row set S(j),
//   Sigma_ij = -(sum_{k in S(j)} Sigma_ik L_kj) L_jj^-1                  i in S(j)
//   Sigma_jj = L_jj^-T (L_jj^-1 - sum_{k in S(j)} L_kj^T Sigma_kj)
// Every Sigma_ik read by column j has i, k in S(j), i.e. belongs to a strictly later round (a round is an independent
// set), so the rounds run in reverse, each in two phases: its off-diagonal blocks, then its diagonal blocks.
struct SelinvDev {
    const int32_t *sel_ptr, *sel_sig;      // selinv_lists (direct_host.cpp)
    double *Sig;                           // [nL][D*D]
};

// off-diagonal blocks of the level's columns, one thread per block row: its D sums in registers, fixed order
template <int D, bool COOP>
__device__ __forceinline__ void sk_offdiag(const DirectDev &P, const SelinvDev &S, int lev, int tid, int nthreads) {
    constexpr int DD = D * D;
    const int c0 = P.lev_ptr[lev], c1 = P.lev_ptr[lev + 1];
    const int t0 = P.cptr[c0], t1 = P.cptr[c1];
    for (int item = tid; item < (t1 - t0) * D; item += nthreads) {
        const int t = t0 + item / D, r = item % D;
        const int j = P.bcol[t];
        if (P.brow[t] == j) continue;
        double acc[D];
#pragma unroll
        for (int c = 0; c < D; ++c) acc[c] = 0;
        const double *Lk = P.L + (size_t)(P.cptr[j] + 1) * DD;      // L_kj of the operands, in list order
        for (int q = S.sel_ptr[t]; q < S.sel_ptr[t + 1]; ++q, Lk += DD) {
            const int s = S.sel_sig[q];
            const double *Sb = S.Sig + (size_t)(s >> 1) * DD;
            double a[D];                                             // row r of Sigma_ik
            if (s & 1) {
#pragma unroll
                for (int m = 0; m < D; ++m) a[m] = ldw<COOP>(Sb + m * D + r);
            } else {
#pragma unroll
                for (int m = 0; m < D; ++m) a[m] = ldw<COOP>(Sb + r * D + m);
            }
#pragma unroll
            for (int m = 0; m < D; ++m)
#pragma unroll
                for (int c = 0; c < D; ++c) acc[c] += a[m] * Lk[m * D + c];
        }
        const double *Li = P.Linv + (size_t)j * DD;                  // lower triangular
        double *out = S.Sig + (size_t)t * DD + r * D;
#pragma unroll
        for (int c = 0; c < D; ++c) {
            double v = 0;
#pragma unroll
            for (int m = c; m < D; ++m) v += acc[m] * Li[m * D + c];
            out[c] = -v;
        }
    }
}

// diagonal blocks of the level's columns, one thread per block column c: W[:, c] = L_jj^-1[:, c] - sum L_kj^T Sigma_kj[:, c],
// then Sigma_jj[r, c] = (L_jj^-T W)[r, c] for r >= c, written to (r, c) and (c, r): exactly symmetric
template <int D, bool COOP>
__device__ __forceinline__ void sk_diag(const DirectDev &P, const SelinvDev &S, int lev, int tid, int nthreads) {
    constexpr int DD = D * D;
    const int c0 = P.lev_ptr[lev], c1 = P.lev_ptr[lev + 1];
    for (int item = tid; item < (c1 - c0) * D; item += nthreads) {
        const int j = c0 + item / D, c = item % D;
        const double *Li = P.Linv + (size_t)j * DD;
        double w[D];
#pragma unroll
        for (int m = 0; m < D; ++m) w[m] = Li[m * D + c];
        for (int t = P.cptr[j] + 1; t < P.cptr[j + 1]; ++t) {
            const double *Lb = P.L + (size_t)t * DD, *Sb = S.Sig + (size_t)t * DD;
            double sc[D];
#pragma unroll
            for (int q = 0; q < D; ++q) sc[q] = ldw<COOP>(Sb + q * D + c);
#pragma unroll
            for (int m = 0; m < D; ++m) {
                double v = 0;
#pragma unroll
                for (int q = 0; q < D; ++q) v += Lb[q * D + m] * sc[q];
                w[m] -= v;
            }
        }
        double *out = S.Sig + (size_t)P.cptr[j] * DD;
#pragma unroll
        for (int r = 0; r < D; ++r) {
            if (r < c) continue;
            double v = 0;
#pragma unroll
            for (int m = r; m < D; ++m) v += Li[m * D + r] * w[m];
            out[r * D + c] = v;
            out[c * D + r] = v;
        }
    }
}

// Schedule of the backward substitution: the narrow tail rounds (the last ones eliminated, so the first ones here) on
// CTA 0 with CTA barriers while the other CTAs wait at one grid barrier, then the wide leading rounds on the grid.
// Reads the factor of the preceding direct_kernel launch (L, Linv are read-only here).
template <int D, bool COOP>
__global__ void __launch_bounds__(kDirectNT, 1) selinv_kernel(DirectDev P, SelinvDev S, int wide, const GridBarrier gb) {
    unsigned phase = 0;
    const int ltid = threadIdx.x;
    const int gtid = blockIdx.x * kDirectNT + threadIdx.x, gthreads = gridDim.x * kDirectNT;
    auto gsync = [&]() {
        if constexpr (COOP) grid_barrier(gb, phase);
        else __syncthreads();
    };
    if (blockIdx.x == 0)
        for (int lev = P.nlev - 1; lev >= wide; --lev) {
            sk_offdiag<D, COOP>(P, S, lev, ltid, kDirectNT);
            __syncthreads();
            sk_diag<D, COOP>(P, S, lev, ltid, kDirectNT);
            __syncthreads();
        }
    if (wide > 0) {
        gsync();
        for (int lev = wide - 1; lev >= 0; --lev) {
            sk_offdiag<D, COOP>(P, S, lev, gtid, gthreads);
            gsync();
            sk_diag<D, COOP>(P, S, lev, gtid, gthreads);
            if (lev > 0) gsync();
        }
    }
}

// requested blocks on the pattern: out[k] = Sigma block pick[k] >> 1 (transposed if pick[k] & 1); pick[k] < 0: skip
template <int D>
__global__ void marg_pick_kernel(const double *__restrict__ Sig, const int32_t *__restrict__ pick, int n_pairs,
                                 double *__restrict__ out) {
    constexpr int DD = D * D;
    for (long long item = blockIdx.x * (long long)blockDim.x + threadIdx.x; item < (long long)n_pairs * DD;
         item += (long long)gridDim.x * blockDim.x) {
        const int k = (int)(item / DD), e = (int)(item - (long long)k * DD);
        const int s = pick[k];
        if (s < 0) continue;
        const int a = e / D, b = e - a * D;
        out[item] = Sig[(size_t)(s >> 1) * DD + ((s & 1) ? b * D + a : e)];
    }
}

// D unit right-hand sides of block column `col`: E[m][i] = (i == col * D + m)
__global__ void marg_unit_kernel(double *__restrict__ E, int nd, int D, int col) {
    for (long long item = blockIdx.x * (long long)blockDim.x + threadIdx.x; item < (long long)nd * D;
         item += (long long)gridDim.x * blockDim.x) {
        const int m = (int)(item / nd), i = (int)(item - (long long)m * nd);
        E[item] = (i == col * D + m) ? 1.0 : 0.0;
    }
}

// requested blocks (row[q], col) of one solved block column: out[dst[q]][a][b] = X[b][row[q] * D + a]
template <int D>
__global__ void marg_column_kernel(const double *__restrict__ X, int nd, const int32_t *__restrict__ row,
                                   const int32_t *__restrict__ dst, int cnt, double *__restrict__ out) {
    constexpr int DD = D * D;
    for (int item = blockIdx.x * blockDim.x + threadIdx.x; item < cnt * DD; item += gridDim.x * blockDim.x) {
        const int q = item / DD, e = item - q * DD;
        const int a = e / D, b = e - a * D;
        out[(size_t)dst[q] * DD + e] = X[(size_t)b * nd + (size_t)row[q] * D + a];
    }
}

DirectDev device_view(const DirectState *D) {
    const DirectPlan &Pl = D->plan;
    DirectDev P{};
    P.n = Pl.n; P.nlev = Pl.nlev; P.nL = (int)Pl.brow.size();
    P.perm = D->d_perm; P.lev_ptr = D->d_lev_ptr; P.cptr = D->d_cptr; P.brow = D->d_brow; P.bcol = D->d_bcol; P.src = D->d_src;
    P.upd_ptr = D->d_upd_ptr; P.upd_a = D->d_upd_a; P.upd_b = D->d_upd_b;
    P.row_ptr = D->d_row_ptr; P.row_blk = D->d_row_blk; P.row_col = D->d_row_col;
    P.L = D->d_L; P.Linv = D->d_Linv; P.y = D->d_y; P.fail = D->d_fail;
    return P;
}

template <class T>
int up(s3o_problem *p, T **dst, const std::vector<T> &src) { return upload(p, dst, src); }

void free_direct_arrays(DirectState *D) {
    dev_free(D->d_perm); dev_free(D->d_lev_ptr); dev_free(D->d_cptr); dev_free(D->d_brow); dev_free(D->d_bcol); dev_free(D->d_src);
    dev_free(D->d_upd_ptr); dev_free(D->d_upd_a); dev_free(D->d_upd_b); dev_free(D->d_row_ptr); dev_free(D->d_row_blk);
    dev_free(D->d_row_col); dev_free(D->d_L); dev_free(D->d_Linv); dev_free(D->d_y); dev_free(D->d_fail);
    dev_free(D->d_sel_ptr); dev_free(D->d_sel_sig); dev_free(D->d_Sig); dev_free(D->d_E); dev_free(D->d_X); dev_free(D->d_msc);
    dev_free(D->d_pick); dev_free(D->d_crow); dev_free(D->d_cdst); dev_free(D->d_out);
    D->out_cap = 0;
}

// one factorisation (do_factor) and/or solve of (H + lambda I) x = b with the plan of S; status in *sc
template <int D>
int launch_direct(s3o_problem *p, const DirectState *S, const DirectDev &P, double lambda, int do_factor,
                  const double *b, double *x, DevScalars *sc) {
    if (S->coop_grid <= 1) {
        direct_kernel<D, false><<<1, kDirectNT, 0, p->stream>>>(P, p->d_H, lambda, b, x, sc, do_factor, 0, GridBarrier{});
        return S3O_OK;
    }
    const double *H = p->d_H;
    DirectDev Pc = P;
    int wide = S->wide_levels;
    GridBarrier gb{};
    void *args[] = { &Pc, &H, &lambda, &b, &x, &sc, &do_factor, &wide, &gb };
    return launch_persistent(p, (const void *)direct_kernel<D, true>, S->coop_grid, kDirectNT, args, 9);
}

template <int D>
int launch_selinv(s3o_problem *p, const DirectState *S, const DirectDev &P, const SelinvDev &Sv) {
    if (S->coop_grid <= 1) {
        selinv_kernel<D, false><<<1, kDirectNT, 0, p->stream>>>(P, Sv, 0, GridBarrier{});
        return S3O_OK;
    }
    DirectDev Pc = P;
    SelinvDev Sc = Sv;
    int wide = S->wide_levels;
    GridBarrier gb{};
    void *args[] = { &Pc, &Sc, &wide, &gb };
    return launch_persistent(p, (const void *)selinv_kernel<D, true>, S->coop_grid, kDirectNT, args, 4);
}

template <int D>
int coop_capacity(int device) {
    int per_sm = 0, sms = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, direct_kernel<D, true>, kDirectNT, 0) != cudaSuccess) return 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) return 0;
    // (selinv_kernel runs on the same grid: it has the same launch bounds and no shared memory, so it fits as well)
    return per_sm > 0 ? sms : 0;      // one CTA per SM
}

}  // namespace

void direct_destroy(s3o_problem *p) {
    if (!p->direct) return;
    if (DirectState *M = p->direct->marg) { free_direct_arrays(M); delete M; }
    free_direct_arrays(p->direct);
    delete p->direct;
    p->direct = nullptr;
}

// Block products above which the AUTO rule stays with PCG / above which the analysis is abandoned.
static constexpr long long kAutoMaxPairs = 400000, kForcedMaxPairs = 60000000;
static constexpr int kAutoMaxLevels = 128;

// Symbolic analysis of p->S into D under the limits and upload; D->available says whether the plan stayed within them.
static int plan_and_upload(s3o_problem *p, DirectState *D, long long max_pairs, int max_levels) {
    static uint64_t plans = 0;
    D->serial = ++plans;
    D->analyzed = true;
    D->available = false;
    if (!direct_analyze(p->S.nf, p->S.rowptr, p->S.colidx, max_pairs, D->plan)) return S3O_OK;
    const DirectPlan &P = D->plan;
    if (P.nlev > max_levels) return S3O_OK;
    const int nL = (int)P.brow.size(), d = p->d;
    std::vector<int32_t> bcol(nL);
    for (int j = 0; j < P.n; ++j)
        for (int t = P.cptr[j]; t < P.cptr[j + 1]; ++t) bcol[t] = j;
    int rc = 0;
    rc = rc ? rc : up(p, &D->d_perm, P.perm);
    rc = rc ? rc : up(p, &D->d_lev_ptr, P.lev_ptr);
    rc = rc ? rc : up(p, &D->d_cptr, P.cptr);
    rc = rc ? rc : up(p, &D->d_brow, P.brow);
    rc = rc ? rc : up(p, &D->d_bcol, bcol);
    rc = rc ? rc : up(p, &D->d_src, P.src);
    rc = rc ? rc : up(p, &D->d_upd_ptr, P.upd_ptr);
    rc = rc ? rc : up(p, &D->d_upd_a, P.upd_a);
    rc = rc ? rc : up(p, &D->d_upd_b, P.upd_b);
    rc = rc ? rc : up(p, &D->d_row_ptr, P.row_ptr);
    rc = rc ? rc : up(p, &D->d_row_blk, P.row_blk);
    rc = rc ? rc : up(p, &D->d_row_col, P.row_col);
    rc = rc ? rc : dev_alloc(&D->d_L, (size_t)nL * d * d);
    rc = rc ? rc : dev_alloc(&D->d_Linv, (size_t)P.n * d * d);
    rc = rc ? rc : dev_alloc(&D->d_y, (size_t)P.n * d);
    rc = rc ? rc : dev_alloc(&D->d_fail, 1);
    if (rc) { free_direct_arrays(D); return rc; }
    S3O_CUDA(cudaStreamSynchronize(p->stream));
    // Grid and schedule: a level is "wide" while its gather phase has more than 8 items per thread of one CTA;
    // the leading wide levels run on a cooperative grid sized for the widest one, everything after the last wide
    // level on CTA 0 alone (CTA barriers are ~10x cheaper than grid barriers, and the tail is pure latency).
    D->coop_grid = 0;
    D->wide_levels = 0;
    {
        long long widest = 0;
        for (int l = 0; l < P.nlev; ++l) {
            const long long items = (long long)(P.cptr[P.lev_ptr[l + 1]] - P.cptr[P.lev_ptr[l]]) * d * d;
            if (items > 8 * kDirectNT) D->wide_levels = l + 1;
            widest = std::max(widest, items);
        }
        if (D->wide_levels > 0) {
            int cap = 0;
            switch (d) {
            case 7: cap = coop_capacity<7>(p->device); break;
            case 6: cap = coop_capacity<6>(p->device); break;
            case 4: cap = coop_capacity<4>(p->device); break;
            case 1: cap = coop_capacity<1>(p->device); break;
            }
            const long long want = (widest + 4 * kDirectNT - 1) / (4 * kDirectNT);
            D->coop_grid = (int)std::max<long long>(1, std::min<long long>(cap, want));
            if (D->coop_grid <= 1) D->wide_levels = 0;
        }
    }
    D->available = true;
    D->factored = false;
    return S3O_OK;
}

// Symbolic analysis + upload, once per structure.  Returns S3O_OK also when the factor is too large
// (direct_available() then says no).
int direct_setup(s3o_problem *p) {
    if (p->direct && p->direct->analyzed) return S3O_OK;
    if (!p->direct) p->direct = new DirectState();
    DirectState *D = p->direct;
    D->analyzed = true;
    D->available = false;
    if (p->dist || p->S.nf == 0) return S3O_OK;
    const bool forced = p->linsolver == S3O_LINSOLVER_DIRECT;
    // AUTO: a factor within kAutoMaxPairs block products cannot have more than ~kAutoMaxPairs / 3 columns (a chain
    // costs 3 products per column), so larger graphs go to the PCG without paying for the analysis
    if (!forced && p->S.nf > kAutoMaxPairs / 3) return S3O_OK;
    const int rc = plan_and_upload(p, D, forced ? kForcedMaxPairs : kAutoMaxPairs, forced ? INT_MAX : kAutoMaxLevels);
    if (rc || !D->available) return rc;
    p->stats.direct_levels = D->plan.nlev;
    p->stats.direct_blocks = (int)D->plan.brow.size();
    return S3O_OK;
}

bool direct_available(const s3o_problem *p) { return p->direct && p->direct->available; }
void direct_invalidate(s3o_problem *p) { if (p->direct) p->direct->factored = false; }

// Solve (H + lambda I) x = b exactly: numeric factorisation (skipped when reuse_factor and a factor of the
// same system is still held) + both triangular solves, one launch.  x in p->d_x; status through DevScalars.
int direct_solve(s3o_problem *p, double lambda, bool reuse_factor) {
    DirectState *D = p->direct;
    if (!D || !D->available) { set_error("direct_solve: no factorisation plan"); return S3O_ERR_INVALID; }
    const DirectDev P = device_view(D);
    const int do_factor = (reuse_factor && D->factored) ? 0 : 1;
    int rc = S3O_OK;
    switch (p->d) {
    case 7: rc = launch_direct<7>(p, D, P, lambda, do_factor, p->d_b, p->d_x, p->d_sc); break;
    case 6: rc = launch_direct<6>(p, D, P, lambda, do_factor, p->d_b, p->d_x, p->d_sc); break;
    case 4: rc = launch_direct<4>(p, D, P, lambda, do_factor, p->d_b, p->d_x, p->d_sc); break;
    case 1: rc = launch_direct<1>(p, D, P, lambda, do_factor, p->d_b, p->d_x, p->d_sc); break;
    default: set_error("direct_solve: block dimension %d", p->d); return S3O_ERR_UNSUPPORTED;
    }
    if (rc) return rc;
    D->factored = true;
    p->stats.direct_solves += 1;
    return check_launch(p, 1);
}

namespace {

// factorisation of H without damping and its selected inverse; ev (may be nullptr): 2 events, after each
template <int D>
int factor_launches(s3o_problem *p, DirectState *S, cudaEvent_t *ev) {
    const DirectDev P = device_view(S);
    const SelinvDev Sv{ S->d_sel_ptr, S->d_sel_sig, S->d_Sig };
    int rc = launch_direct<D>(p, S, P, 0.0, 1, S->d_E, S->d_X, S->d_msc);     // H = L L^T (no damping)
    if (rc) return rc;
    if (ev) cudaEventRecord(ev[0], p->stream);
    if ((rc = launch_selinv<D>(p, S, P, Sv))) return rc;
    if (ev) cudaEventRecord(ev[1], p->stream);
    return check_launch(p, 2);
}

// the requested blocks into d_out: on the pattern from the selected inverse, off it from column solves
template <int D>
int pick_launches(s3o_problem *p, DirectState *S, int n_pairs) {
    const DirectDev P = device_view(S);
    const std::vector<int32_t> &col_ptr = S->col_ptr, &col_id = S->col_id;
    const int nd = S->plan.n * D;
    int rc, launches = 0;
    if (n_pairs > 0) {
        const int grid = (int)std::min<long long>(1024, ((long long)n_pairs * D * D + 255) / 256);
        marg_pick_kernel<D><<<grid, 256, 0, p->stream>>>(S->d_Sig, S->d_pick, n_pairs, S->d_out);
        ++launches;
    }
    // pairs off the pattern of L: H X = E_c for each distinct block column c, D solves with the factor above
    for (size_t g = 0; g + 1 < col_ptr.size(); ++g) {
        marg_unit_kernel<<<(int)std::min<long long>(1024, ((long long)nd * D + 255) / 256), 256, 0, p->stream>>>(S->d_E, nd, D, col_id[g]);
        for (int m = 0; m < D; ++m)
            if ((rc = launch_direct<D>(p, S, P, 0.0, 0, S->d_E + (size_t)m * nd, S->d_X + (size_t)m * nd, S->d_msc))) return rc;
        const int cnt = col_ptr[g + 1] - col_ptr[g];
        marg_column_kernel<D><<<std::min(1024, (cnt * D * D + 255) / 256), 256, 0, p->stream>>>(
            S->d_X, nd, S->d_crow + col_ptr[g], S->d_cdst + col_ptr[g], cnt, S->d_out);
        launches += D + 2;
    }
    return check_launch(p, launches);
}

void free_marginal_arrays(DirectState *S) {
    dev_free(S->d_sel_ptr); dev_free(S->d_sel_sig); dev_free(S->d_Sig); dev_free(S->d_E); dev_free(S->d_X); dev_free(S->d_msc);
}

}  // namespace

// The plan of the marginals: the linear solver's own when it has one (the same analysis, only the size limits
// differ), otherwise one under the forced cap kept for the marginals -- the choice of the linear solver does not move.
// *S = nullptr when the factor exceeds the forced cap (the analysis is run once and its verdict kept).
static int marginals_plan(s3o_problem *p, DirectState **S) {
    *S = nullptr;
    int rc;
    if (p->linsolver != S3O_LINSOLVER_PCG) {
        if ((rc = direct_setup(p))) return rc;
        if (direct_available(p)) { *S = p->direct; return S3O_OK; }
    }
    if (!p->direct) p->direct = new DirectState();
    DirectState *&M = p->direct->marg;
    if (!M) {
        M = new DirectState();
        if ((rc = plan_and_upload(p, M, kForcedMaxPairs, INT_MAX))) { delete M; M = nullptr; return rc; }
    }
    if (M->available) *S = M;
    return S3O_OK;
}

int marginals_iterative(s3o_problem *p, bool *iterative) {
    // S3O_MARGINALS_ROUTE=pcg: the iterative route also where the factor fits (both routes on the same H)
    const char *route = getenv("S3O_MARGINALS_ROUTE");
    if (route && !strcmp(route, "pcg")) { *iterative = true; return S3O_OK; }
    DirectState *S = nullptr;
    const int rc = marginals_plan(p, &S);
    *iterative = !rc && !S;
    return rc;
}

// Plan, buffers and pair lists of one marginals call (see problem.h).
int marginals_open(s3o_problem *p, const char *who, int n_pairs, const int32_t *rows, const int32_t *cols, MarginalsRun *R) {
    DirectState *S = nullptr;
    int rc;
    if ((rc = marginals_plan(p, &S))) return rc;
    if (!S) {
        set_error("%s: the factor of this graph needs more than %lld block products", who, kForcedMaxPairs);
        return S3O_ERR_UNSUPPORTED;
    }
    const DirectPlan &Pl = S->plan;
    const int n = Pl.n, d = p->d, dd = d * d;
    if (!S->d_Sig) {      // first marginals call on this plan: gather lists and buffers
        std::vector<int32_t> sel_ptr, sel_sig;
        selinv_lists(Pl, sel_ptr, sel_sig);
        rc = up(p, &S->d_sel_ptr, sel_ptr);
        rc = rc ? rc : up(p, &S->d_sel_sig, sel_sig);
        rc = rc ? rc : dev_alloc(&S->d_E, (size_t)n * dd);
        rc = rc ? rc : dev_alloc(&S->d_X, (size_t)n * dd);
        rc = rc ? rc : dev_alloc(&S->d_msc, 1);
        rc = rc ? rc : dev_alloc(&S->d_Sig, Pl.brow.size() * dd);
        if (!rc && cudaMemsetAsync(S->d_E, 0, sizeof(double) * n * dd, p->stream) != cudaSuccess) rc = S3O_ERR_CUDA;
        if (!rc && cudaStreamSynchronize(p->stream) != cudaSuccess) rc = S3O_ERR_CUDA;
        if (rc) { free_marginal_arrays(S); set_error("%s: device allocation failed", who); return rc; }
    }
    // requested pairs -> block of Sigma (elimination order) and transpose flag; the rest by block column
    std::vector<int32_t> ipos(n);
    for (int k = 0; k < n; ++k) ipos[Pl.perm[k]] = k;
    std::vector<int32_t> pick(n_pairs);
    std::vector<std::pair<int32_t, int32_t>> off;       // (column, pair) of the pairs off the pattern
    for (int k = 0; k < n_pairs; ++k) {
        const int r = rows ? rows[k] : k, c = cols ? cols[k] : k;
        const int pr = ipos[r], pc = ipos[c];
        const int32_t t = direct_find_block(Pl, std::min(pr, pc), std::max(pr, pc));
        pick[k] = t >= 0 ? (t << 1) | (pr < pc ? 1 : 0) : -1;
        if (t < 0) off.push_back({ c, k });
    }
    std::sort(off.begin(), off.end());
    std::vector<int32_t> crow(off.size()), cdst(off.size());
    S->col_ptr.clear();
    S->col_id.clear();
    for (size_t q = 0; q < off.size(); ++q) {
        if (q == 0 || off[q].first != off[q - 1].first) { S->col_ptr.push_back((int32_t)q); S->col_id.push_back(off[q].first); }
        crow[q] = rows[off[q].second];
        cdst[q] = off[q].second;
    }
    if (!off.empty()) S->col_ptr.push_back((int32_t)off.size());
    if (n_pairs > S->out_cap) {
        dev_free(S->d_pick); dev_free(S->d_crow); dev_free(S->d_cdst); dev_free(S->d_out);
        S->out_cap = 0;
        rc = dev_alloc(&S->d_pick, (size_t)n_pairs);
        rc = rc ? rc : dev_alloc(&S->d_crow, (size_t)n_pairs);
        rc = rc ? rc : dev_alloc(&S->d_cdst, (size_t)n_pairs);
        rc = rc ? rc : dev_alloc(&S->d_out, (size_t)n_pairs * dd);
        if (rc) { set_error("%s: device allocation failed", who); return rc; }
        S->out_cap = n_pairs;
    }
    auto h2d = [&](int32_t *dst, const std::vector<int32_t> &v) -> int {
        if (v.empty()) return S3O_OK;
        S3O_CUDA(cudaMemcpyAsync(dst, v.data(), v.size() * sizeof(int32_t), cudaMemcpyHostToDevice, p->stream));
        p->stats.h2d_bytes += (int64_t)(v.size() * sizeof(int32_t));
        return S3O_OK;
    };
    if ((rc = h2d(S->d_pick, pick)) || (rc = h2d(S->d_crow, crow)) || (rc = h2d(S->d_cdst, cdst))) return rc;
    R->S = S;
    R->plan = &S->plan;
    R->serial = S->serial;
    R->Sig = S->d_Sig;
    R->out = S->d_out;
    R->fail = S->d_fail;
    return S3O_OK;
}

int marginals_factor(s3o_problem *p, const MarginalsRun &R, cudaEvent_t *ev) {
    int rc;
    switch (p->d) {
    case 7: rc = factor_launches<7>(p, R.S, ev); break;
    case 6: rc = factor_launches<6>(p, R.S, ev); break;
    case 4: rc = factor_launches<4>(p, R.S, ev); break;
    case 1: rc = factor_launches<1>(p, R.S, ev); break;
    default: set_error("marginals: block dimension %d", p->d); return S3O_ERR_UNSUPPORTED;
    }
    R.S->factored = false;      // the factor of H without damping: a later solve with reuse_factor factorises again
    return rc;
}

int marginals_pick(s3o_problem *p, const MarginalsRun &R, int n_pairs) {
    switch (p->d) {
    case 7: return pick_launches<7>(p, R.S, n_pairs);
    case 6: return pick_launches<6>(p, R.S, n_pairs);
    case 4: return pick_launches<4>(p, R.S, n_pairs);
    case 1: return pick_launches<1>(p, R.S, n_pairs);
    }
    set_error("marginals: block dimension %d", p->d);
    return S3O_ERR_UNSUPPORTED;
}

// Marginal covariances for the H in p->d_H (see problem.h).
int direct_marginals(s3o_problem *p, int n_pairs, const int32_t *rows, const int32_t *cols, double *out, cudaEvent_t *ev) {
    MarginalsRun R;
    int rc = marginals_open(p, "s3o_compute_marginals", n_pairs, rows, cols, &R);
    if (rc) return rc;
    if ((rc = marginals_factor(p, R, ev)) || (rc = marginals_pick(p, R, n_pairs))) return rc;
    if (ev) cudaEventRecord(ev[2], p->stream);
    const int dd = p->d * p->d;
    int failed = 0;
    if (n_pairs > 0) S3O_CUDA(cudaMemcpyAsync(out, R.out, sizeof(double) * n_pairs * dd, cudaMemcpyDeviceToHost, p->stream));
    S3O_CUDA(cudaMemcpyAsync(&failed, R.fail, sizeof(int), cudaMemcpyDeviceToHost, p->stream));
    S3O_CUDA(cudaStreamSynchronize(p->stream));
    p->stats.d2h_bytes += (int64_t)n_pairs * dd * 8 + 4;
    if (failed) { set_error("s3o_compute_marginals: the Hessian is not positive definite (a pivot of its factorisation failed)"); return S3O_ERR_SOLVE; }
    return S3O_OK;
}

}  // namespace s3o
