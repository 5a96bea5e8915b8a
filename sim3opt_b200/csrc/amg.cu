// amg.cu -- multilevel preconditioner of the pose-graph PCG (Sim3, scale-trans, scale): device side (see amg.h).
//
// Values flow per LM trial:   frames (per linearisation)  ->  Galerkin operators level by level
// ->  block-Jacobi inverses per level  ->  dense inverse of the coarsest level.
// Per PCG iteration:          restriction of r  ->  V(1,1)-cycle on the coarse levels  ->
//                             z = D^-1 r + P0 x_1,  r.z  and the PCG scalar bookkeeping.
// All sums run in list order (no atomics), so a solve is bitwise reproducible.
#include <algorithm>
#include <cstdlib>
#include <functional>

#include <cooperative_groups.h>

#include "amg.h"
#include "comm.h"
#include "problem.h"
#include "reduce.cuh"
#include "sim3_math.cuh"

namespace s3o {

namespace {

#define DD (D * D)       /* D: template parameter in the kernels, p->d in the host code */
constexpr int NREL = 13;             // doubles of transfer data per vertex: a 3x3 matrix, a 3-vector, a scalar
constexpr int kCoarsestMax = 16;        // dense inverse held in shared memory: (16*7)^2 doubles = 98 KB
constexpr int kCoarsestMaxBig = 128;    // large graphs: the hierarchy stops at <= 128 vertices, inverted by a cooperative
                                        // block Gauss-Jordan in global memory (896^2 doubles = 6.4 MB); one level fewer
                                        // to recurse through in every K-cycle visit
constexpr int kBigGraph = 20000;        // free vertices from which the deep-hierarchy settings apply
constexpr int kMaxLevels = 12;
constexpr double kOmega = 0.7;          // damping of the block-Jacobi smoother on the coarse levels
constexpr int kPlanHeader = 9;          // amg_plan_info: entries before the per-level (n, nblk, G) triples

struct LevelDev {       // transfer level l -> l+1 plus operator and vectors of level l+1
    int n_fine = 0, n = 0, nblk = 0, nub = 0, pad_fine = 0;
    int32_t *agg = nullptr, *mem_ptr = nullptr, *mem_idx = nullptr, *vid = nullptr;
    int32_t *rowptr = nullptr, *colidx = nullptr, *blk_row = nullptr, *dpos = nullptr;
    int32_t *gal_ptr = nullptr, *gal_ent = nullptr, *gal_i = nullptr, *gal_j = nullptr, *gal_out = nullptr, *gal_mirror = nullptr;
    int32_t *gal_order = nullptr;
    double *rel = nullptr;      // [13][pad_fine]: R (row-major), t, s of S_i S_root^-1 for every level-l vertex
    double *A = nullptr, *Dinv = nullptr, *r = nullptr, *x = nullptr, *x2 = nullptr, *t = nullptr;
    double *z1 = nullptr, *q1 = nullptr, *rp = nullptr, *z2 = nullptr;      // K-cycle (two inner conjugate-gradient steps)
    int32_t *acol = nullptr;    // [nblk] aggregate (in the transfer to the next level) of every block's column vertex
    // A = K + lambda M with K = P^T H P (Galerkin product of the undamped Hessian) and M = P^T P, which is block
    // diagonal on every level (one nonzero block per row of P): a new lambda only rewrites the diagonal blocks
    double *Kd = nullptr, *M = nullptr;     // [n][D*D] diagonal blocks of K, blocks of M
};

// scalars of the two-step inner conjugate-gradient iteration of one K-cycle level (device resident)
struct KScal { double rho1, alpha1, c1, c2; };

}  // namespace

struct AmgState {
    std::vector<AmgHostLevel> host;
    std::vector<LevelDev> lev;
    int32_t *d_vid0 = nullptr;      // level-0 vertex ids (free2v)
    double *d_dense = nullptr;      // inverse of the coarsest operator, [N][N]
    bool dense = false;
    bool frames_valid = false;
    // K = P^T H P is rebuilt when the linearisation point has moved; a new lambda at the same point (LM retry) only
    // shifts the diagonal blocks.  (Keeping K across linearisations does NOT work, measured on the 1M-pose sphere: with
    // a Hessian whose diagonal blocks had moved by < 2 % the PCG no longer converged in 20 000 iterations -- the coarse
    // energy of the near-null gauge modes must be the current Hessian's, else the coarse solve over-corrects them.)
    bool k_valid = false, lin_changed = true;
    std::vector<size_t> m_off, m_cnt;   // partitioned solve: all-gather segments of M_1
    int64_t rebuilds = 0, reuses = 0;
    // partitioned solve: the fine level is local (owned + ghost rows), level 1 and below are replicated.
    // Rank q computes the level-1 rows [crow[q], crow[q+1]) (its own aggregates); the segments are
    // exchanged with in-place all-gathers: the residual r_1 every PCG iteration, the operator A_1 every trial.
    bool dist = false;
    int n_own = 0;
    std::vector<size_t> r_off, r_cnt, a_off, a_cnt;
    // r_1 goes through ONE equal-count ncclAllGather (padded to the largest segment) plus an unpad
    // kernel: eight grouped broadcasts cost several times the latency of one all-gather
    size_t r_max = 0;
    double *d_rpad = nullptr;       // [world][r_max]
    int32_t *d_unpad_src = nullptr; // [n_1 * 7] position in d_rpad of every entry of r_1
    int32_t *d_scal_pos = nullptr;  // [world] position in d_rpad of every rank's two partial scalars
    size_t r_seg = 0;               // doubles per rank in d_rpad: r_max + 2
    // K-cycle: the first `kdepth` coarse levels run two inner conjugate-gradient steps preconditioned by the
    // cycle below them (Notay's K-cycle) instead of one V-cycle visit; every level from `coop_first` down is
    // walked by ONE cooperative kernel (grid barriers instead of kernel boundaries)
    int kdepth = 0, coop_first = 0, coop_grid = 0;
    unsigned kmask = 0;         // bit l: level l is a K-cycle level (default: the first kdepth levels; S3O_KMASK overrides)
    KScal *d_ks = nullptr;          // [kMaxLevels]
    bool dense_coop = false;        // coarsest level inverted by the cooperative kernel (too large for shared memory)
    double *d_rowbuf = nullptr;     // [2][d*N + d*d]: scaled pivot row + pivot inverse of the dense inversion, double-buffered
    double *d_cdots = nullptr;      // [3][coop_grid] partial sums of the cooperative kernel's dot products
};

namespace {

struct Rel { double R[9], t[3], s; };

__device__ __forceinline__ Rel load_rel(const double *__restrict__ rel, int pad, int i) {
    Rel r;
#pragma unroll
    for (int k = 0; k < 9; ++k) r.R[k] = __ldg(rel + (size_t)k * pad + i);
#pragma unroll
    for (int k = 0; k < 3; ++k) r.t[k] = __ldg(rel + (size_t)(9 + k) * pad + i);
    r.s = __ldg(rel + (size_t)12 * pad + i);
    return r;
}

// The prolongation block P_i maps the tangent of an aggregate's root to the tangent of member i along
// the gauge freedom of the graph (a right-multiplied world similarity G):
//   Sim3 (d=7)        S_i G = exp(delta_i) S_i          =>  P_i = Ad(S_i S_root^-1)
//   scale-trans (d=4) delta_i = (s_i sigma, s_i R_i c)  =>  P_i = (s_i/s_root) diag(1, R_i R_root^T)
//   scale (d=1)       delta_i = s_i sigma               =>  P_i = s_i/s_root
// All three are held as Rel = (3x3 matrix R, 3-vector t, scalar s).
template <int D> struct Xf;

template <> struct Xf<7> {
    // out = Ad(S) v,  Ad(S) = [[R,0,0],[[t]x R, sR, -t],[0,0,1]]  on tangents [omega, upsilon, sigma]
    static __device__ __forceinline__ void apply(const Rel &S, const double v[7], double out[7]) {
        double a[3], b[3];
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            a[r] = S.R[r * 3] * v[0] + S.R[r * 3 + 1] * v[1] + S.R[r * 3 + 2] * v[2];
            b[r] = S.R[r * 3] * v[3] + S.R[r * 3 + 1] * v[4] + S.R[r * 3 + 2] * v[5];
        }
        out[0] = a[0]; out[1] = a[1]; out[2] = a[2];
        out[3] = (S.t[1] * a[2] - S.t[2] * a[1]) + S.s * b[0] - S.t[0] * v[6];
        out[4] = (S.t[2] * a[0] - S.t[0] * a[2]) + S.s * b[1] - S.t[1] * v[6];
        out[5] = (S.t[0] * a[1] - S.t[1] * a[0]) + S.s * b[2] - S.t[2] * v[6];
        out[6] = v[6];
    }
    // out = Ad(S)^T w:  [R^T (a + b x t);  s R^T b;  c - t.b]   for w = [a, b, c]
    static __device__ __forceinline__ void applyT(const Rel &S, const double w[7], double out[7]) {
        const double u0 = w[0] + (w[4] * S.t[2] - w[5] * S.t[1]);
        const double u1 = w[1] + (w[5] * S.t[0] - w[3] * S.t[2]);
        const double u2 = w[2] + (w[3] * S.t[1] - w[4] * S.t[0]);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            out[c] = S.R[c] * u0 + S.R[3 + c] * u1 + S.R[6 + c] * u2;
            out[3 + c] = S.s * (S.R[c] * w[3] + S.R[3 + c] * w[4] + S.R[6 + c] * w[5]);
        }
        out[6] = w[6] - (S.t[0] * w[3] + S.t[1] * w[4] + S.t[2] * w[5]);
    }
};

template <> struct Xf<4> {      // P = s diag(1, R)
    static __device__ __forceinline__ void apply(const Rel &S, const double v[4], double out[4]) {
        out[0] = S.s * v[0];
#pragma unroll
        for (int r = 0; r < 3; ++r) out[1 + r] = S.s * (S.R[r * 3] * v[1] + S.R[r * 3 + 1] * v[2] + S.R[r * 3 + 2] * v[3]);
    }
    static __device__ __forceinline__ void applyT(const Rel &S, const double w[4], double out[4]) {
        out[0] = S.s * w[0];
#pragma unroll
        for (int c = 0; c < 3; ++c) out[1 + c] = S.s * (S.R[c] * w[1] + S.R[3 + c] * w[2] + S.R[6 + c] * w[3]);
    }
};

template <> struct Xf<1> {      // P = s
    static __device__ __forceinline__ void apply(const Rel &S, const double v[1], double out[1]) { out[0] = S.s * v[0]; }
    static __device__ __forceinline__ void applyT(const Rel &S, const double w[1], double out[1]) { out[0] = S.s * w[0]; }
};

// ---- frames: the transfer data of every level-l vertex relative to its aggregate's root -------
template <int KIND>
__global__ void amg_rel_kernel(const double *__restrict__ est, const double *__restrict__ aux, int nv_pad,
                               const int32_t *__restrict__ vid_fine, const int32_t *__restrict__ agg,
                               const int32_t *__restrict__ vid_coarse, int n_fine, int pad, double *__restrict__ rel) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_fine) return;
    const int vi = vid_fine[i], vr = vid_coarse[agg[i]];
    double R[9] = { 1, 0, 0, 0, 1, 0, 0, 0, 1 }, t[3] = { 0, 0, 0 }, sc = 1;
    if constexpr (KIND == S3O_KIND_SIM3) {
        Sim3 Si, Sr;
        Si.qx = est[vi]; Si.qy = est[(size_t)nv_pad + vi]; Si.qz = est[(size_t)2 * nv_pad + vi]; Si.qw = est[(size_t)3 * nv_pad + vi];
        Si.tx = est[(size_t)4 * nv_pad + vi]; Si.ty = est[(size_t)5 * nv_pad + vi]; Si.tz = est[(size_t)6 * nv_pad + vi];
        Si.s = est[(size_t)7 * nv_pad + vi];
        Sr.qx = est[vr]; Sr.qy = est[(size_t)nv_pad + vr]; Sr.qz = est[(size_t)2 * nv_pad + vr]; Sr.qw = est[(size_t)3 * nv_pad + vr];
        Sr.tx = est[(size_t)4 * nv_pad + vr]; Sr.ty = est[(size_t)5 * nv_pad + vr]; Sr.tz = est[(size_t)6 * nv_pad + vr];
        Sr.s = est[(size_t)7 * nv_pad + vr];
        const Sim3 S = sim3_mul(Si, sim3_inv(Sr));
        const double qn = 1.0 / sqrt(S.qx * S.qx + S.qy * S.qy + S.qz * S.qz + S.qw * S.qw);
        quat_to_rot(S.qx * qn, S.qy * qn, S.qz * qn, S.qw * qn, R);
        t[0] = S.tx; t[1] = S.ty; t[2] = S.tz;
        sc = S.s;
    } else if constexpr (KIND == S3O_KIND_SCALE_TRANS) {
        // estimate planes [s tx ty tz]; aux planes = the fixed rotation quaternion of every vertex
        double Ri[9], Rr[9];
        quat_to_rot(aux[vi], aux[(size_t)nv_pad + vi], aux[(size_t)2 * nv_pad + vi], aux[(size_t)3 * nv_pad + vi], Ri);
        quat_to_rot(aux[vr], aux[(size_t)nv_pad + vr], aux[(size_t)2 * nv_pad + vr], aux[(size_t)3 * nv_pad + vr], Rr);
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int c = 0; c < 3; ++c)
                R[r * 3 + c] = Ri[r * 3] * Rr[c * 3] + Ri[r * 3 + 1] * Rr[c * 3 + 1] + Ri[r * 3 + 2] * Rr[c * 3 + 2];   // R_i R_root^T
        sc = est[vi] / est[vr];
    } else {
        sc = est[vi] / est[vr];
    }
#pragma unroll
    for (int k = 0; k < 9; ++k) rel[(size_t)k * pad + i] = R[k];
    rel[(size_t)9 * pad + i] = t[0]; rel[(size_t)10 * pad + i] = t[1]; rel[(size_t)11 * pad + i] = t[2];
    rel[(size_t)12 * pad + i] = sc;
}

// ---- Galerkin product: one 8-lane group per upper coarse block ---------------------------------
// Entry lists carry (block | flag, row vertex, column vertex) so the only dependent loads per entry are the frames
// and the block itself; the next entry's indices are fetched one step ahead.  Per entry X = P_l^T A P_r is formed in
// two structured applications with a transposition in between: lane r reads ROW r of A (7 loads instead of the whole
// block) and turns it into row r of A P_r; the group transposes through shared memory; lane c turns column c of
// A P_r into column c of X.  flag 0: X = P_i^T A P_j;  1: X = P_j^T A^T P_i (block stored on the other side);
// 2: both (an off-diagonal fine block inside one aggregate) -- the second is the transpose of the first, so those X
// are also summed separately and their transpose is added once at the end.
template <int D, bool FINE_UPPER>
__global__ void __launch_bounds__(128, 4) amg_galerkin_kernel(const double *__restrict__ Af, const int32_t *__restrict__ gal_i,
                                                              const int32_t *__restrict__ gal_j, const double *__restrict__ rel,
                                                              int pad, int nub,
                                                              const int32_t *__restrict__ gal_ptr, const int32_t *__restrict__ gal_ent,
                                                              const int32_t *__restrict__ gal_out,
                                                              const int32_t *__restrict__ gal_mirror, double *__restrict__ Ac,
                                                              int write_mirror, const int32_t *__restrict__ gal_order) {
    __shared__ double tr[16][D * D + 1];
    const int grp = threadIdx.x / 8;
    const int slot = blockIdx.x * (blockDim.x / 8) + grp;
    const int c = threadIdx.x & 7;
    if (slot >= nub) return;              // the whole group leaves
    const unsigned gmask = 0xffu << (threadIdx.x & 24);
    const bool act = c < D;
    const int cc = act ? c : 0;           // lane 7 shadows lane 0 (keeps the group convergent), stores nothing
    const int ub = gal_order[slot];       // lists of equal length share a warp
    double acc[D], accS[D];
#pragma unroll
    for (int r = 0; r < D; ++r) { acc[r] = 0; accS[r] = 0; }
    bool any2 = false;
    const int ebeg = gal_ptr[ub], eend = gal_ptr[ub + 1];
    int ent = 0, i = 0, j = 0;
    if (ebeg < eend) { ent = __ldg(gal_ent + ebeg); i = __ldg(gal_i + ebeg); j = __ldg(gal_j + ebeg); }
    for (int e = ebeg; e < eend; ++e) {
        const int k = ent >> 2, flag = ent & 3;
        const int vl = flag == 1 ? j : i, vr = flag == 1 ? i : j;      // left and right factor of X
        if (e + 1 < eend) { ent = __ldg(gal_ent + e + 1); i = __ldg(gal_i + e + 1); j = __ldg(gal_j + e + 1); }
        const Rel rl = load_rel(rel, pad, vl);
        const Rel rr = (vl == vr) ? rl : load_rel(rel, pad, vr);
        const double *A = Af + (size_t)k * DD;
        double a[D], b[D], w[D], u[D];
        if (flag != 1) {
#pragma unroll
            for (int q = 0; q < D; ++q) a[q] = __ldg(A + cc * D + q);
        } else {
#pragma unroll
            for (int q = 0; q < D; ++q) a[q] = __ldg(A + q * D + cc);
        }
        Xf<D>::applyT(rr, a, b);          // row cc of (A P_r)
        __syncwarp(gmask);
        if (act) {
#pragma unroll
            for (int q = 0; q < D; ++q) tr[grp][cc * D + q] = b[q];
        }
        __syncwarp(gmask);
#pragma unroll
        for (int r = 0; r < D; ++r) w[r] = tr[grp][r * D + cc];
        Xf<D>::applyT(rl, w, u);          // column cc of P_l^T (A P_r)
#pragma unroll
        for (int r = 0; r < D; ++r) acc[r] += u[r];
        if (flag == 2) {
            any2 = true;
#pragma unroll
            for (int r = 0; r < D; ++r) accS[r] += u[r];
        }
    }
    if (any2) {                            // uniform over the group: T += S^T
        __syncwarp(gmask);
        if (act) {
#pragma unroll
            for (int r = 0; r < D; ++r) tr[grp][r * D + cc] = accS[r];
        }
        __syncwarp(gmask);
#pragma unroll
        for (int r = 0; r < D; ++r) acc[r] += tr[grp][cc * D + r];
    }
    if (!act) return;
    double *out = Ac + (size_t)gal_out[ub] * DD;
#pragma unroll
    for (int r = 0; r < D; ++r) out[r * D + c] = acc[r];
    const int m = write_mirror ? gal_mirror[ub] : -1;
    if (m >= 0) {
        double *om = Ac + (size_t)m * DD;
#pragma unroll
        for (int r = 0; r < D; ++r) om[c * D + r] = acc[r];
    }
}

// M_I = sum_{i in I} P_i^T Mf_i P_i  (Mf == nullptr: identity): an 8-lane group per aggregate, lane c holds column c
template <int D>
__global__ void amg_mass_kernel(int n, const int32_t *__restrict__ mem_ptr, const int32_t *__restrict__ mem_idx,
                                const double *__restrict__ rel, int pad, const double *__restrict__ Mf, double *__restrict__ M) {
    const int I = blockIdx.x * (blockDim.x / 8) + threadIdx.x / 8;
    const int c = threadIdx.x & 7;
    if (I >= n || c >= D) return;
    double acc[D], ec[D];
#pragma unroll
    for (int r = 0; r < D; ++r) { acc[r] = 0; ec[r] = (r == c) ? 1.0 : 0.0; }
    for (int m = mem_ptr[I]; m < mem_ptr[I + 1]; ++m) {
        const int i = mem_idx[m];
        const Rel S = load_rel(rel, pad, i);
        double v[D], w[D], u[D];
        Xf<D>::apply(S, ec, v);
        if (Mf) {
            const double *B = Mf + (size_t)i * DD;
#pragma unroll
            for (int r = 0; r < D; ++r) {
                double a = 0;
#pragma unroll
                for (int q = 0; q < D; ++q) a += __ldg(B + r * D + q) * v[q];
                w[r] = a;
            }
        } else {
#pragma unroll
            for (int r = 0; r < D; ++r) w[r] = v[r];
        }
        Xf<D>::applyT(S, w, u);
#pragma unroll
        for (int r = 0; r < D; ++r) acc[r] += u[r];
    }
#pragma unroll
    for (int r = 0; r < D; ++r) M[(size_t)I * DD + r * D + c] = acc[r];
}

// Kd_I = diagonal block of A (called while A still holds K)
template <int D>
__global__ void amg_save_diag_kernel(int n, const int32_t *__restrict__ dpos, const double *__restrict__ A, double *__restrict__ Kd) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * DD) return;
    const int I = t / DD, e = t - I * DD;
    Kd[t] = A[(size_t)dpos[I] * DD + e];
}

// diagonal block of A = Kd + lambda M
template <int D>
__global__ void amg_shift_diag_kernel(int n, const int32_t *__restrict__ dpos, const double *__restrict__ Kd,
                                      const double *__restrict__ M, double lambda, double *__restrict__ A) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * DD) return;
    const int I = t / DD, e = t - I * DD;
    A[(size_t)dpos[I] * DD + e] = Kd[t] + lambda * M[t];
}

// lower blocks of a level from its upper blocks (partitioned solve: after the all-gather of A_1)
template <int D>
__global__ void amg_mirror_kernel(int nub, const int32_t *__restrict__ gal_out, const int32_t *__restrict__ gal_mirror,
                                  double *__restrict__ A) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int ub = t / DD, e = t - ub * DD;
    if (ub >= nub) return;
    const int m = gal_mirror[ub];
    if (m < 0) return;
    const int r = e / D, c = e - r * D;
    A[(size_t)m * DD + c * D + r] = A[(size_t)gal_out[ub] * DD + e];
}

// ---- dense inverse of the coarsest operator (one CTA, matrix in shared memory) -----------------
template <int D>
__global__ void __launch_bounds__(256) amg_dense_inverse_kernel(const double *__restrict__ A, const int32_t *__restrict__ rowptr,
                                                                const int32_t *__restrict__ colidx, int n,
                                                                double *__restrict__ inv, DevScalars *sc) {
    extern __shared__ double a[];
    const int N = n * D;
    double *col = a + N * N;
    for (int t = threadIdx.x; t < N * N; t += blockDim.x) a[t] = 0;
    __syncthreads();
    for (int I = 0; I < n; ++I)
        for (int k = rowptr[I]; k < rowptr[I + 1]; ++k) {
            const int J = colidx[k];
            for (int t = threadIdx.x; t < DD; t += blockDim.x) a[(I * D + t / D) * N + J * D + t % D] = A[(size_t)k * DD + t];
        }
    __syncthreads();
    for (int k = 0; k < N; ++k) {       // in-place Gauss-Jordan, no pivoting (SPD)
        for (int t = threadIdx.x; t < N; t += blockDim.x) col[t] = a[t * N + k];
        __syncthreads();
        double piv = col[k];
        if (!(piv > 0)) { piv = 1; if (threadIdx.x == 0) sc->precond_fail = 1; }
        const double ip = 1.0 / piv;
        for (int t = threadIdx.x; t < N; t += blockDim.x) a[k * N + t] = (t == k) ? ip : a[k * N + t] * ip;
        __syncthreads();
        for (int t = threadIdx.x; t < N * N; t += blockDim.x) {
            const int i = t / N, j = t - i * N;
            if (i == k) continue;
            a[t] = (j == k) ? -col[i] * ip : a[t] - col[i] * a[k * N + j];
        }
        __syncthreads();
    }
    for (int t = threadIdx.x; t < N * N; t += blockDim.x) inv[t] = a[t];
}

// most threads per CTA of amg_dense_inverse_coop_kernel (one CTA per SM).  Every pivot step is a latency chain of
// d*N/threads loads and updates per thread (S1M, 96 pivots: 1.09 ms with 256 threads, 0.89 with 512, 0.84 with 1024);
// S3O_DENSE_THREADS overrides for experiments.
constexpr int kDenseCoopThreads = 1024;
// dynamic shared memory of amg_dense_inverse_coop_kernel: block row, pivot row, P, C, inversion work space
inline size_t dense_coop_smem(int n, int d) { return ((size_t)2 * d * n * d + 2 * d * d + 2 * d * d) * sizeof(double); }

// Same inverse for a coarsest level that does not fit one CTA's shared memory: block Gauss-Jordan on the d x d block
// grid, CTA i keeps block row i (d x N) in shared memory for the whole elimination.  Step k needs the pivot block's
// inverse P = A_kk^-1 and the scaled pivot row  rowbuf = P A_k,:  from CTA k; everything else is local:
//   row k:   A_kj <- rowbuf_j, A_kk <- P          other rows:  C = A_ik;  A_ik <- -C P;  A_ij <- A_ij - C rowbuf_j
// CTA k+1 prepares P and rowbuf of the next step right after its own update, so there is ONE grid barrier per pivot
// block.  No pivoting (the matrix is SPD).  pub: [2][d*N + d*d] double-buffered rowbuf + P in global memory.
template <int D>
__global__ void __launch_bounds__(kDenseCoopThreads) amg_dense_inverse_coop_kernel(const double *__restrict__ A, const int32_t *__restrict__ rowptr,
                                                                     const int32_t *__restrict__ colidx, int n, double *inv,
                                                                     double *pub, DevScalars *sc, const GridBarrier gb) {
    extern __shared__ double smem[];
    unsigned phase = 0;
    const int N = n * D, ib = blockIdx.x, NT = blockDim.x;
    double *row = smem;                 // [D][N]   this CTA's block row
    double *rb = row + (size_t)D * N;   // [D][N]   scaled pivot row of the current step
    double *Ps = rb + (size_t)D * N;    // [D][D]   inverse of the pivot block
    double *Cb = Ps + DD;               // [D][D]   this row's pivot-column block before the update
    double *Ms = Cb + DD;               // [D][2D]  work space of the d x d inversion
    const size_t pub_stride = (size_t)D * N + DD;
    for (int t = threadIdx.x; t < D * N; t += NT) row[t] = 0;
    __syncthreads();
    for (int k = rowptr[ib] * DD + threadIdx.x; k < rowptr[ib + 1] * DD; k += NT) {
        const int blk = k / DD, e = k - blk * DD;
        row[(e / D) * N + colidx[blk] * D + e % D] = A[k];
    }
    __syncthreads();
    // P = (row[:, kb block])^-1 and rowbuf = P row -> pub[slot]; called by all threads of the CTA that owns block row kb
    auto publish = [&](int kb, int slot) {
        if (threadIdx.x < 32) {         // Gauss-Jordan on [M | I] (d x 2d) by one warp
            const int lane = threadIdx.x;
            for (int e = lane; e < D * 2 * D; e += 32) {
                const int r = e / (2 * D), c = e - r * 2 * D;
                Ms[e] = c < D ? row[r * N + kb * D + c] : (c - D == r ? 1.0 : 0.0);
            }
            __syncwarp();
            for (int c = 0; c < D; ++c) {
                double piv = Ms[c * 2 * D + c];
                if (!(piv > 0)) { piv = 1; if (lane == 0) sc->precond_fail = 1; }
                const double ip = 1.0 / piv;
                double f[(D * 2 * D + 31) / 32];
#pragma unroll
                for (int q = 0; q < (D * 2 * D + 31) / 32; ++q) {
                    const int e = lane + 32 * q, r = e / (2 * D);
                    f[q] = (e < D * 2 * D && r != c) ? Ms[r * 2 * D + c] : 0.0;
                }
                __syncwarp();
                if (lane < 2 * D) Ms[c * 2 * D + lane] *= ip;
                __syncwarp();
#pragma unroll
                for (int q = 0; q < (D * 2 * D + 31) / 32; ++q) {
                    const int e = lane + 32 * q, r = e / (2 * D), cc = e - r * 2 * D;
                    if (e < D * 2 * D && r != c) Ms[e] -= f[q] * Ms[c * 2 * D + cc];
                }
                __syncwarp();
            }
            for (int e = lane; e < DD; e += 32) Ps[e] = Ms[(e / D) * 2 * D + D + e % D];
        }
        __syncthreads();
        double *out = pub + (size_t)slot * pub_stride;
        for (int t = threadIdx.x; t < D * N; t += NT) {
            const int r = t / N, j = t - r * N;
            double acc = 0;
#pragma unroll
            for (int m = 0; m < D; ++m) acc += Ps[r * D + m] * row[m * N + j];
            out[t] = acc;
        }
        for (int e = threadIdx.x; e < DD; e += NT) out[(size_t)D * N + e] = Ps[e];
    };
    if (ib == 0) publish(0, 0);
    grid_barrier(gb, phase);
    for (int kb = 0; kb < n; ++kb) {
        const double *in = pub + (size_t)(kb & 1) * pub_stride;
        for (int t = threadIdx.x; t < D * N; t += NT) rb[t] = __ldcg(in + t);
        for (int e = threadIdx.x; e < DD; e += NT) {
            Ps[e] = __ldcg(in + (size_t)D * N + e);
            Cb[e] = row[(e / D) * N + kb * D + e % D];
        }
        __syncthreads();
        if (ib == kb) {
            for (int t = threadIdx.x; t < D * N; t += NT) {
                const int r = t / N, j = t - r * N, jb = j / D;
                row[t] = (jb == kb) ? Ps[r * D + (j - kb * D)] : rb[t];
            }
        } else {
            for (int t = threadIdx.x; t < D * N; t += NT) {
                const int r = t / N, j = t - r * N, jb = j / D;
                double acc = 0;
                if (jb == kb) {
#pragma unroll
                    for (int m = 0; m < D; ++m) acc -= Cb[r * D + m] * Ps[m * D + (j - kb * D)];
                    row[t] = acc;
                } else {
#pragma unroll
                    for (int m = 0; m < D; ++m) acc += Cb[r * D + m] * rb[m * N + j];
                    row[t] -= acc;
                }
            }
        }
        __syncthreads();
        if (kb + 1 < n) {
            if (ib == kb + 1) publish(kb + 1, (kb + 1) & 1);
            grid_barrier(gb, phase);
        }
    }
    for (int t = threadIdx.x; t < D * N; t += NT) inv[(size_t)(ib * D) * N + t] = row[t];
}

// ---- coarse-level row kernels: an 8-lane group owns one block row, lane l one component ---------
// mode 0: x_out = omega Dinv r                      (first smoothing sweep from x = 0)
// mode 1: t_out = r - A x                           (residual)
// mode 2: x_out = x + omega Dinv (r - A x)          (smoothing sweep)
template <int D, int MODE>
__global__ void __launch_bounds__(128) amg_row_kernel(int n, const int32_t *__restrict__ rowptr, const int32_t *__restrict__ colidx,
                                                      const double *__restrict__ A, const double *__restrict__ Dinv,
                                                      const double *__restrict__ r, const double *__restrict__ x,
                                                      double *__restrict__ out, double omega, const DevScalars *sc,
                                                      int check_done) {
    if (check_done && sc->done) return;
    const int i = blockIdx.x * (blockDim.x / 8) + threadIdx.x / 8;
    const int l = threadIdx.x & 7;
    const bool act = i < n && l < D;
    double res = act ? r[(size_t)i * D + l] : 0.0;
    if (MODE != 0 && act) {
        double acc = 0;
        for (int k = rowptr[i]; k < rowptr[i + 1]; ++k) {
            const double *xj = x + (size_t)colidx[k] * D;
            const double *Ak = A + (size_t)k * DD + l * D;
#pragma unroll
            for (int c = 0; c < D; ++c) acc += Ak[c] * xj[c];
        }
        res -= acc;
    }
    if (MODE == 1) {
        if (act) out[(size_t)i * D + l] = res;
        return;
    }
    double z = 0;
#pragma unroll
    for (int c = 0; c < D; ++c) {
        const double rc = __shfl_sync(0xffffffffu, res, c, 8);
        if (act) z += Dinv[(size_t)i * sym_size<D>() + sym_off<D>(l, c)] * rc;
    }
    if (act) out[(size_t)i * D + l] = (MODE == 2 ? x[(size_t)i * D + l] : 0.0) + omega * z;
}

// Partitioned solve: every rank's all-gather segment carries, after its rows of r_1, its partial sums
// r.zJ and |r|^2 (two doubles) -- the second all-reduce of a PCG iteration rides on this all-gather.
__global__ void amg_scalars_to_vec_kernel(double *__restrict__ slot, const DevScalars *sc, int check_done) {
    if (check_done && sc->done) return;
    slot[0] = sc->rz_new;
    slot[1] = sc->rr;
}
// r_1 out of the padded all-gather buffer; thread 0 also sums the ranks' partial scalars in rank order
__global__ void amg_unpad_kernel(int n, const int32_t *__restrict__ src, const double *__restrict__ padded,
                                 double *__restrict__ out, DevScalars *sc, int check_done, int world,
                                 const int32_t *__restrict__ scal_pos) {
    if (check_done && sc->done) return;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) out[t] = padded[src[t]];
    if (t == 0) {
        double rz = 0, rr = 0;
        for (int q = 0; q < world; ++q) { rz += padded[scal_pos[q]]; rr += padded[scal_pos[q] + 1]; }
        sc->rz_new = rz;
        sc->rr = rr;
    }
}

// ---- transfers ---------------------------------------------------------------------------------
// r_coarse[I] = sum over members i of Ad(rel_i)^T t_i.  An 8-lane group owns one aggregate: lane m
// takes members m, m+8, ... (ascending), the eight partial sums are combined by a fixed butterfly,
// so the result is reproducible.
template <int D>
__global__ void __launch_bounds__(128) amg_restrict_kernel(int n, const int32_t *__restrict__ mem_ptr,
                                                           const int32_t *__restrict__ mem_idx, const double *__restrict__ rel,
                                                           int pad, const double *__restrict__ t, double *__restrict__ rc,
                                                           const DevScalars *sc, int check_done) {
    if (check_done && sc->done) return;
    const int I = blockIdx.x * (blockDim.x / 8) + threadIdx.x / 8;
    const int lane = threadIdx.x & 7;
    const bool act = I < n;
    double acc[D];
#pragma unroll
    for (int c = 0; c < D; ++c) acc[c] = 0;
    if (act) {
        const int mb = mem_ptr[I], me = mem_ptr[I + 1];
        for (int m = mb + lane; m < me; m += 8) {
            const int i = mem_idx[m];
            const Rel S = load_rel(rel, pad, i);
            double w[D], u[D];
#pragma unroll
            for (int c = 0; c < D; ++c) w[c] = t[(size_t)i * D + c];
            Xf<D>::applyT(S, w, u);
#pragma unroll
            for (int c = 0; c < D; ++c) acc[c] += u[c];
        }
    }
#pragma unroll
    for (int off = 4; off > 0; off >>= 1) {
#pragma unroll
        for (int c = 0; c < D; ++c) acc[c] += __shfl_xor_sync(0xffffffffu, acc[c], off, 8);
    }
    if (act && lane < D) {
        double v = acc[0];
#pragma unroll
        for (int c = 1; c < D; ++c) v = (lane == c) ? acc[c] : v;
        rc[(size_t)I * D + lane] = v;
    }
}

// x_i += Ad(rel_i) xc[agg_i]
template <int D>
__global__ void __launch_bounds__(128) amg_prolong_kernel(int n_fine, const int32_t *__restrict__ agg, const double *__restrict__ rel,
                                                          int pad, const double *__restrict__ xc, double *__restrict__ x,
                                                          const DevScalars *sc, int check_done) {
    if (check_done && sc->done) return;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_fine) return;
    const Rel S = load_rel(rel, pad, i);
    const int I = agg[i];
    double v[D], u[D];
#pragma unroll
    for (int c = 0; c < D; ++c) v[c] = xc[(size_t)I * D + c];
    Xf<D>::apply(S, v, u);
#pragma unroll
    for (int c = 0; c < D; ++c) x[(size_t)i * D + c] += u[c];
}

// r.z of the multilevel preconditioner without forming z:  r.(zJ + P0 x_1) = r.zJ + (P0^T r).x_1 = r.zJ + r_1.x_1.
// r.zJ is already in sc->rz_new (pcg_update / pcg_init; summed over the ranks in the partitioned solve), this
// adds the coarse dot product and finishes the PCG scalars (beta, convergence test).
template <int NT>
__global__ void __launch_bounds__(NT) amg_coarse_dot_kernel(int n, const double *__restrict__ r1, const double *__restrict__ x1,
                                                            double *__restrict__ partials, DevScalars *sc, int init, double tol,
                                                            int max_iter) {
    __shared__ double sh[32];
    if (!init && sc->done) return;
    double local = 0;
    for (int t = blockIdx.x * NT + threadIdx.x; t < n; t += gridDim.x * NT) local += r1[t] * x1[t];
    const double bs = block_sum<NT>(local, sh);
    if (threadIdx.x == 0) partials[blockIdx.x] = bs;
    if (last_block(&sc->counters[6])) {
        const double dot = sum_partials<NT>(partials, gridDim.x, sh);
        if (threadIdx.x == 0) {
            sc->rz_new += dot;
            if (init) fin_init(sc, tol, max_iter);
            else fin_update(sc);
        }
    }
}

// Fine level, fused with the search-direction update:  p_i = (zJ_i + P_i x_1[agg_i]) + beta p_i  (zJ = D^-1 r in z).
template <int D, int NT>
__global__ void __launch_bounds__(NT) amg_prolong0_kernel(int nf, const int32_t *__restrict__ agg, const double *__restrict__ rel,
                                                          int pad, const double *__restrict__ xc, const double *__restrict__ z,
                                                          double *__restrict__ p, const DevScalars *sc, int init) {
    if (!init && sc->done) return;
    const double beta = init ? 0.0 : sc->beta;
    for (int i = blockIdx.x * NT + threadIdx.x; i < nf; i += gridDim.x * NT) {
        const Rel S = load_rel(rel, pad, i);
        const int I = agg[i];
        double v[D], u[D];
#pragma unroll
        for (int c = 0; c < D; ++c) v[c] = xc[(size_t)I * D + c];
        Xf<D>::apply(S, v, u);
#pragma unroll
        for (int c = 0; c < D; ++c) {
            const double zc = z[(size_t)i * D + c] + u[c];
            p[(size_t)i * D + c] = init ? zc : zc + beta * p[(size_t)i * D + c];
        }
    }
}

// ---- tail of the V-cycle: every level with at most kTailRows rows, in ONE launch ---------------
// The small levels are latency-bound (dependent index -> value loads, a handful of rows each).
// One thread-block cluster of 8 CTAs walks them all, separated by cluster barriers instead of
// ~5 kernel boundaries per level.  Vectors that change between phases are read with ld.cg (L2),
// since another CTA of the cluster wrote them.
constexpr int kTailRows = 1024, kTailThreads = 512, kTailCtas = 8, kTailMaxLevels = kMaxLevels;

struct TailLevel {
    int n, pad_fine;                                  // rows of this level; pad of the transfer's rel planes
    const int32_t *rowptr, *colidx;                   // operator of this level
    const int32_t *mem_ptr, *mem_idx, *agg;           // transfer (previous level -> this level)
    const double *A, *Dinv, *rel;
    double *r, *x, *x2, *t;
};
struct TailParams {
    int nlev, dense, N;
    const double *inv;
    TailLevel lev[kTailMaxLevels];
};

__device__ __forceinline__ void tail_sync() {
    __threadfence();
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ unsigned tail_cta_rank() {
    unsigned r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}

template <int D, int MODE>
__device__ __forceinline__ void tail_rows(const TailLevel &L, const double *x, double *out, double omega, int gtid) {
    constexpr int groups = kTailThreads * kTailCtas / 8;
    const int g = gtid / 8, l = gtid & 7;
    for (int base = 0; base < L.n; base += groups) {
        const int i = base + g;
        const bool act = i < L.n && l < D;
        double res = act ? __ldcg(L.r + (size_t)i * D + l) : 0.0;
        if (MODE != 0 && act) {
            double acc = 0;
            const int kb = L.rowptr[i], ke = L.rowptr[i + 1];
            for (int k = kb; k < ke; ++k) {
                const double *xj = x + (size_t)L.colidx[k] * D;
                const double *Ak = L.A + (size_t)k * DD + l * D;
#pragma unroll
                for (int c = 0; c < D; ++c) acc += Ak[c] * __ldcg(xj + c);
            }
            res -= acc;
        }
        if (MODE == 1) {
            if (act) out[(size_t)i * D + l] = res;
            continue;
        }
        double z = 0;
#pragma unroll
        for (int c = 0; c < D; ++c) {
            const double rc = __shfl_sync(0xffffffffu, res, c, 8);
            if (act) z += L.Dinv[(size_t)i * sym_size<D>() + sym_off<D>(l, c)] * rc;
        }
        if (act) out[(size_t)i * D + l] = (MODE == 2 ? __ldcg(x + (size_t)i * D + l) : 0.0) + omega * z;
    }
}

template <int D>
__global__ void __cluster_dims__(kTailCtas, 1, 1) __launch_bounds__(kTailThreads)
amg_tail_kernel(const __grid_constant__ TailParams P, double omega, const DevScalars *sc, int check_done) {
    if (check_done && sc->done) return;       // uniform over the cluster: nobody reaches a barrier
    constexpr int NTH = kTailThreads * kTailCtas;
    const int gtid = (int)tail_cta_rank() * kTailThreads + threadIdx.x;
    const int last = P.nlev - 1;
    for (int l = 0; l <= last; ++l) {
        const TailLevel &L = P.lev[l];
        if (l == last) {
            if (P.dense) {
                for (int t = gtid; t < P.N; t += NTH) {
                    double acc = 0;
                    for (int c = 0; c < P.N; ++c) acc += P.inv[(size_t)c * P.N + t] * __ldcg(L.r + c);
                    L.x2[t] = acc;
                }
            } else {            // no dense inverse: five damped block-Jacobi sweeps (a fixed linear operator)
                tail_rows<D, 0>(L, nullptr, L.x, omega, gtid);
                tail_sync();
                for (int k = 0; k < 2; ++k) {
                    tail_rows<D, 2>(L, L.x, L.x2, omega, gtid);
                    tail_sync();
                    tail_rows<D, 2>(L, L.x2, L.x, omega, gtid);
                    tail_sync();
                }
                for (int t = gtid; t < L.n * D; t += NTH) L.x2[t] = __ldcg(L.x + t);
            }
            tail_sync();
            break;
        }
        tail_rows<D, 0>(L, nullptr, L.x, omega, gtid);
        tail_sync();
        tail_rows<D, 1>(L, L.x, L.t, omega, gtid);
        tail_sync();
        const TailLevel &C = P.lev[l + 1];
        for (int I = gtid; I < C.n; I += NTH) {
            double acc[D];
#pragma unroll
            for (int c = 0; c < D; ++c) acc[c] = 0;
            for (int m = C.mem_ptr[I]; m < C.mem_ptr[I + 1]; ++m) {
                const int i = C.mem_idx[m];
                const Rel S = load_rel(C.rel, C.pad_fine, i);
                double w[D], u[D];
#pragma unroll
                for (int c = 0; c < D; ++c) w[c] = __ldcg(L.t + (size_t)i * D + c);
                Xf<D>::applyT(S, w, u);
#pragma unroll
                for (int c = 0; c < D; ++c) acc[c] += u[c];
            }
#pragma unroll
            for (int c = 0; c < D; ++c) C.r[(size_t)I * D + c] = acc[c];
        }
        tail_sync();
    }
    // every level leaves its result in x2 (the host swaps x and x2 after the launch)
    for (int l = last - 1; l >= 0; --l) {
        const TailLevel &L = P.lev[l];
        const TailLevel &C = P.lev[l + 1];
        for (int i = gtid; i < L.n; i += NTH) {
            const Rel S = load_rel(C.rel, C.pad_fine, i);
            const int I = C.agg[i];
            double v[D], u[D];
#pragma unroll
            for (int c = 0; c < D; ++c) v[c] = __ldcg(C.x2 + (size_t)I * D + c);
            Xf<D>::apply(S, v, u);
#pragma unroll
            for (int c = 0; c < D; ++c) L.x[(size_t)i * D + c] = __ldcg(L.x + (size_t)i * D + c) + u[c];
        }
        tail_sync();
        tail_rows<D, 2>(L, L.x, L.x2, omega, gtid);
        tail_sync();
    }
}

// ---- K-cycle ---------------------------------------------------------------------------------------
// A V-cycle over plain aggregates loses a constant factor of the coarse correction at every level (the
// Galerkin operators of piecewise-rigid transfers are too stiff), so the PCG iteration count grows with the
// depth of the hierarchy.  On the first `kdepth` coarse levels the coarse problem  A_l x = r  is therefore solved
// by TWO conjugate-gradient steps preconditioned with the cycle below (Notay's K-cycle), in closed form:
//   z1 = C(r);          q1 = A z1;  rho1 = z1.q1;  alpha1 = z1.r / rho1;   r' = r - alpha1 q1
//   z2 = C(r');         q2 = A z2;  gamma = z2.q1; beta = z2.q2;  alpha2 = z2.r'
//   rho2 = beta - gamma^2 / rho1;   x = (alpha1 - alpha2 gamma / (rho1 rho2)) z1 + (alpha2 / rho2) z2
// Levels with many rows run as ordinary launches (they are bandwidth-bound and want the whole machine in
// flight); every level from `coop_first` down is latency-bound and is walked by one cooperative kernel.
// All reductions are two-stage with a fixed order, so the preconditioner stays bitwise reproducible.

__device__ __forceinline__ void kscal_first(KScal *k, double zq, double zr) {
    const bool ok = zq > 0 && isfinite(zq);
    k->rho1 = ok ? zq : 1.0;
    k->alpha1 = ok ? zr / zq : 0.0;
    k->c1 = k->alpha1;
    k->c2 = 0.0;
}
__device__ __forceinline__ void kscal_second(KScal *k, double beta, double alpha2, double gamma) {
    const double rho2 = beta - gamma * gamma / k->rho1;
    if (rho2 > 0 && isfinite(rho2)) {
        k->c1 = k->alpha1 - alpha2 * gamma / (k->rho1 * rho2);
        k->c2 = alpha2 / rho2;
    } else {        // the second direction adds nothing (or broke down): keep the one-step result
        k->c1 = k->alpha1;
        k->c2 = 0.0;
    }
}

// q = A z (optional store) and the dot products z.q, z.v1, z.v2 of one K-cycle step; second = 0: first step
// (v1 = r), second = 1: second step (v1 = r', v2 = q1).  An 8-lane group owns one block row.
template <int D, int NT>
__global__ void __launch_bounds__(NT) amg_kdots_kernel(int n, const int32_t *__restrict__ rowptr, const int32_t *__restrict__ colidx,
                                                       const double *__restrict__ A, const double *__restrict__ z,
                                                       const double *__restrict__ v1, const double *__restrict__ v2,
                                                       double *__restrict__ q, double *__restrict__ partials, KScal *ks,
                                                       int second, DevScalars *sc, int check_done) {
    __shared__ double sh[32];
    if (check_done && sc->done) return;
    const int g0 = blockIdx.x * (NT / 8) + threadIdx.x / 8, l = threadIdx.x & 7, ng = gridDim.x * (NT / 8);
    double d0 = 0, d1 = 0, d2 = 0;
    for (int i = g0; i < n; i += ng) {
        if (l >= D) continue;
        double acc = 0;
        for (int k = rowptr[i]; k < rowptr[i + 1]; ++k) {
            const double *zj = z + (size_t)colidx[k] * D;
            const double *Ak = A + (size_t)k * DD + l * D;
#pragma unroll
            for (int c = 0; c < D; ++c) acc += Ak[c] * zj[c];
        }
        const double zi = z[(size_t)i * D + l];
        if (q) q[(size_t)i * D + l] = acc;
        d0 += zi * acc;
        d1 += zi * v1[(size_t)i * D + l];
        if (v2) d2 += zi * v2[(size_t)i * D + l];
    }
    const double s0 = block_sum<NT>(d0, sh);
    const double s1 = block_sum<NT>(d1, sh);
    const double s2 = block_sum<NT>(d2, sh);
    if (threadIdx.x == 0) {
        partials[blockIdx.x] = s0;
        partials[kMaxPartials + blockIdx.x] = s1;
        partials[2 * kMaxPartials + blockIdx.x] = s2;
    }
    if (last_block(&sc->counters[7])) {
        const double t0 = sum_partials<NT>(partials, gridDim.x, sh);
        const double t1 = sum_partials<NT>(partials + kMaxPartials, gridDim.x, sh);
        const double t2 = sum_partials<NT>(partials + 2 * kMaxPartials, gridDim.x, sh);
        if (threadIdx.x == 0) {
            if (!second) kscal_first(ks, t0, t1);
            else kscal_second(ks, t0, t1, t2);
        }
    }
}

// out = a - alpha1 q   (mode 0: the residual after the first inner step)
// out = c1 a + c2 q    (mode 1: the combined correction)
__global__ void amg_kaxpy_kernel(int n, const double *__restrict__ a, const double *__restrict__ q, double *__restrict__ out,
                                 const KScal *ks, int mode, const DevScalars *sc, int check_done) {
    if (check_done && sc->done) return;
    const double c1 = mode ? ks->c1 : 1.0, c2 = mode ? ks->c2 : -ks->alpha1;
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < n; t += gridDim.x * blockDim.x) out[t] = c1 * a[t] + c2 * q[t];
}

// ---- cooperative kernel: every level from `coop_first` down, K-cycle on the first P.kdepth of them ----
constexpr int kCoopThreads = 512, kCoopRows = 24000;

struct CoopLevel {
    int n, pad_fine;
    int G;                      // 8-lane groups that share one block row in the cooperative kernel (1, 2 or 4)
    const int32_t *rowptr, *colidx, *mem_ptr, *mem_idx, *agg, *acol;
    const double *A, *Dinv, *rel;
    double *r, *x, *x2, *t, *z1, *q1, *rp, *z2;
};
struct CoopParams {
    int nlev, dense, N, kdepth;
    unsigned kmask;
    const double *inv;
    double *dots;                 // [3][gridDim.x]
    long long *dbg;               // S3O_COOP_DBG: clock64() of CTA 0 after every barrier (diagnostic), else null
    CoopLevel lev[kMaxLevels];
};

// A residual given as  a - alpha b  (b == nullptr: a).  The second inner step of a K-cycle level works on
// r' = r - alpha1 q1, which is formed where it is read instead of being stored.
struct RSpec { const double *a, *b; double alpha; };
__device__ __forceinline__ double rget(const RSpec &R, size_t t) {
    double v = __ldcg(R.a + t);
    if (R.b) v -= R.alpha * __ldcg(R.b + t);
    return v;
}
// A coarse correction given as  c1 a + c2 b  (b == nullptr: a): the result of a K-cycle level is combined where
// the parent prolongs it.
struct XSpec { const double *a, *b; double c1, c2; };
__device__ __forceinline__ double xget(const XSpec &X, size_t t) {
    double v = __ldcg(X.a + t);
    if (X.b) v = X.c1 * v + X.c2 * __ldcg(X.b + t);
    return v;
}

// shuffle inside the 8-lane group of a warp (groups of one warp may run different trip counts)
__device__ __forceinline__ double gshfl(unsigned gmask, double v, int src_in_group) {
    return __shfl_sync(gmask, v, (threadIdx.x & 24) + src_in_group);
}

// mode 0: out = omega Dinv rin;  2: out = x + omega Dinv (rin - A x)      (coarsest level without a dense inverse)
template <int D, int MODE>
__device__ __forceinline__ void coop_rows(const CoopLevel &L, const double *rin, const double *x, double *out, double omega,
                                          int gtid, int nth) {
    const int groups = nth / 8, g = gtid / 8, l = gtid & 7;
    for (int base = 0; base < L.n; base += groups) {
        const int i = base + g;
        const bool act = i < L.n && l < D;
        double res = act ? __ldcg(rin + (size_t)i * D + l) : 0.0;
        if (MODE != 0 && act) {
            double acc = 0;
            const int kb = L.rowptr[i], ke = L.rowptr[i + 1];
            for (int k = kb; k < ke; ++k) {
                const double *xj = x + (size_t)L.colidx[k] * D;
                const double *Ak = L.A + (size_t)k * DD + l * D;
#pragma unroll
                for (int c = 0; c < D; ++c) acc += Ak[c] * __ldcg(xj + c);
            }
            res -= acc;
        }
        double z = 0;
#pragma unroll
        for (int c = 0; c < D; ++c) {
            const double rc = __shfl_sync(0xffffffffu, res, c, 8);
            if (act) z += L.Dinv[(size_t)i * sym_size<D>() + sym_off<D>(l, c)] * rc;
        }
        if (act) out[(size_t)i * D + l] = (MODE == 2 ? __ldcg(x + (size_t)i * D + l) : 0.0) + omega * z;
    }
}

// ---- row phases of the cooperative kernel -------------------------------------------------------
// These levels live in L2 and a phase is a chain of load latencies, so (1) a block row is shared by G 8-lane groups
// (G = 4: a whole warp) when the level has fewer rows than the grid has groups -- group g takes the blocks
// g*U.., (g+G)*U.. and the partial sums meet in a fixed butterfly -- and (2) every batch of U blocks issues ALL its loads
// (indices, then vectors / inverses / block rows, spread over the lanes and completed by shuffles) before any arithmetic.
template <int G> __device__ __forceinline__ unsigned row_mask() {
    const int lane = threadIdx.x & 31;
    return G == 4 ? 0xffffffffu : (G == 2 ? 0xffffu << (lane & 16) : 0xffu << (lane & 24));
}
template <int G> __device__ __forceinline__ double row_sum(unsigned rmask, double v) {
    if (G >= 2) v += __shfl_xor_sync(rmask, v, 8);
    if (G == 4) v += __shfl_xor_sync(rmask, v, 16);
    return v;
}

// Way down, fused: the first smoothing sweep starts from zero, x = omega Dinv r, so the residual after it is
// t_i = r_i - sum_j A_ij (omega Dinv_j r_j) with the neighbours' sweep formed on the fly: one phase instead of two.
template <int D, int G>
__device__ __forceinline__ void coop_down(const CoopLevel &L, const RSpec R, double omega, int gtid, int nth) {
    constexpr int U = 3, LPR = 8 * G;
    const int lane = threadIdx.x & 31, sub = lane & (LPR - 1), g = sub >> 3, l = sub & 7;
    const unsigned gmask = 0xffu << (lane & 24), rmask = row_mask<G>();
    const int lc = l < D ? l : 0;             // lane 7 shadows lane 0 (keeps the group's shuffles convergent)
    for (int i = gtid / LPR; i < L.n; i += nth / LPR) {
        const double ri = rget(R, (size_t)i * D + lc);
        double xi = 0;
#pragma unroll
        for (int c = 0; c < D; ++c) xi += L.Dinv[(size_t)i * sym_size<D>() + sym_off<D>(lc, c)] * gshfl(gmask, ri, c);
        xi *= omega;
        double acc = 0;
        const int kb = L.rowptr[i], ke = L.rowptr[i + 1];
        for (int k0 = kb + g * U; k0 < ke; k0 += G * U) {
            int j[U];
            double rj[U], dv[U][D], av[U][D];
#pragma unroll
            for (int u = 0; u < U; ++u) j[u] = L.colidx[min(k0 + u, ke - 1)];
#pragma unroll
            for (int u = 0; u < U; ++u) rj[u] = rget(R, (size_t)j[u] * D + lc);
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const double *Ak = L.A + (size_t)min(k0 + u, ke - 1) * DD + lc * D;
#pragma unroll
                for (int c = 0; c < D; ++c) {
                    dv[u][c] = L.Dinv[(size_t)j[u] * sym_size<D>() + sym_off<D>(lc, c)];
                    av[u][c] = Ak[c];
                }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (k0 + u >= ke) break;                 // uniform inside the group
                double xj = 0;
#pragma unroll
                for (int c = 0; c < D; ++c) xj += dv[u][c] * gshfl(gmask, rj[u], c);
                xj *= omega;
#pragma unroll
                for (int c = 0; c < D; ++c) acc += av[u][c] * gshfl(gmask, xj, c);
            }
        }
        acc = row_sum<G>(rmask, acc);
        if (g == 0 && l < D) {
            L.x[(size_t)i * D + l] = xi;
            L.t[(size_t)i * D + l] = ri - acc;
        }
    }
}

// r_{l+1} = P^T t: an 8-lane group per aggregate, lane m takes members m, m+8, ... and a fixed butterfly adds them
template <int D>
__device__ __forceinline__ void coop_restrict(const CoopLevel &C, const double *t, int gtid, int nth) {
    const int groups = nth / 8, g = gtid / 8, lane = gtid & 7;
    const unsigned gmask = 0xffu << (threadIdx.x & 24);
    for (int I = g; I < C.n; I += groups) {
        double acc[D];
#pragma unroll
        for (int c = 0; c < D; ++c) acc[c] = 0;
        for (int m = C.mem_ptr[I] + lane; m < C.mem_ptr[I + 1]; m += 8) {
            const int i = C.mem_idx[m];
            const Rel S = load_rel(C.rel, C.pad_fine, i);
            double w[D], u[D];
#pragma unroll
            for (int c = 0; c < D; ++c) w[c] = __ldcg(t + (size_t)i * D + c);
            Xf<D>::applyT(S, w, u);
#pragma unroll
            for (int c = 0; c < D; ++c) acc[c] += u[c];
        }
#pragma unroll
        for (int off = 4; off > 0; off >>= 1) {
#pragma unroll
            for (int c = 0; c < D; ++c) acc[c] += __shfl_xor_sync(gmask, acc[c], off, 8);
        }
        if (lane < D) {
            double v = acc[0];
#pragma unroll
            for (int c = 1; c < D; ++c) v = (lane == c) ? acc[c] : v;
            C.r[(size_t)I * D + lane] = v;
        }
    }
}

// Way up, fused: x' = x + P xc (the child's correction, combined on the fly) and the second smoothing sweep
// out = x' + omega Dinv (r - A x'), with the neighbours' prolonged values formed where they are read.  Per block a lane
// loads two of the 13 frame entries, one entry of the correction and of x, and its row of the block.
template <int D, int G>
__device__ __forceinline__ void coop_up(const CoopLevel &F, const CoopLevel &C, const XSpec X, const RSpec R, double *out,
                                        double omega, int gtid, int nth) {
    constexpr int U = 2, LPR = 8 * G;
    const int lane = threadIdx.x & 31, sub = lane & (LPR - 1), g = sub >> 3, l = sub & 7;
    const unsigned gmask = 0xffu << (lane & 24), rmask = row_mask<G>();
    const int lc = l < D ? l : 0;
    const size_t pad = (size_t)C.pad_fine;
    for (int i = gtid / LPR; i < F.n; i += nth / LPR) {
        double acc = 0, xi_l = 0;
        const int kb = F.rowptr[i], ke = F.rowptr[i + 1];
        for (int k0 = kb + g * U; k0 < ke; k0 += G * U) {
            int j[U], I[U];
            double f0[U], f1[U], xcv[U], xv[U], av[U][D];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int k = min(k0 + u, ke - 1);
                j[u] = F.colidx[k];
                I[u] = F.acol[k];
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                f0[u] = __ldg(C.rel + (size_t)l * pad + j[u]);                       // frame entries 0..7
                f1[u] = __ldg(C.rel + (size_t)(8 + (l < 5 ? l : 4)) * pad + j[u]);   // frame entries 8..12
                xcv[u] = xget(X, (size_t)I[u] * D + lc);
                xv[u] = __ldcg(F.x + (size_t)j[u] * D + lc);
                const double *Ak = F.A + (size_t)min(k0 + u, ke - 1) * DD + lc * D;
#pragma unroll
                for (int c = 0; c < D; ++c) av[u][c] = Ak[c];
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (k0 + u >= ke) break;
                Rel S;
#pragma unroll
                for (int q = 0; q < 8; ++q) S.R[q] = gshfl(gmask, f0[u], q);
                S.R[8] = gshfl(gmask, f1[u], 0);
                S.t[0] = gshfl(gmask, f1[u], 1); S.t[1] = gshfl(gmask, f1[u], 2); S.t[2] = gshfl(gmask, f1[u], 3);
                S.s = gshfl(gmask, f1[u], 4);
                double xc[D], v[D];
#pragma unroll
                for (int c = 0; c < D; ++c) xc[c] = gshfl(gmask, xcv[u], c);
                Xf<D>::apply(S, xc, v);
                double own = 0;
#pragma unroll
                for (int c = 0; c < D; ++c) {
                    const double xpc = gshfl(gmask, xv[u], c) + v[c];
                    acc += av[u][c] * xpc;
                    own = (c == lc) ? xpc : own;
                }
                if (j[u] == i) xi_l = own;
            }
        }
        acc = row_sum<G>(rmask, acc);
        xi_l = row_sum<G>(rmask, xi_l);         // the diagonal block sits in exactly one group
        const double res = rget(R, (size_t)i * D + lc) - acc;
        double z = 0;
#pragma unroll
        for (int c = 0; c < D; ++c) z += F.Dinv[(size_t)i * sym_size<D>() + sym_off<D>(lc, c)] * gshfl(gmask, res, c);
        if (g == 0 && l < D) out[(size_t)i * D + l] = xi_l + omega * z;
    }
}

// dot products of one inner step over the grid: per-CTA partials -> grid barrier -> every CTA adds the
// partials in the same fixed order (all CTAs obtain identical bits).  The barrier inside also orders the
// store of q before whatever phase follows.
template <int D, int G>
__device__ __forceinline__ void coop_kdots(const CoopLevel &L, const double *z, const RSpec V1, const double *v2, double *q,
                                           double *dots, double out[3], int gtid, int nth, double *sh, const GridBarrier &gb,
                                           unsigned &phase) {
    constexpr int U = 6, LPR = 8 * G;
    const int lane = threadIdx.x & 31, sub = lane & (LPR - 1), g = sub >> 3, l = sub & 7;
    const unsigned gmask = 0xffu << (lane & 24), rmask = row_mask<G>();
    const int lc = l < D ? l : 0;
    double d0 = 0, d1 = 0, d2 = 0;
    for (int i = gtid / LPR; i < L.n; i += nth / LPR) {
        double acc = 0;
        const int kb = L.rowptr[i], ke = L.rowptr[i + 1];
        for (int k0 = kb + g * U; k0 < ke; k0 += G * U) {
            int j[U];
            double zv[U], av[U][D];
#pragma unroll
            for (int u = 0; u < U; ++u) j[u] = L.colidx[min(k0 + u, ke - 1)];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                zv[u] = __ldcg(z + (size_t)j[u] * D + lc);
                const double *Ak = L.A + (size_t)min(k0 + u, ke - 1) * DD + lc * D;
#pragma unroll
                for (int c = 0; c < D; ++c) av[u][c] = Ak[c];
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (k0 + u >= ke) break;
#pragma unroll
                for (int c = 0; c < D; ++c) acc += av[u][c] * gshfl(gmask, zv[u], c);
            }
        }
        acc = row_sum<G>(rmask, acc);
        if (g == 0 && l < D) {
            const double zi = __ldcg(z + (size_t)i * D + l);
            if (q) q[(size_t)i * D + l] = acc;
            d0 += zi * acc;
            d1 += zi * rget(V1, (size_t)i * D + l);
            if (v2) d2 += zi * __ldcg(v2 + (size_t)i * D + l);
        }
    }
    const double s0 = block_sum<kCoopThreads>(d0, sh);
    const double s1 = block_sum<kCoopThreads>(d1, sh);
    const double s2 = block_sum<kCoopThreads>(d2, sh);
    const int Gd = gridDim.x;
    if (threadIdx.x == 0) { dots[blockIdx.x] = s0; dots[Gd + blockIdx.x] = s1; dots[2 * Gd + blockIdx.x] = s2; }
    grid_barrier(gb, phase);
    __shared__ double tot[3];
    if (threadIdx.x < 32) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            double v = 0;
            for (int t = threadIdx.x; t < Gd; t += 32) v += __ldcg(dots + k * Gd + t);
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
            if (threadIdx.x == 0) tot[k] = v;
        }
    }
    __syncthreads();
    out[0] = tot[0]; out[1] = tot[1]; out[2] = tot[2];
    __syncthreads();
}

// Phases per level visit: way down 2 (fused sweep + residual, restriction), way up 1 (fused prolongation + sweep);
// a K-cycle level adds one phase per inner step (product + dot products).  The dots buffer alternates between two
// halves, so a step's partial sums are never overwritten while a slow CTA still reads the previous step's.
template <int D>
__global__ void __launch_bounds__(kCoopThreads, 1)
amg_coop_kernel(const __grid_constant__ CoopParams P, double omega, const DevScalars *sc, int check_done,
                const GridBarrier gb) {
    if (check_done && sc->done) return;       // uniform over the grid: nobody reaches a barrier
    unsigned phase = 0;
    __shared__ double sh[32];
    const int nth = gridDim.x * kCoopThreads, gtid = blockIdx.x * kCoopThreads + threadIdx.x;
    auto stamp = [&]() { if (P.dbg && gtid == 0 && phase < 120) P.dbg[phase] = clock64(); };
    auto gsync = [&]() { grid_barrier(gb, phase); stamp(); };
    stamp();
    const int last = P.nlev - 1;
    // explicit recursion state: residual of the cycle in progress at every level, where its result goes, the
    // inner step of a K-cycle level and its scalars
    RSpec cur_r[kMaxLevels];
    double *cur_out[kMaxLevels];
    int step[kMaxLevels];
    KScal ks[kMaxLevels];
    int flip = 0;
    auto is_k = [&](int l) { return ((P.kmask >> l) & 1u) && l < last; };
    int l = 0;
    cur_r[0] = RSpec{ P.lev[0].r, nullptr, 0.0 };
    cur_out[0] = is_k(0) ? P.lev[0].z1 : P.lev[0].x2;
    step[0] = 0;
    for (;;) {
        // ---------------- descend: cycle at level l on cur_r[l] -----------------------------------
        for (;;) {
            const CoopLevel &L = P.lev[l];
            if (l == last) {
                // the coarsest level is never a K-cycle level: its residual is the plain vector L.r
                if (P.dense) {
                    // x = A^-1 r: a warp per entry, reading a row of the (symmetric) inverse contiguously
                    const int lane = threadIdx.x & 31;
                    for (int t = gtid >> 5; t < P.N; t += nth >> 5) {
                        double acc = 0;
#pragma unroll 8
                        for (int c = lane; c < P.N; c += 32) acc += P.inv[(size_t)t * P.N + c] * __ldcg(L.r + c);
#pragma unroll
                        for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
                        if (lane == 0) cur_out[l][t] = acc;
                    }
                } else if (l == 0) {    // a single coarse level too large for the dense inverse: five damped sweeps
                    coop_rows<D, 0>(L, L.r, nullptr, L.x, omega, gtid, nth);
                    gsync();
                    coop_rows<D, 2>(L, L.r, L.x, L.t, omega, gtid, nth);
                    gsync();
                    coop_rows<D, 2>(L, L.r, L.t, L.x, omega, gtid, nth);
                    gsync();
                    coop_rows<D, 2>(L, L.r, L.x, L.t, omega, gtid, nth);
                    gsync();
                    coop_rows<D, 2>(L, L.r, L.t, cur_out[l], omega, gtid, nth);
                } else {
                    coop_rows<D, 0>(L, L.r, nullptr, L.x, omega, gtid, nth);
                    gsync();
                    coop_rows<D, 2>(L, L.r, L.x, L.t, omega, gtid, nth);
                    gsync();
                    coop_rows<D, 2>(L, L.r, L.t, L.x, omega, gtid, nth);
                    gsync();
                    coop_rows<D, 2>(L, L.r, L.x, L.t, omega, gtid, nth);
                    gsync();
                    coop_rows<D, 2>(L, L.r, L.t, cur_out[l], omega, gtid, nth);
                }
                gsync();
                break;
            }
            if (L.G == 4) coop_down<D, 4>(L, cur_r[l], omega, gtid, nth);
            else if (L.G == 2) coop_down<D, 2>(L, cur_r[l], omega, gtid, nth);
            else coop_down<D, 1>(L, cur_r[l], omega, gtid, nth);
            gsync();
            coop_restrict<D>(P.lev[l + 1], L.t, gtid, nth);
            gsync();
            ++l;
            cur_r[l] = RSpec{ P.lev[l].r, nullptr, 0.0 };
            cur_out[l] = is_k(l) ? P.lev[l].z1 : P.lev[l].x2;
            step[l] = 0;
        }
        // ---------------- ascend: cur_out[l] holds the result of a cycle at level l ---------------
        bool again = false;
        for (;;) {
            const CoopLevel &L = P.lev[l];
            XSpec X{ L.x2, nullptr, 1.0, 0.0 };       // how the parent reads the solution of level l
            if (is_k(l)) {
                double d[3];
                double *dots = P.dots + (flip ? 3 * gridDim.x : 0);
                flip ^= 1;
                if (step[l] == 0) {
                    if (L.G == 4) coop_kdots<D, 4>(L, L.z1, cur_r[l], nullptr, L.q1, dots, d, gtid, nth, sh, gb, phase);
                    else if (L.G == 2) coop_kdots<D, 2>(L, L.z1, cur_r[l], nullptr, L.q1, dots, d, gtid, nth, sh, gb, phase);
                    else coop_kdots<D, 1>(L, L.z1, cur_r[l], nullptr, L.q1, dots, d, gtid, nth, sh, gb, phase);
                    stamp();
                    kscal_first(&ks[l], d[0], d[1]);
                    step[l] = 1;
                    cur_r[l] = RSpec{ L.r, L.q1, ks[l].alpha1 };      // r' = r - alpha1 q1, formed where it is read
                    cur_out[l] = L.z2;
                    again = true;
                    break;                      // second cycle at the same level
                }
                if (L.G == 4) coop_kdots<D, 4>(L, L.z2, cur_r[l], L.q1, nullptr, dots, d, gtid, nth, sh, gb, phase);
                else if (L.G == 2) coop_kdots<D, 2>(L, L.z2, cur_r[l], L.q1, nullptr, dots, d, gtid, nth, sh, gb, phase);
                else coop_kdots<D, 1>(L, L.z2, cur_r[l], L.q1, nullptr, dots, d, gtid, nth, sh, gb, phase);
                stamp();
                kscal_second(&ks[l], d[0], d[1], d[2]);
                X = XSpec{ L.z1, L.z2, ks[l].c1, ks[l].c2 };
                if (l == 0) {                   // the caller reads a plain vector
                    for (int t = gtid; t < L.n * D; t += nth) L.x2[t] = xget(X, t);
                    return;
                }
            }
            if (l == 0) return;
            --l;
            if (P.lev[l].G == 4) coop_up<D, 4>(P.lev[l], P.lev[l + 1], X, cur_r[l], cur_out[l], omega, gtid, nth);
            else if (P.lev[l].G == 2) coop_up<D, 2>(P.lev[l], P.lev[l + 1], X, cur_r[l], cur_out[l], omega, gtid, nth);
            else coop_up<D, 1>(P.lev[l], P.lev[l + 1], X, cur_r[l], cur_out[l], omega, gtid, nth);
            gsync();
        }
        (void)again;
    }
}

// V-cycle: first level handled by the cluster tail kernel (a large coarsest level: the tail still runs its sweeps)
int tail_first(const AmgState *st) {
    const int nl = (int)st->lev.size();
    int lt = 0;
    while (lt < nl && st->lev[lt].n > kTailRows) ++lt;
    return lt == nl ? nl - 1 : lt;
}
// K-cycle: grid of the cooperative kernel entered at level l, and the 8-lane groups that share one block row of an
// n-row level on that grid (as many as the grid has to spare)
int coop_grid_at(const AmgState *st, int l) {
    const int grid = (st->lev[l].n * 8 + kCoopThreads - 1) / kCoopThreads;
    return std::max(8, std::min(grid, st->coop_grid));
}
int coop_row_groups(int grid, int n) {
    const long long lanes = (long long)grid * kCoopThreads;
    return (long long)n * 32 <= lanes ? 4 : ((long long)n * 16 <= lanes ? 2 : 1);
}

template <class T>
int up(s3o_problem *p, T **dst, const std::vector<T> &src) { return upload(p, dst, src); }

void free_level(LevelDev &L) {
    dev_free(L.agg); dev_free(L.mem_ptr); dev_free(L.mem_idx); dev_free(L.vid);
    dev_free(L.rowptr); dev_free(L.colidx); dev_free(L.blk_row); dev_free(L.dpos);
    dev_free(L.gal_ptr); dev_free(L.gal_ent); dev_free(L.gal_i); dev_free(L.gal_j); dev_free(L.gal_order); dev_free(L.gal_out); dev_free(L.gal_mirror);
    dev_free(L.rel); dev_free(L.A); dev_free(L.Dinv); dev_free(L.r); dev_free(L.x); dev_free(L.x2); dev_free(L.t);
    dev_free(L.z1); dev_free(L.q1); dev_free(L.rp); dev_free(L.z2); dev_free(L.acol);
    dev_free(L.Kd); dev_free(L.M);
}

// Partitioned solve: rewrite level 0 of the global hierarchy in this rank's local indices.
// Local fine indices are the rank's Hessian rows (owned first, then ghosts); coarse indices stay global.
void localize_fine_level(s3o_problem *p, const HostStructure &Sg, AmgState *st) {
    const PartitionPlan &P = p->plan;
    const HostStructure &S = p->S;
    const int D = p->d;
    AmgHostLevel &H = st->host[0];
    const int nloc = S.nf, world = P.world;
    st->dist = true;
    st->n_own = P.n_own;
    // coarse rows per rank: aggregates are numbered by ascending root, roots never leave their rank's range
    std::vector<int> crow(world + 1, H.n);
    for (int q = 0; q <= world; ++q)
        crow[q] = (int)(std::lower_bound(H.root.begin(), H.root.end(), (int32_t)std::min<int64_t>((int64_t)q * P.seg, P.nf_global)) - H.root.begin());
    crow[world] = H.n;
    st->r_off.resize(world); st->r_cnt.resize(world); st->a_off.resize(world); st->a_cnt.resize(world);
    for (int q = 0; q < world; ++q) {
        st->r_off[q] = (size_t)crow[q] * D;
        st->r_cnt[q] = (size_t)(crow[q + 1] - crow[q]) * D;
        st->a_off[q] = (size_t)H.rowptr[crow[q]] * DD;
        st->a_cnt[q] = (size_t)(H.rowptr[crow[q + 1]] - H.rowptr[crow[q]]) * DD;
        st->r_max = std::max(st->r_max, st->r_cnt[q]);
    }
    const int Ilo = crow[P.rank], Ihi = crow[P.rank + 1];
    auto local_of = [&](int g) { return P.lhidx[Sg.free2v[g]]; };     // global Hessian index -> local index (or -1)
    // aggregate (global coarse id) of every local vertex
    std::vector<int32_t> agg(nloc);
    for (int li = 0; li < nloc; ++li) agg[li] = H.agg[P.ghidx[S.free2v[li]]];
    // members of my aggregates, in local indices (all owned)
    std::vector<int32_t> mem_ptr(H.n + 1, 0), mem_idx;
    for (int I = 0; I < H.n; ++I) {
        if (I >= Ilo && I < Ihi)
            for (int m = H.mem_ptr[I]; m < H.mem_ptr[I + 1]; ++m) mem_idx.push_back(local_of(H.mem_idx[m]));
        mem_ptr[I + 1] = (int32_t)mem_idx.size();
    }
    // Galerkin entries of my coarse rows, with local block / vertex indices
    std::vector<int32_t> gptr(H.nub + 1, 0), gent, gi, gj;
    for (int ub = 0; ub < H.nub; ++ub) {
        if (H.gal_I[ub] >= Ilo && H.gal_I[ub] < Ihi) {
            for (int e = H.gal_ptr[ub]; e < H.gal_ptr[ub + 1]; ++e) {
                const int flag = H.gal_ent[e] & 3;
                const int li = local_of(H.gal_i[e]), lj = local_of(H.gal_j[e]);
                int k = S.rowptr[li];                                   // diagonal block
                if (li != lj) {
                    const int32_t *b = S.colidx.data() + S.rowptr[li] + 1, *en = S.colidx.data() + S.rowptr[li + 1];
                    k = (int)(std::lower_bound(b, en, lj) - S.colidx.data());
                }
                gent.push_back((k << 2) | flag);
                gi.push_back(li);
                gj.push_back(lj);
            }
        }
        gptr[ub + 1] = (int32_t)gent.size();
    }
    H.n_fine = nloc;
    H.agg.swap(agg);
    H.mem_ptr.swap(mem_ptr);
    H.mem_idx.swap(mem_idx);
    H.gal_ptr.swap(gptr);
    H.gal_ent.swap(gent);
    H.gal_i.swap(gi);
    H.gal_j.swap(gj);
}

}  // namespace

void amg_destroy(s3o_problem *p) {
    if (!p->amg) return;
    for (auto &L : p->amg->lev) free_level(L);
    dev_free(p->amg->d_vid0);
    dev_free(p->amg->d_dense);
    dev_free(p->amg->d_rpad);
    dev_free(p->amg->d_unpad_src);
    dev_free(p->amg->d_scal_pos);
    dev_free(p->amg->d_ks);
    dev_free(p->amg->d_rowbuf);
    dev_free(p->amg->d_cdots);
    delete p->amg;
    p->amg = nullptr;
}

int amg_levels(const s3o_problem *p) { return p->amg ? (int)p->amg->lev.size() : 0; }

// Builds the hierarchy for the current structure (host) and uploads it.  Returns S3O_OK with no
// levels when the graph is too small to coarsen (the caller then stays with block-Jacobi).
int amg_setup(s3o_problem *p) {
    if (p->amg) return S3O_OK;
    if (p->kind == S3O_KIND_BA) { set_error("multilevel preconditioner: pose-graph problems only"); return S3O_ERR_UNSUPPORTED; }
    const int D = p->d;
    AmgState *st = new AmgState();
    p->amg = st;
    if (p->dist) {
        // every rank builds the same global hierarchy (aggregates confined to the ranks' vertex ranges),
        // then keeps the part of the fine transfer that touches its own rows
        HostStructure Sg;
        build_structure_host(p->nv, p->fixed.data(), (int)p->gv0.size(), p->gv0.data(), p->gv1.data(), Sg);
        amg_build_hierarchy(Sg, Sg.nf >= kBigGraph ? kCoarsestMaxBig : kCoarsestMax, kMaxLevels, st->host, p->plan.seg);
        if (!st->host.empty()) localize_fine_level(p, Sg, st);
    } else {
        amg_build_hierarchy(p->S, p->S.nf >= kBigGraph ? kCoarsestMaxBig : kCoarsestMax, kMaxLevels, st->host);
    }
    const int nl = (int)st->host.size();
    if (nl == 0) return S3O_OK;
    setup_mark("  hierarchy: host build");
    int rc = up(p, &st->d_vid0, p->S.free2v);
    st->lev.resize(nl);
    for (int l = 0; l < nl && !rc; ++l) {
        const AmgHostLevel &H = st->host[l];
        LevelDev &L = st->lev[l];
        L.n_fine = H.n_fine; L.n = H.n; L.nblk = (int)H.colidx.size(); L.nub = H.nub; L.pad_fine = pad32(H.n_fine);
        rc = rc ? rc : up(p, &L.agg, H.agg);
        rc = rc ? rc : up(p, &L.mem_ptr, H.mem_ptr);
        rc = rc ? rc : up(p, &L.mem_idx, H.mem_idx);
        rc = rc ? rc : up(p, &L.vid, H.vid);
        rc = rc ? rc : up(p, &L.rowptr, H.rowptr);
        rc = rc ? rc : up(p, &L.colidx, H.colidx);
        rc = rc ? rc : up(p, &L.blk_row, H.blk_row);
        rc = rc ? rc : up(p, &L.dpos, H.dpos);
        rc = rc ? rc : up(p, &L.gal_ptr, H.gal_ptr);
        rc = rc ? rc : up(p, &L.gal_ent, H.gal_ent);
        rc = rc ? rc : up(p, &L.gal_i, H.gal_i);
        rc = rc ? rc : up(p, &L.gal_j, H.gal_j);
        rc = rc ? rc : up(p, &L.gal_out, H.gal_out);
        setup_mark("    level: list uploads");
        {   // the lists may have been localised (partitioned solve): order by their final lengths
            std::vector<int32_t> order(H.nub);
            for (int u = 0; u < H.nub; ++u) order[u] = u;
            std::stable_sort(order.begin(), order.end(), [&](int32_t a, int32_t b) {
                return H.gal_ptr[a + 1] - H.gal_ptr[a] > H.gal_ptr[b + 1] - H.gal_ptr[b];
            });
            rc = rc ? rc : up(p, &L.gal_order, order);
        }
        rc = rc ? rc : up(p, &L.gal_mirror, H.gal_mirror);
        setup_mark("    level: order sort");
        rc = rc ? rc : dev_alloc(&L.rel, (size_t)NREL * L.pad_fine);
        rc = rc ? rc : dev_alloc(&L.A, (size_t)L.nblk * DD);
        rc = rc ? rc : dev_alloc(&L.Dinv, (size_t)L.n * DD);
        rc = rc ? rc : dev_alloc(&L.Kd, (size_t)L.n * DD);
        rc = rc ? rc : dev_alloc(&L.M, (size_t)L.n * DD);
        rc = rc ? rc : dev_alloc(&L.r, (size_t)L.n * D + (l == 0 ? st->r_max + 2 : 0));
        rc = rc ? rc : dev_alloc(&L.x, (size_t)L.n * D);
        rc = rc ? rc : dev_alloc(&L.x2, (size_t)L.n * D);
        rc = rc ? rc : dev_alloc(&L.t, (size_t)L.n * D);
        rc = rc ? rc : dev_alloc(&L.z1, (size_t)L.n * D);
        rc = rc ? rc : dev_alloc(&L.q1, (size_t)L.n * D);
        rc = rc ? rc : dev_alloc(&L.rp, (size_t)L.n * D);
        rc = rc ? rc : dev_alloc(&L.z2, (size_t)L.n * D);
        setup_mark("    level: allocations");
        if (l + 1 < nl) {       // aggregate of every block's column vertex in the transfer to the next level
            const AmgHostLevel &N = st->host[l + 1];
            std::vector<int32_t> acol(H.colidx.size());
            for (size_t k = 0; k < H.colidx.size(); ++k) acol[k] = N.agg[H.colidx[k]];
            rc = rc ? rc : up(p, &L.acol, acol);
        }
    }
    setup_mark("  hierarchy: uploads");
    if (!rc && st->dist) {
        const int world = (int)st->r_cnt.size();
        st->r_seg = st->r_max + 2;
        std::vector<int32_t> src((size_t)st->host[0].n * D), spos(world);
        for (int q = 0; q < world; ++q) {
            for (size_t t = 0; t < st->r_cnt[q]; ++t) src[st->r_off[q] + t] = (int32_t)(q * st->r_seg + t);
            spos[q] = (int32_t)(q * st->r_seg + st->r_cnt[q]);
        }
        rc = up(p, &st->d_unpad_src, src);
        rc = rc ? rc : up(p, &st->d_scal_pos, spos);
        rc = rc ? rc : dev_alloc(&st->d_rpad, (size_t)world * st->r_seg);
        st->m_off.resize(world); st->m_cnt.resize(world);
        for (int q = 0; q < world; ++q) { st->m_off[q] = st->r_off[q] / D * DD; st->m_cnt[q] = st->r_cnt[q] / D * DD; }
    }
    const int nc = st->host.back().n;
    st->dense = nc <= kCoarsestMaxBig;
    st->dense_coop = st->dense && nc > kCoarsestMax;
    if (!rc && st->dense) {
        rc = dev_alloc(&st->d_dense, (size_t)nc * D * nc * D);
        if (st->dense_coop) {
            rc = rc ? rc : dev_alloc(&st->d_rowbuf, (size_t)2 * (nc * D * D + D * D));
            const int smem = (int)dense_coop_smem(nc, D);
            cudaError_t ea = D == 7 ? cudaFuncSetAttribute(amg_dense_inverse_coop_kernel<7>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)
                           : D == 4 ? cudaFuncSetAttribute(amg_dense_inverse_coop_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)
                                    : cudaFuncSetAttribute(amg_dense_inverse_coop_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
            if (!rc && ea != cudaSuccess) {
                set_error("amg_setup: cannot reserve %d bytes of shared memory", smem);
                rc = S3O_ERR_CUDA;
            }
        } else {
            const int smem = (nc * D * nc * D + nc * D) * (int)sizeof(double);
            cudaError_t ea = D == 7 ? cudaFuncSetAttribute(amg_dense_inverse_kernel<7>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)
                           : D == 4 ? cudaFuncSetAttribute(amg_dense_inverse_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)
                                    : cudaFuncSetAttribute(amg_dense_inverse_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
            if (!rc && ea != cudaSuccess) {
                set_error("amg_setup: cannot reserve %d bytes of shared memory", smem);
                rc = S3O_ERR_CUDA;
            }
        }
    }
    if (!rc) {
        // K-cycle on every level above the coarsest for large graphs (measured on the 1M-pose sphere: PCG iterations of a
        // late LM iteration 334 with the V-cycle, 166 with one K level, 63 with three; K on some levels and V below them
        // can be worse than either); small graphs keep the V-cycle.  S3O_KCYCLE=<levels> overrides (0: V-cycle everywhere).
        const int n_fine_global = p->dist ? p->plan.nf_global : st->host[0].n_fine;     // host[0].n_fine is local when partitioned
        st->kdepth = (nl >= 2 && n_fine_global >= kBigGraph) ? nl - 1 : 0;
        st->kmask = (1u << st->kdepth) - 1u;
        // ... except the first coarse level when there are K levels below it: two inner steps there double the work of
        // the largest coarse level and of everything under it for ~1.35x fewer PCG iterations (1M-pose sphere, complete
        // solve: 175 iterations / 0.455 s with K everywhere, 239 / 0.424 s with V on level 1; 100k: 0.183 -> 0.155 s)
        if (st->kdepth >= 2) st->kmask &= ~1u;
        if (const char *v = getenv("S3O_KCYCLE")) {     // experiment switch: K on the first <levels> levels exactly
            st->kdepth = std::max(0, std::min(atoi(v), nl - 1));
            st->kmask = (1u << st->kdepth) - 1u;
        }
        if (const char *v = getenv("S3O_KMASK")) {      // experiment switch: any subset of levels
            st->kmask = (unsigned)strtoul(v, nullptr, 0) & ((1u << (nl - 1)) - 1u);
            st->kdepth = 0;
            for (int l = 0; l < nl - 1; ++l) if ((st->kmask >> l) & 1u) st->kdepth = l + 1;
            if (st->kdepth == 0 && n_fine_global >= kBigGraph) { st->kdepth = 1; }      // keep the K-cycle code path (all V)
        }
        int coop_rows = kCoopRows;
        if (const char *v = getenv("S3O_COOP_ROWS")) coop_rows = atoi(v);       // experiment switch
        st->coop_first = 0;
        while (st->coop_first < nl - 1 && st->lev[st->coop_first].n > coop_rows) ++st->coop_first;
        if (st->kdepth > 0 || st->dense_coop) {
            int per_sm = 0, sms = 0;
            cudaError_t eo = D == 7 ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, amg_coop_kernel<7>, kCoopThreads, 0)
                           : D == 4 ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, amg_coop_kernel<4>, kCoopThreads, 0)
                                    : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, amg_coop_kernel<1>, kCoopThreads, 0);
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, p->device);
            if (eo != cudaSuccess || per_sm < 1 || sms < 8) { st->kdepth = 0; if (st->dense_coop) { set_error("amg_setup: cooperative launch unavailable"); rc = S3O_ERR_CUDA; } }
            else {
                st->coop_grid = sms;
                rc = dev_alloc(&st->d_ks, kMaxLevels);
                rc = rc ? rc : dev_alloc(&st->d_cdots, (size_t)6 * sms);
            }
        }
    }
    if (!rc) { cudaError_t e = cudaStreamSynchronize(p->stream); if (e != cudaSuccess) { set_error("amg_setup: %s", cudaGetErrorString(e)); rc = S3O_ERR_CUDA; } }
    // the host lists are only needed for the upload; keep the small per-level sizes
    for (auto &H : st->host) {
        std::vector<int32_t>().swap(H.gal_ent); std::vector<int32_t>().swap(H.gal_i); std::vector<int32_t>().swap(H.gal_j);
        std::vector<int32_t>().swap(H.agg); std::vector<int32_t>().swap(H.mem_idx);
    }
    if (rc) amg_destroy(p);
    return rc;
}

namespace {
// Relative frames of every level at the current linearisation point.
template <int D, int KIND>
int update_frames_t(s3o_problem *p) {
    AmgState *st = p->amg;
    if (!st || st->lev.empty()) return S3O_OK;
    const double *est = p->d_est[p->cur];
    for (size_t l = 0; l < st->lev.size(); ++l) {
        LevelDev &L = st->lev[l];
        const int32_t *vid_fine = l == 0 ? st->d_vid0 : st->lev[l - 1].vid;
        amg_rel_kernel<KIND><<<(L.n_fine + 127) / 128, 128, 0, p->stream>>>(est, p->d_aux, p->nv_pad, vid_fine, L.agg, L.vid,
                                                                             L.n_fine, L.pad_fine, L.rel);
    }
    st->frames_valid = true;
    return check_launch(p, (int)st->lev.size());
}

// Galerkin operators, smoother inverses and the coarsest inverse for (H + lambda I).
template <int D, int KIND>
int update_values_t(s3o_problem *p, double lambda) {
    AmgState *st = p->amg;
    if (!st || st->lev.empty()) return S3O_OK;
    int rc;
    int launches = 0;
    // K = P^T H P has to be rebuilt for a new linearisation point, not for a new lambda at the same one (LM retry)
    const bool rebuild = !st->k_valid || st->lin_changed;
    st->lin_changed = false;
    if (rebuild) {
        ++st->rebuilds;
        if ((rc = update_frames_t<D, KIND>(p))) return rc;
        for (size_t l = 0; l < st->lev.size(); ++l) {
            LevelDev &L = st->lev[l];
            const int grid = (L.nub + 15) / 16;
            if (l == 0) {
                amg_galerkin_kernel<D, true><<<grid, 128, 0, p->stream>>>(p->d_H, L.gal_i, L.gal_j, L.rel, L.pad_fine,
                                                                        L.nub, L.gal_ptr, L.gal_ent, L.gal_out, L.gal_mirror, L.A,
                                                                        st->dist ? 0 : 1, L.gal_order);
                amg_mass_kernel<D><<<(L.n + 15) / 16, 128, 0, p->stream>>>(L.n, L.mem_ptr, L.mem_idx, L.rel, L.pad_fine, nullptr, L.M);
                if (st->dist) {     // every rank computed the upper blocks of its own coarse rows and the mass blocks of its aggregates
                    if (comm_allgatherv(p->comm, L.A, st->a_off.data(), st->a_cnt.data(), p->stream) ||
                        comm_allgatherv(p->comm, L.M, st->m_off.data(), st->m_cnt.data(), p->stream)) {
                        set_error("%s", comm_last_error());
                        return S3O_ERR_NCCL;
                    }
                    amg_mirror_kernel<D><<<(L.nub * DD + 255) / 256, 256, 0, p->stream>>>(L.nub, L.gal_out, L.gal_mirror, L.A);
                    ++launches;
                }
            } else {
                const LevelDev &F = st->lev[l - 1];      // F.A still holds K of the level above: the shifts come last
                amg_galerkin_kernel<D, false><<<grid, 128, 0, p->stream>>>(F.A, L.gal_i, L.gal_j, L.rel, L.pad_fine, L.nub,
                                                                         L.gal_ptr, L.gal_ent, L.gal_out, L.gal_mirror, L.A, 1, L.gal_order);
                amg_mass_kernel<D><<<(L.n + 15) / 16, 128, 0, p->stream>>>(L.n, L.mem_ptr, L.mem_idx, L.rel, L.pad_fine, F.M, L.M);
            }
            amg_save_diag_kernel<D><<<(L.n * DD + 255) / 256, 256, 0, p->stream>>>(L.n, L.dpos, L.A, L.Kd);
            launches += 3;
        }
        st->k_valid = true;
    } else {
        ++st->reuses;
    }
    for (size_t l = 0; l < st->lev.size(); ++l) {
        LevelDev &L = st->lev[l];
        amg_shift_diag_kernel<D><<<(L.n * DD + 255) / 256, 256, 0, p->stream>>>(L.n, L.dpos, L.Kd, L.M, lambda, L.A);
        launch_precond(D, L.A, L.dpos, L.n, 0.0, L.Dinv, p->d_sc, p->stream);
        launches += 2;
    }
    if (st->dense) {
        const LevelDev &C = st->lev.back();
        const int N = C.n * D;
        if (st->dense_coop) {
            const double *Ap = C.A;
            const int32_t *rp = C.rowptr, *ci = C.colidx;
            int n = C.n;
            double *inv = st->d_dense, *pub = st->d_rowbuf;
            DevScalars *scp = p->d_sc;
            GridBarrier gb{};
            void *args[] = { &Ap, &rp, &ci, &n, &inv, &pub, &scp, &gb };
            static const int dense_threads = getenv("S3O_DENSE_THREADS") ? std::max(64, std::min(kDenseCoopThreads, atoi(getenv("S3O_DENSE_THREADS")))) : kDenseCoopThreads;
            int rcl = launch_persistent(p, (const void *)amg_dense_inverse_coop_kernel<D>, n, dense_threads, args, 8, dense_coop_smem(n, D));
            if (rcl) return rcl;
        } else {
            amg_dense_inverse_kernel<D><<<1, 256, (size_t)(N * N + N) * sizeof(double), p->stream>>>(C.A, C.rowptr, C.colidx, C.n,
                                                                                                  st->d_dense, p->d_sc);
        }
        launches += 1;
    }
    return check_launch(p, launches);
}

// One application of the multilevel preconditioner inside the PCG, fused with what follows it:
// r_1 = P0^T r, x_1 = V(r_1), r.z = r.zJ + r_1.x_1 (PCG scalars: beta, convergence test), and the new search
// direction p = (zJ + P0 x_1) + beta p.  z holds zJ = D^-1 r on entry and is not completed -- nothing needs z
// itself.  init: first application of a solve (p = z).
template <int D>
int apply_t(s3o_problem *p, int init, double tol, int max_iter) {
    AmgState *st = p->amg;
    const int nl = (int)st->lev.size();
    const DevScalars *sc = p->d_sc;
    const int chk = init ? 0 : 1;
    cudaStream_t s = p->stream;
    int launches = 0;
    auto rows = [](int n) { return (n + 15) / 16; };
    const int lt = tail_first(st);
    {   // fine residual -> level 1
        LevelDev &L = st->lev[0];
        amg_restrict_kernel<D><<<(L.n + 15) / 16, 128, 0, s>>>(L.n, L.mem_ptr, L.mem_idx, L.rel, L.pad_fine, p->d_r, L.r, sc, chk);
        ++launches;
        trace_mark(p, "fine restrict");
        if (st->dist) {
            // my segment starts at L.r + r_off[rank], followed by my partial r.zJ and |r|^2; the padded tail of
            // the send is ignored by the unpad map
            double *mine = L.r + st->r_off[p->comm.rank];
            amg_scalars_to_vec_kernel<<<1, 1, 0, s>>>(mine + st->r_cnt[p->comm.rank], sc, chk);
            if (comm_allgather(p->comm, mine, st->d_rpad, st->r_seg, s)) {
                set_error("%s", comm_last_error());
                return S3O_ERR_NCCL;
            }
            amg_unpad_kernel<<<(L.n * D + 255) / 256, 256, 0, s>>>(L.n * D, st->d_unpad_src, st->d_rpad, L.r, p->d_sc, chk,
                                                                   p->comm.world, st->d_scal_pos);
            launches += 2;
        }
    }
    if (st->kdepth > 0) {
        // K-cycle path: levels above coop_first by ordinary launches (host-side recursion), the rest in one
        // cooperative kernel per visit; the solve of level l leaves its result in lev[l].x2
        const int nk = st->kdepth;
        int rc_inner = S3O_OK;
        auto kgrid = [](int n) { int g = (n + 15) / 16; return g > 148 * 8 ? 148 * 8 : (g < 1 ? 1 : g); };
        std::function<void(int)> solve;
        auto cycle = [&](int l, const double *rin, double *xout) {
            LevelDev &L = st->lev[l];
            LevelDev &C = st->lev[l + 1];
            amg_row_kernel<D, 0><<<rows(L.n), 128, 0, s>>>(L.n, L.rowptr, L.colidx, L.A, L.Dinv, rin, nullptr, L.x, kOmega, sc, chk);
            amg_row_kernel<D, 1><<<rows(L.n), 128, 0, s>>>(L.n, L.rowptr, L.colidx, L.A, L.Dinv, rin, L.x, L.t, kOmega, sc, chk);
            amg_restrict_kernel<D><<<(C.n + 15) / 16, 128, 0, s>>>(C.n, C.mem_ptr, C.mem_idx, C.rel, C.pad_fine, L.t, C.r, sc, chk);
            launches += 3;
            trace_mark(p, "lev: sweep+residual+restrict");
            solve(l + 1);
            amg_prolong_kernel<D><<<(L.n + 127) / 128, 128, 0, s>>>(L.n, C.agg, C.rel, C.pad_fine, C.x2, L.x, sc, chk);
            amg_row_kernel<D, 2><<<rows(L.n), 128, 0, s>>>(L.n, L.rowptr, L.colidx, L.A, L.Dinv, rin, L.x, xout, kOmega, sc, chk);
            launches += 2;
            trace_mark(p, "lev: prolong+sweep");
        };
        solve = [&](int l) {
            LevelDev &L = st->lev[l];
            if (l >= st->coop_first) {
                CoopParams P{};
                P.nlev = nl - l;
                P.dense = st->dense ? 1 : 0;
                P.N = st->lev.back().n * D;
                P.inv = st->d_dense;
                P.kdepth = nk > l ? nk - l : 0;
                P.kmask = st->kmask >> l;
                P.dots = st->d_cdots;
                static long long *d_dbg = nullptr;
                static int dbg_calls = 0;
                static const bool dbg_on = getenv("S3O_COOP_DBG") != nullptr;
                if (dbg_on && !d_dbg) { cudaMalloc(&d_dbg, 128 * sizeof(long long)); }
                const bool dbg_now = dbg_on && ++dbg_calls == 200;
                if (dbg_now) { cudaMemsetAsync(d_dbg, 0, 128 * sizeof(long long), s); P.dbg = d_dbg; }
                for (int k = l; k < nl; ++k) {
                    LevelDev &S = st->lev[k];
                    CoopLevel &T = P.lev[k - l];
                    T.n = S.n; T.pad_fine = S.pad_fine;
                    T.rowptr = S.rowptr; T.colidx = S.colidx; T.mem_ptr = S.mem_ptr; T.mem_idx = S.mem_idx; T.agg = S.agg;
                    T.A = S.A; T.Dinv = S.Dinv; T.rel = S.rel; T.r = S.r; T.x = S.x; T.x2 = S.x2; T.t = S.t;
                    T.z1 = S.z1; T.q1 = S.q1; T.rp = S.rp; T.z2 = S.z2; T.acol = S.acol;
                }
                double omega = kOmega;
                int chk_ = chk;
                GridBarrier gb{};
                void *args[] = { &P, &omega, (void *)&sc, &chk_, &gb };
                const int grid = coop_grid_at(st, l);
                for (int k = 0; k < P.nlev; ++k) P.lev[k].G = coop_row_groups(grid, P.lev[k].n);
                if (launch_persistent(p, (const void *)amg_coop_kernel<D>, grid, kCoopThreads, args, 5)) rc_inner = S3O_ERR_CUDA;
                ++launches;
                trace_mark(p, "cooperative kernel");
                if (dbg_now) {
                    long long h[128];
                    cudaStreamSynchronize(s);
                    cudaMemcpy(h, d_dbg, sizeof h, cudaMemcpyDeviceToHost);
                    int khz = 1; cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, p->device);
                    fprintf(stderr, "S3O_COOP_DBG: phase times of one cooperative-kernel call (us, SM clock %d kHz)\n ", khz);
                    for (int q = 1; q < 120 && h[q]; ++q) fprintf(stderr, " %d:%.1f", q, (double)(h[q] - h[q - 1]) / khz * 1e3);
                    fprintf(stderr, "\n");
                }
                return;
            }
            if ((st->kmask >> l) & 1u) {
                KScal *ks = st->d_ks + l;
                const int n = L.n * D;
                cycle(l, L.r, L.z1);
                amg_kdots_kernel<D, 128><<<kgrid(L.n), 128, 0, s>>>(L.n, L.rowptr, L.colidx, L.A, L.z1, L.r, nullptr, L.q1, p->d_partials, ks, 0, p->d_sc, chk);
                amg_kaxpy_kernel<<<std::min((n + 255) / 256, 148 * 8), 256, 0, s>>>(n, L.r, L.q1, L.rp, ks, 0, sc, chk);
                trace_mark(p, "lev: kdots+axpy");
                cycle(l, L.rp, L.z2);
                amg_kdots_kernel<D, 128><<<kgrid(L.n), 128, 0, s>>>(L.n, L.rowptr, L.colidx, L.A, L.z2, L.rp, L.q1, nullptr, p->d_partials, ks, 1, p->d_sc, chk);
                amg_kaxpy_kernel<<<std::min((n + 255) / 256, 148 * 8), 256, 0, s>>>(n, L.z1, L.z2, L.x2, ks, 1, sc, chk);
                launches += 4;
                trace_mark(p, "lev: kdots+combine");
            } else {
                cycle(l, L.r, L.x2);
            }
        };
        solve(0);
        if (rc_inner) { set_error("multilevel K-cycle: persistent-kernel launch failed: %s", s3o_last_error()); return rc_inner; }
        std::swap(st->lev[0].x, st->lev[0].x2);
    } else {
        for (int l = 0; l < lt; ++l) {
            LevelDev &L = st->lev[l];
            LevelDev &C = st->lev[l + 1];
            amg_row_kernel<D, 0><<<rows(L.n), 128, 0, s>>>(L.n, L.rowptr, L.colidx, L.A, L.Dinv, L.r, nullptr, L.x, kOmega, sc, chk);
            amg_row_kernel<D, 1><<<rows(L.n), 128, 0, s>>>(L.n, L.rowptr, L.colidx, L.A, L.Dinv, L.r, L.x, L.t, kOmega, sc, chk);
            amg_restrict_kernel<D><<<(C.n + 15) / 16, 128, 0, s>>>(C.n, C.mem_ptr, C.mem_idx, C.rel, C.pad_fine, L.t, C.r, sc, chk);
            launches += 3;
        }
        {
            TailParams P{};
            P.nlev = nl - lt;
            P.dense = st->dense ? 1 : 0;
            P.N = st->lev.back().n * D;
            P.inv = st->d_dense;
            for (int l = lt; l < nl; ++l) {
                LevelDev &L = st->lev[l];
                TailLevel &T = P.lev[l - lt];
                T.n = L.n; T.pad_fine = L.pad_fine;
                T.rowptr = L.rowptr; T.colidx = L.colidx; T.mem_ptr = L.mem_ptr; T.mem_idx = L.mem_idx; T.agg = L.agg;
                T.A = L.A; T.Dinv = L.Dinv; T.rel = L.rel; T.r = L.r; T.x = L.x; T.x2 = L.x2; T.t = L.t;
            }
            amg_tail_kernel<D><<<kTailCtas, kTailThreads, 0, s>>>(P, kOmega, sc, chk);
            for (int l = lt; l < nl; ++l) std::swap(st->lev[l].x, st->lev[l].x2);
            ++launches;
        }
        for (int l = lt - 1; l >= 0; --l) {
            LevelDev &L = st->lev[l];
            LevelDev &C = st->lev[l + 1];
            amg_prolong_kernel<D><<<(L.n + 127) / 128, 128, 0, s>>>(L.n, C.agg, C.rel, C.pad_fine, C.x, L.x, sc, chk);
            amg_row_kernel<D, 2><<<rows(L.n), 128, 0, s>>>(L.n, L.rowptr, L.colidx, L.A, L.Dinv, L.r, L.x, L.x2, kOmega, sc, chk);
            std::swap(L.x, L.x2);
            launches += 2;
        }
    }
    {
        LevelDev &L = st->lev[0];
        constexpr int NT = 256;
        const int rows = st->dist ? st->n_own : L.n_fine;
        int grid = (rows + NT - 1) / NT;
        if (grid > 148 * 8) grid = 148 * 8;
        if (grid < 1) grid = 1;
        int dgrid = (L.n * D + NT - 1) / NT;
        if (dgrid > 148) dgrid = 148;
        if (dgrid < 1) dgrid = 1;
        amg_coarse_dot_kernel<NT><<<dgrid, NT, 0, s>>>(L.n * D, L.r, L.x, p->d_partials, p->d_sc, init, tol, max_iter);
        amg_prolong0_kernel<D, NT><<<grid, NT, 0, s>>>(rows, L.agg, L.rel, L.pad_fine, L.x, p->d_z, p->d_p, sc, init);
        launches += 2;
        trace_mark(p, "coarse dot + fine prolong");
    }
    return check_launch(p, launches);
}

}  // namespace

#define S3O_AMG_DISPATCH(CALL7, CALL4, CALL1)                  \
    switch (p->kind) {                                         \
    case S3O_KIND_SIM3: return CALL7;                          \
    case S3O_KIND_SCALE_TRANS: return CALL4;                   \
    case S3O_KIND_SCALE: return CALL1;                         \
    default: set_error("multilevel preconditioner: pose-graph problems only"); return S3O_ERR_UNSUPPORTED; \
    }
int amg_update_frames(s3o_problem *p) {
    S3O_AMG_DISPATCH((update_frames_t<7, S3O_KIND_SIM3>(p)), (update_frames_t<4, S3O_KIND_SCALE_TRANS>(p)),
                     (update_frames_t<1, S3O_KIND_SCALE>(p)))
}
int amg_update_values(s3o_problem *p, double lambda) {
    S3O_AMG_DISPATCH((update_values_t<7, S3O_KIND_SIM3>(p, lambda)), (update_values_t<4, S3O_KIND_SCALE_TRANS>(p, lambda)),
                     (update_values_t<1, S3O_KIND_SCALE>(p, lambda)))
}
int amg_apply(s3o_problem *p, int init, double tol, int max_iter) {
    S3O_AMG_DISPATCH(apply_t<7>(p, init, tol, max_iter), apply_t<4>(p, init, tol, max_iter), apply_t<1>(p, init, tol, max_iter))
}
#undef S3O_AMG_DISPATCH

void amg_counts(const s3o_problem *p, int64_t *rebuilds, int64_t *reuses) {
    if (!rebuilds || !reuses) { if (p->amg) p->amg->rebuilds = p->amg->reuses = 0; return; }
    *rebuilds = p->amg ? p->amg->rebuilds : 0;
    *reuses = p->amg ? p->amg->reuses : 0;
}
void amg_set_counts(s3o_problem *p, int64_t rebuilds, int64_t reuses) {
    if (p->amg) { p->amg->rebuilds = rebuilds; p->amg->reuses = reuses; }
}
void amg_invalidate_frames(s3o_problem *p) { if (p->amg) { p->amg->frames_valid = false; p->amg->lin_changed = true; } }

// ---- read-outs of the hierarchy for tests (s3o_multilevel_prepare, s3o_get_multilevel_*) ---------------------
int amg_plan_info(const s3o_problem *p, bool active, int32_t *info, int cap) {
    const AmgState *st = active ? p->amg : nullptr;
    const int nl = st ? (int)st->lev.size() : 0;
    if (cap < kPlanHeader + 3 * nl) { set_error("s3o_multilevel_prepare: info needs %d entries", kPlanHeader + 3 * nl); return S3O_ERR_INVALID; }
    for (int k = 0; k < cap; ++k) info[k] = 0;
    if (nl == 0) return S3O_OK;
    const int grid = st->kdepth > 0 ? coop_grid_at(st, st->coop_first) : 0;
    info[0] = nl; info[1] = st->kdepth; info[2] = (int32_t)st->kmask; info[3] = st->coop_first; info[4] = tail_first(st);
    info[5] = st->dense; info[6] = st->dense_coop; info[7] = st->coop_grid; info[8] = grid;
    for (int l = 0; l < nl; ++l) {
        info[kPlanHeader + 3 * l] = st->lev[l].n;
        info[kPlanHeader + 3 * l + 1] = st->lev[l].nblk;
        info[kPlanHeader + 3 * l + 2] = (grid && l >= st->coop_first) ? coop_row_groups(grid, st->lev[l].n) : 0;
    }
    return S3O_OK;
}

namespace {
template <class T>
int download(s3o_problem *p, T *dst, const T *src, size_t count) {
    if (dst && count) S3O_CUDA(cudaMemcpyAsync(dst, src, count * sizeof(T), cudaMemcpyDeviceToHost, p->stream));
    return S3O_OK;
}
}  // namespace

int amg_read_level(s3o_problem *p, int level, int32_t *agg, int32_t *root_vid, int32_t *rowptr, int32_t *colidx,
                   double *A, double *Dinv, double *rel) {
    const AmgState *st = p->amg;
    if (!st || level < 0 || level >= (int)st->lev.size()) {
        set_error("s3o_get_multilevel_level: no level %d (%d levels prepared)", level, st ? (int)st->lev.size() : 0);
        return S3O_ERR_INVALID;
    }
    const LevelDev &L = st->lev[level];
    const int D = p->d, S = D * (D + 1) / 2;
    std::vector<double> dpk(Dinv ? (size_t)L.n * S : 0), rpl(rel ? (size_t)NREL * L.pad_fine : 0);
    int rc = download(p, agg, L.agg, (size_t)L.n_fine);
    rc = rc ? rc : download(p, root_vid, L.vid, (size_t)L.n);
    rc = rc ? rc : download(p, rowptr, L.rowptr, (size_t)L.n + 1);
    rc = rc ? rc : download(p, colidx, L.colidx, (size_t)L.nblk);
    rc = rc ? rc : download(p, A, L.A, (size_t)L.nblk * DD);
    rc = rc ? rc : download(p, dpk.data(), L.Dinv, dpk.size());
    rc = rc ? rc : download(p, rpl.data(), L.rel, rpl.size());
    if (rc) return rc;
    S3O_CUDA(cudaStreamSynchronize(p->stream));
    if (Dinv) {         // packed upper triangle (sym_off) -> d x d
        for (int I = 0; I < L.n; ++I)
            for (int r = 0; r < D; ++r)
                for (int c = 0; c < D; ++c) {
                    const int lo = std::min(r, c), hi = std::max(r, c);
                    Dinv[((size_t)I * D + r) * D + c] = dpk[(size_t)I * S + lo * D - lo * (lo - 1) / 2 + (hi - lo)];
                }
    }
    if (rel)            // [13][pad_fine] planes -> [n_fine][13]
        for (int i = 0; i < L.n_fine; ++i)
            for (int k = 0; k < NREL; ++k) rel[(size_t)i * NREL + k] = rpl[(size_t)k * L.pad_fine + i];
    return S3O_OK;
}

int amg_read_coarsest_inverse(s3o_problem *p, double *inv) {
    const AmgState *st = p->amg;
    if (!st || st->lev.empty() || !st->dense) {
        set_error("s3o_get_multilevel_coarsest_inverse: no dense inverse of the coarsest level (%s)",
                  !st || st->lev.empty() ? "no levels prepared" : "more than 128 vertices: smoothed instead");
        return S3O_ERR_INVALID;
    }
    const size_t N = (size_t)st->lev.back().n * p->d;
    int rc = download(p, inv, (const double *)st->d_dense, N * N);
    if (rc) return rc;
    S3O_CUDA(cudaStreamSynchronize(p->stream));
    return S3O_OK;
}

}  // namespace s3o
