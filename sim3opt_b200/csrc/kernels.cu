// kernels.cu -- hand-written sm_100a kernels of the LM hot path (all arithmetic fp64).
//
//   chi2 / edge error          EdgeSim3::computeError + activeRobustChi2         (rows a10, a13)
//   linearize                  BaseBinaryEdge::linearizeOplus (numeric h or analytic)
//                              + constructQuadraticForm per edge                  (rows a11, a12)
//   assemble                   deterministic gather of the per-edge products into the BSR-upper
//                              Hessian and b (fixed summation order, no floating-point atomics)
//   precond / spmv / pcg_*     block-Jacobi PCG replacing LinearSolverEigen::solve (row a16)
//   retract                    VertexSim3Expmap::oplusImpl  S <- exp(delta) S      (row a9)
//   maxdiag / scale            computeLambdaInit / computeScale                    (row a15)
//
// Every global reduction writes one partial per CTA and lets the last CTA to arrive (integer
// ticket) add the partials in index order, so results are bitwise reproducible run to run.
#include <assert.h>
#include <stdlib.h>

#include "../../include/sim3opt_b200.h"
#include "kernels.cuh"
#include "sim3_math.cuh"
#include "reduce.cuh"

namespace s3o {

// ======================================================================================
// packing
// ======================================================================================
__global__ void pack_vertices_kernel(const double *__restrict__ aos, int n, int n_pad, int dim,
                                     double *__restrict__ soa) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * dim) return;
    const int v = t / dim, k = t % dim;
    soa[(size_t)k * n_pad + v] = aos[t];
}
__global__ void unpack_vertices_kernel(const double *__restrict__ soa, int n, int n_pad, int dim,
                                       double *__restrict__ aos) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * dim) return;
    const int v = t / dim, k = t % dim;
    aos[t] = soa[(size_t)k * n_pad + v];
}
void launch_pack_vertices(const double *aos, int n, int n_pad, int dim, double *soa, cudaStream_t st) {
    if (n == 0) return;
    pack_vertices_kernel<<<(n * dim + 255) / 256, 256, 0, st>>>(aos, n, n_pad, dim, soa);
}
void launch_unpack_vertices(const double *soa, int n, int n_pad, int dim, double *aos, cudaStream_t st) {
    if (n == 0) return;
    unpack_vertices_kernel<<<(n * dim + 255) / 256, 256, 0, st>>>(soa, n, n_pad, dim, aos);
}

// gathers the caller-ordered AoS edge records into vertex-pair-sorted SoA planes; the
// information matrix is packed to its upper triangle (row-major, r<=c).
__global__ void pack_edges_kernel(const double *__restrict__ meas_aos, const double *__restrict__ info_aos,
                                  const int32_t *__restrict__ perm, int ne, int ne_pad, int est_dim, int d, int info_diag,
                                  double *__restrict__ meas, double *__restrict__ info, const int32_t *__restrict__ dst) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ne) return;
    const size_t o = (size_t)perm[i], t = dst ? (size_t)dst[i] : (size_t)i;
    for (int k = 0; k < est_dim; ++k) meas[(size_t)k * ne_pad + t] = meas_aos[o * est_dim + k];
    if (info_aos && info_diag) {         // d diagonal entries per edge in, d planes out
        for (int r = 0; r < d; ++r) info[(size_t)r * ne_pad + t] = info_aos[o * d + r];
    } else if (info_aos) {
        int f = 0;
        for (int r = 0; r < d; ++r)
            for (int c = r; c < d; ++c) info[(size_t)(f++) * ne_pad + t] = info_aos[o * d * d + r * d + c];
    }
}
void launch_pack_edges(const double *meas_aos, const double *info_aos, const int32_t *perm, int ne, int ne_pad,
                       int est_dim, int d, int info_diag, double *meas, double *info, cudaStream_t st, const int32_t *dst) {
    if (ne == 0) return;
    pack_edges_kernel<<<(ne + 127) / 128, 128, 0, st>>>(meas_aos, info_aos, perm, ne, ne_pad, est_dim, d, info_diag, meas, info, dst);
}

__global__ void convert_info_kernel(const double *__restrict__ src, int n, int d, int rep_src, int rep_dst,
                                    double *__restrict__ dst) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    for (int r = 0; r < d; ++r) {
        const double diag = rep_src == 1 ? src[(size_t)k * d + r] : 1.0;
        if (rep_dst == 1) { dst[(size_t)k * d + r] = diag; continue; }
        for (int c = 0; c < d; ++c) dst[((size_t)k * d + r) * d + c] = r == c ? diag : 0.0;
    }
}
void launch_convert_info(const double *src, int n, int d, int rep_src, int rep_dst, double *dst, cudaStream_t st) {
    if (n == 0) return;
    convert_info_kernel<<<(n + 127) / 128, 128, 0, st>>>(src, n, d, rep_src, rep_dst, dst);
}

// ======================================================================================
// edge models
// ======================================================================================
template <int KIND> struct Model;
template <> struct Model<S3O_KIND_SIM3> { static constexpr int D = 7, EST = 8; static constexpr bool AUX = false; };
template <> struct Model<S3O_KIND_SCALE_TRANS> { static constexpr int D = 4, EST = 4; static constexpr bool AUX = true; };
template <> struct Model<S3O_KIND_SCALE> { static constexpr int D = 1, EST = 1; static constexpr bool AUX = false; };

template <int N>
__device__ __forceinline__ void load_planes(const double *__restrict__ planes, int pad, int idx, double out[N]) {
#pragma unroll
    for (int k = 0; k < N; ++k) out[k] = __ldg(planes + (size_t)k * pad + idx);
}

__device__ __forceinline__ Sim3 to_sim3(const double x[8]) {
    Sim3 S;
    S.qx = x[0]; S.qy = x[1]; S.qz = x[2]; S.qw = x[3];
    S.tx = x[4]; S.ty = x[5]; S.tz = x[6]; S.s = x[7];
    return S;
}
__device__ __forceinline__ void from_sim3(const Sim3 &S, double x[8]) {
    x[0] = S.qx; x[1] = S.qy; x[2] = S.qz; x[3] = S.qw;
    x[4] = S.tx; x[5] = S.ty; x[6] = S.tz; x[7] = S.s;
}

// e = error(measurement m, vertex(0)=xi, vertex(1)=xj); qi/qj: fixed rotations (scale-trans only)
// flags: bit 0 = S3O_MATH_CORRECTED (Sim3 coefficients), bit 1 = S3O_SCALE_MODEL_LOGRATIO (scale / scale-trans kinds)
template <int KIND>
__device__ S3O_ERR_INLINE void model_error(const double *m, const double *xi, const double *xj, const double *qi,
                                         const double *qj, double *e, int flags) {
    if constexpr (KIND == S3O_KIND_SIM3) {
        sim3_edge_error(to_sim3(m), to_sim3(xi), to_sim3(xj), e, (flags & 1) != 0);
    } else if constexpr (KIND == S3O_KIND_SCALE_TRANS) {
        // [EXT vio_g2o] G2oEdgeScaleTrans model restated from kitti_surf.cpp:897-906 (scale rows
        // s_ji*s_i - s_j) and :969-985 (translation rows t_j - (s_j/s_i) R_j R_i^T t_i - t_ji)
        double ax, ay, az, bx, by, bz;
        quat_rotate(-qi[0], -qi[1], -qi[2], qi[3], xi[1], xi[2], xi[3], ax, ay, az);
        quat_rotate(qj[0], qj[1], qj[2], qj[3], ax, ay, az, bx, by, bz);
        const double sr = xj[0] / xi[0];
        e[0] = (flags & 2) ? log(m[0] * xi[0] / xj[0]) : m[0] * xi[0] - xj[0];
        e[1] = xj[1] - sr * bx - m[1];
        e[2] = xj[2] - sr * by - m[2];
        e[3] = xj[3] - sr * bz - m[3];
    } else {
        e[0] = (flags & 2) ? log(m[0] * xi[0] / xj[0]) : m[0] * xi[0] - xj[0];
    }
}

template <int KIND>
__device__ __forceinline__ void model_oplus(double *x, const double *delta, int flags) {
    if constexpr (KIND == S3O_KIND_SIM3) {
        const Sim3 U = sim3_exp(delta, (flags & 1) != 0);
        from_sim3(sim3_mul(U, to_sim3(x)), x);
    } else {
#pragma unroll
        for (int c = 0; c < Model<KIND>::D; ++c) x[c] += delta[c];
        if (flags & 2) x[0] = (x[0] - delta[0]) * exp(delta[0]);       // multiplicative scale update s <- s exp(d_sigma)
    }
}

template <int KIND>
__device__ __forceinline__ void model_jac_analytic(const double *m, const double *xi, const double *xj,
                                                   const double *qi, const double *qj, const double *e, double *A,
                                                   double *B, int flags) {
    if constexpr (KIND == S3O_KIND_SIM3) {
        sim3_edge_jacobians(to_sim3(m), e, A, B);
    } else if constexpr (KIND == S3O_KIND_SCALE_TRANS) {
        double Ri[9], Rj[9], Q[9];
        quat_to_rot(qi[0], qi[1], qi[2], qi[3], Ri);
        quat_to_rot(qj[0], qj[1], qj[2], qj[3], Rj);
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int c = 0; c < 3; ++c)
                Q[r * 3 + c] = Rj[r * 3] * Ri[c * 3] + Rj[r * 3 + 1] * Ri[c * 3 + 1] + Rj[r * 3 + 2] * Ri[c * 3 + 2];
        const double si = xi[0], sj = xj[0];
        double b[3];
#pragma unroll
        for (int r = 0; r < 3; ++r) b[r] = Q[r * 3] * xi[1] + Q[r * 3 + 1] * xi[2] + Q[r * 3 + 2] * xi[3];
#pragma unroll
        for (int k = 0; k < 16; ++k) { A[k] = 0; B[k] = 0; }
        const bool lr = (flags & 2) != 0;      // log-ratio error, multiplicative scale update: d s = s d sigma
        A[0] = lr ? 1.0 : m[0];
        B[0] = -1;
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            A[(1 + r) * 4] = lr ? sj / si * b[r] : sj / (si * si) * b[r];
            B[(1 + r) * 4] = lr ? -(sj / si) * b[r] : -b[r] / si;
#pragma unroll
            for (int c = 0; c < 3; ++c) A[(1 + r) * 4 + 1 + c] = -(sj / si) * Q[r * 3 + c];
            B[(1 + r) * 4 + 1 + r] = 1;
        }
    } else {
        A[0] = (flags & 2) ? 1.0 : m[0];
        B[0] = -1;
    }
}

// rho[0..1] of the robust kernels (g2o RobustKernelHuber / PTAM MEstimator.h:54-198)
__device__ __forceinline__ void robustify(int kind, double param, double e2, double &rho0, double &rho1) {
    switch (kind) {
    case S3O_ROBUST_HUBER: {
        const double dsqr = param * param;
        if (e2 <= dsqr) { rho0 = e2; rho1 = 1; }
        else { const double sq = sqrt(e2); rho0 = 2 * sq * param - dsqr; rho1 = param / sq; }
        break;
    }
    case S3O_ROBUST_PTAM_TUKEY:
        if (e2 > param) { rho0 = 1.0; rho1 = 0.0; }
        else { const double dd = 1.0 - e2 / param; rho0 = 1.0 - dd * dd * dd; rho1 = dd * dd; }
        break;
    case S3O_ROBUST_PTAM_CAUCHY:
        rho0 = log(1.0 + e2 / param);
        rho1 = 1.0 / (1.0 + e2 / param);
        break;
    case S3O_ROBUST_PTAM_HUBER:
        if (e2 < param) { rho0 = 0.5 * e2; rho1 = 1; }
        else { const double ds = sqrt(param), de = sqrt(e2); rho0 = ds * (de - 0.5 * ds); rho1 = sqrt(param / e2); }
        break;
    default:
        rho0 = e2; rho1 = 1;
        break;
    }
}

template <int D>
__device__ __forceinline__ double quad_form_packed(const double *__restrict__ info, bool info_diag, int pad, int t, const double *e) {
    if (!info) {
        double s = 0;
#pragma unroll
        for (int i = 0; i < D; ++i) s += e[i] * e[i];
        return s;
    }
    if (info_diag) {        // D planes: the diagonal only
        double s = 0;
#pragma unroll
        for (int i = 0; i < D; ++i) s += __ldg(info + (size_t)i * pad + t) * e[i] * e[i];
        return s;
    }
    double s = 0;
    int f = 0;
#pragma unroll
    for (int r = 0; r < D; ++r)
#pragma unroll
        for (int c = r; c < D; ++c) {
            const double o = __ldg(info + (size_t)(f++) * pad + t);
            s += (r == c ? 1.0 : 2.0) * o * e[r] * e[c];
        }
    return s;
}

// ======================================================================================
// chi2 / edge errors
// ======================================================================================
template <int KIND, int NT>
__global__ void __launch_bounds__(NT) chi2_kernel(GraphDev g, double *__restrict__ partials, DevScalars *sc) {
    constexpr int D = Model<KIND>::D, EST = Model<KIND>::EST;
    __shared__ double sh[32];
    double local = 0;
    for (int t = blockIdx.x * NT + threadIdx.x; t < g.ne; t += gridDim.x * NT) {
        if (g.primary && !g.primary[t]) continue;   // partitioned solve: cut edges are counted by one rank
        const int vi = g.sv0[t], vj = g.sv1[t];
        double xi[EST], xj[EST], m[EST], qi[4], qj[4], e[D];
        load_planes<EST>(g.est, g.nv_pad, vi, xi);
        load_planes<EST>(g.est, g.nv_pad, vj, xj);
        load_planes<EST>(g.meas, g.ne_pad, t, m);
        if constexpr (Model<KIND>::AUX) {
            load_planes<4>(g.aux, g.nv_pad, vi, qi);
            load_planes<4>(g.aux, g.nv_pad, vj, qj);
        }
        model_error<KIND>(m, xi, xj, qi, qj, e, g.model_flags);
        double c = quad_form_packed<D>(g.info, g.info_diag, g.ne_pad, t, e);
        if (g.robust_kind != S3O_ROBUST_NONE) {
            double r0, r1;
            robustify(g.robust_kind, g.robust_param, c, r0, r1);
            c = r0;
        }
        local += c;
    }
    const double bs = block_sum<NT>(local, sh);
    if (threadIdx.x == 0) partials[blockIdx.x] = bs;
    if (last_block(&sc->counters[0])) {
        const double tot = sum_partials<NT>(partials, gridDim.x, sh);
        if (threadIdx.x == 0) sc->chi2 = tot;
    }
}

template <int KIND>
__global__ void edge_errors_kernel(GraphDev g, double *__restrict__ err, double *__restrict__ chi) {
    constexpr int D = Model<KIND>::D, EST = Model<KIND>::EST;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= g.ne) return;
    const int vi = g.sv0[t], vj = g.sv1[t];
    double xi[EST], xj[EST], m[EST], qi[4], qj[4], e[D];
    load_planes<EST>(g.est, g.nv_pad, vi, xi);
    load_planes<EST>(g.est, g.nv_pad, vj, xj);
    load_planes<EST>(g.meas, g.ne_pad, t, m);
    if constexpr (Model<KIND>::AUX) {
        load_planes<4>(g.aux, g.nv_pad, vi, qi);
        load_planes<4>(g.aux, g.nv_pad, vj, qj);
    }
    model_error<KIND>(m, xi, xj, qi, qj, e, g.model_flags);
    for (int k = 0; k < D; ++k) err[(size_t)t * D + k] = e[k];
    if (chi) chi[t] = quad_form_packed<D>(g.info, g.info_diag, g.ne_pad, t, e);
}

static int reduce_grid(int n, int nt) {
    int g = (n + nt - 1) / nt;
    if (g > 148 * 8) g = 148 * 8;
    if (g < 1) g = 1;
    return g;
}

void launch_chi2(const GraphDev &g, double *partials, DevScalars *sc, cudaStream_t st) {
    constexpr int NT = 128;
    const int grid = reduce_grid(g.ne, NT);
    switch (g.kind) {
    case S3O_KIND_SIM3: chi2_kernel<S3O_KIND_SIM3, NT><<<grid, NT, 0, st>>>(g, partials, sc); break;
    case S3O_KIND_SCALE_TRANS: chi2_kernel<S3O_KIND_SCALE_TRANS, NT><<<grid, NT, 0, st>>>(g, partials, sc); break;
    case S3O_KIND_SCALE: chi2_kernel<S3O_KIND_SCALE, NT><<<grid, NT, 0, st>>>(g, partials, sc); break;
    }
}

void launch_edge_errors(const GraphDev &g, double *err, double *chi, cudaStream_t st) {
    if (g.ne == 0) return;
    const int grid = (g.ne + 127) / 128;
    switch (g.kind) {
    case S3O_KIND_SIM3: edge_errors_kernel<S3O_KIND_SIM3><<<grid, 128, 0, st>>>(g, err, chi); break;
    case S3O_KIND_SCALE_TRANS: edge_errors_kernel<S3O_KIND_SCALE_TRANS><<<grid, 128, 0, st>>>(g, err, chi); break;
    case S3O_KIND_SCALE: edge_errors_kernel<S3O_KIND_SCALE><<<grid, 128, 0, st>>>(g, err, chi); break;
    }
}

// ======================================================================================
// linearize: per-edge Jacobians and quadratic-form products
// ======================================================================================
// Scratch (doubles): side records [ne_pad][Hii packed NS | bi D | Hjj packed NS | bj D], one contiguous stream in edge order
// (entry e of an incidence list, 2*edge + side, is piece e), followed by the cross terms [ne_pad][Hij D*D] -- only the
// edges of multi-edge blocks write theirs, every other cross term goes straight into the Hessian.
// Hii = A^T O' A, bi = -A^T O' e, Hjj = B^T O' B, bj = -B^T O' e, Hij = A^T O' B, O' = rho1 * Omega.
__host__ __device__ constexpr int packed_size(int d) { return d * (d + 1) / 2; }
__host__ __device__ constexpr int scr_stride(int d) { return 2 * (packed_size(d) + d) + d * d; }
int scratch_stride(int d) { return scr_stride(d); }

// The warp's staging buffer holds S values per edge (edge-major); they leave as one coalesced stream into the
// per-edge records (stride doubles apart).  Full warps with S >= 32: round i moves the values 32 i .. 32 i + 31, which
// belong to at most two edges -- the split point is a compile-time constant, so there is no division in the loop.
// The warp's staging buffer holds S values per edge (edge-major); they leave as one coalesced stream into the
// per-edge records (stride doubles apart).  The (edge, entry) pair of a lane advances by 32 entries per round: no
// division in the loop.  The loops stay rolled on purpose: this kernel is bound by instruction fetch as soon as
// its straight-line code grows (unrolling them cost 10 % although it saved 11 % of the instructions).
template <int S>
__device__ __forceinline__ void warp_copy_piece(const double *stage, double *__restrict__ dst0, int stride, int lane, int nvalid) {
    static_assert(S >= 32, "one wrap per round");
    __syncwarp();
    int el = 0, f = lane;
    if (f >= S) { f -= S; el = 1; }
    const int n = nvalid * S;
#pragma unroll 1
    for (int idx = lane; idx < n; idx += 32) {
        dst0[el * stride + f] = stage[idx];
        f += 32;
        if (f >= S) { f -= S; ++el; }
    }
    __syncwarp();
}
template <int S>
__device__ __forceinline__ void warp_copy_piece_small(const double *stage, double *__restrict__ dst0, int stride, int lane, int nvalid) {
    __syncwarp();
    for (int idx = lane; idx < nvalid * S; idx += 32) {
        const int el = idx / S, f = idx - el * S;
        dst0[(size_t)el * stride + f] = stage[idx];
    }
    __syncwarp();
}

// same, but every element of the warp has its own destination (dptr[el], staged in shared memory)
template <int S>
__device__ __forceinline__ void warp_copy_piece_to(const double *stage, double **dptr, double *mine, int lane, int nvalid) {
    dptr[lane] = mine;
    __syncwarp();
    if constexpr (S >= 32) {
        int el = 0, f = lane;
        if (f >= S) { f -= S; el = 1; }
        const int n = nvalid * S;
#pragma unroll 1
        for (int idx = lane; idx < n; idx += 32) {
            dptr[el][f] = stage[idx];
            f += 32;
            if (f >= S) { f -= S; ++el; }
        }
    } else {
        for (int idx = lane; idx < nvalid * S; idx += 32) {
            const int el = idx / S, f = idx - el * S;
            dptr[el][f] = stage[idx];
        }
    }
    __syncwarp();
}

// Zero pattern of the analytic Sim3 Jacobians (sim3_edge_jacobians): [[J11,0,0],[J21,J22,j23],[0,0,+-1]] on the
// tangent [omega, upsilon, sigma].  The products below are fully unrolled, so the test folds at compile time
// and the multiplications with structural zeros disappear (31 of 49 entries are non-zero).
template <bool SP>
__device__ __forceinline__ constexpr bool jnz(int k, int c) { return !SP || (k < 3 ? c < 3 : (k < 6 || c == 6)); }

// The cross term of an edge that is the only one feeding its off-diagonal block goes straight into
// the Hessian (Hdirect != null): assemble_kernel then has nothing to do for that block.
// DIAG: the information matrices are diagonal (or absent = identity): Omega' is held as D weights, A^T O' and
// B^T O' are column scalings -- same numbers as the dense path (its extra terms are exact zeros), 2 of the 5
// 7x7x7 products and a 49-double array less.
// 6 CTAs of 64 threads per SM: 168 registers, no spills worth the name (244 at one CTA; 128 spills 0.5 KB).  The
// dense-information and numeric-Jacobian instantiations keep all registers (they would spill 0.7-1.3 KB).
#ifndef S3O_LIN_MINB
#define S3O_LIN_MINB 6
#endif
template <int KIND, int JAC, int NT, bool DIAG>
__global__ void __launch_bounds__(NT, (DIAG && JAC == S3O_JAC_ANALYTIC) ? S3O_LIN_MINB : 1) linearize_kernel(GraphDev g, double h, double *__restrict__ scratch,
                                                       const int32_t *__restrict__ e_blk,
                                                       const int32_t *__restrict__ blk_src, double *__restrict__ Hdirect) {
    constexpr int D = Model<KIND>::D, EST = Model<KIND>::EST, DD = D * D;
    constexpr int NS = packed_size(D), STRIDE = 2 * (NS + D);       // the two side pieces of an edge are one record
    constexpr int SMAX = DD > NS + D ? DD : NS + D;
    constexpr bool SP = KIND == S3O_KIND_SIM3 && JAC == S3O_JAC_ANALYTIC;      // structured Jacobians
    __shared__ double stage_all[(NT / 32) * 32 * SMAX];
    __shared__ double *dptr_all[NT];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double *stage = stage_all + warp * 32 * SMAX;
    double **dptr = dptr_all + warp * 32;
    const int e0 = (blockIdx.x * NT + warp * 32);
    if (e0 >= g.ne) return;
    const int t = e0 + lane;
    const bool valid = t < g.ne;
    const int nvalid = min(32, g.ne - e0);

    double A[DD], B[DD], O[DIAG ? D : DD], e[D];
    bool fi = false, fj = false;
    int kb = -1, src = -1;      // off-diagonal block of this edge; its only source edge (or -1: summed by assemble_kernel)
    if (valid) {
        // everything that does not depend on the vertex indices goes out with them: one round trip to DRAM
        // covers the edge record, a second one the vertex states
        const int vi = g.sv0[t], vj = g.sv1[t];
        if (Hdirect) kb = __ldg(e_blk + t);
        double xi[EST], xj[EST], m[EST], qi[4], qj[4];
        load_planes<EST>(g.meas, g.ne_pad, t, m);
        if constexpr (DIAG) {
#pragma unroll
            for (int r = 0; r < D; ++r)
                O[r] = g.info ? __ldg(g.info + (size_t)r * g.ne_pad + t) : 1.0;       // diagonal information: D planes
        }
        fi = g.hidx[vi] >= 0;
        fj = g.hidx[vj] >= 0;
        load_planes<EST>(g.est, g.nv_pad, vi, xi);
        load_planes<EST>(g.est, g.nv_pad, vj, xj);
        if (kb >= 0) src = __ldg(blk_src + kb);
        if constexpr (Model<KIND>::AUX) {
            load_planes<4>(g.aux, g.nv_pad, vi, qi);
            load_planes<4>(g.aux, g.nv_pad, vj, qj);
        }
        model_error<KIND>(m, xi, xj, qi, qj, e, g.model_flags);
        if constexpr (JAC == S3O_JAC_ANALYTIC) {
            model_jac_analytic<KIND>(m, xi, xj, qi, qj, e, A, B, g.model_flags);
        } else {
            // g2o BaseBinaryEdge::linearizeOplus: central differences through oplus, +h then -h
            const double scalar = 1.0 / (2 * h);
            for (int side = 0; side < 2; ++side) {
                double *J = side == 0 ? A : B;
                if ((side == 0 && !fi) || (side == 1 && !fj)) {
                    for (int k = 0; k < DD; ++k) J[k] = 0;
                    continue;
                }
                for (int c = 0; c < D; ++c) {
                    double add[D], xp[EST], e1[D], e2[D];
                    for (int k = 0; k < D; ++k) add[k] = 0;
                    add[c] = h;
                    for (int k = 0; k < EST; ++k) xp[k] = side == 0 ? xi[k] : xj[k];
                    model_oplus<KIND>(xp, add, g.model_flags);
                    model_error<KIND>(m, side == 0 ? xp : xi, side == 0 ? xj : xp, qi, qj, e1, g.model_flags);
                    add[c] = -h;
                    for (int k = 0; k < EST; ++k) xp[k] = side == 0 ? xi[k] : xj[k];
                    model_oplus<KIND>(xp, add, g.model_flags);
                    model_error<KIND>(m, side == 0 ? xp : xi, side == 0 ? xj : xp, qi, qj, e2, g.model_flags);
                    for (int r = 0; r < D; ++r) J[r * D + c] = scalar * (e1[r] - e2[r]);
                }
            }
        }
        // O' = rho1 * Omega (full symmetric, row-major; or its diagonal)
        if constexpr (DIAG) {
            if (g.robust_kind != S3O_ROBUST_NONE) {
                double c2 = 0;
#pragma unroll
                for (int r = 0; r < D; ++r) c2 += e[r] * (O[r] * e[r]);
                double r0, r1;
                robustify(g.robust_kind, g.robust_param, c2, r0, r1);
#pragma unroll
                for (int k = 0; k < D; ++k) O[k] *= r1;
            }
        } else {
        if (g.info) {
            int f = 0;
#pragma unroll
            for (int r = 0; r < D; ++r)
#pragma unroll
                for (int c = r; c < D; ++c) {
                    const double o = __ldg(g.info + (size_t)(f++) * g.ne_pad + t);
                    O[r * D + c] = o;
                    O[c * D + r] = o;
                }
        } else {
#pragma unroll
            for (int k = 0; k < DD; ++k) O[k] = 0;
#pragma unroll
            for (int k = 0; k < D; ++k) O[k * D + k] = 1;
        }
        if (g.robust_kind != S3O_ROBUST_NONE) {
            double c2 = 0;
#pragma unroll
            for (int r = 0; r < D; ++r) {
                double acc = 0;
#pragma unroll
                for (int c = 0; c < D; ++c) acc += O[r * D + c] * e[c];
                c2 += e[r] * acc;
            }
            double r0, r1;
            robustify(g.robust_kind, g.robust_param, c2, r0, r1);
#pragma unroll
            for (int k = 0; k < DD; ++k) O[k] *= r1;
        }
        }
    }
    double *rec0 = scratch + (size_t)e0 * STRIDE;
    // Row r of J^T O' (J = A or B) -- recomputed where it is needed (a column scaling when the information is diagonal)
    // instead of a 49-entry array kept across the three products.
    auto jto_row = [&](const double *J, int r, double *Pr) {
#pragma unroll
        for (int c = 0; c < D; ++c) {
            double acc = 0;
            if constexpr (DIAG) { if (jnz<SP>(c, r)) acc = J[c * D + r] * O[c]; }
            else {
#pragma unroll
                for (int k = 0; k < D; ++k) if (jnz<SP>(k, r)) acc += J[k * D + r] * O[k * D + c];
            }
            Pr[c] = acc;
        }
    };
    // Every product row goes to the staging buffer as soon as it is formed: at most one row of accumulators is live.
    // [J^T O' J packed | -J^T O' e] of one side
    auto side_piece = [&](const double *J) {
        if (valid) {
            double *mine = stage + lane * (NS + D);
            int f = 0;
#pragma unroll
            for (int r = 0; r < D; ++r) {
                double Pr[D];
                jto_row(J, r, Pr);
#pragma unroll
                for (int c = r; c < D; ++c) {
                    double acc = 0;
#pragma unroll
                    for (int k = 0; k < D; ++k) if ((!DIAG || jnz<SP>(k, r)) && jnz<SP>(k, c)) acc += Pr[k] * J[k * D + c];
                    mine[f++] = acc;
                }
                double acc = 0;
#pragma unroll
                for (int k = 0; k < D; ++k) if (!DIAG || jnz<SP>(k, r)) acc += Pr[k] * e[k];
                mine[NS + r] = -acc;
            }
        }
    };
    // ---- vertex(0) side
    side_piece(A);
    if constexpr (NS + D >= 32) warp_copy_piece<NS + D>(stage, rec0, STRIDE, lane, nvalid);
    else warp_copy_piece_small<NS + D>(stage, rec0, STRIDE, lane, nvalid);
    // ---- cross term Hij = (A^T O') B
    double *cross_dst = scratch + (size_t)g.ne_pad * STRIDE + (size_t)t * DD;
    bool flip = false;         // stored block is (min,max): vertex(0) on the max side -> transpose
    if (src >= 0) { cross_dst = Hdirect + (size_t)kb * DD; flip = (src & 1) != 0; }
    if (valid) {
        double *mine = stage + lane * DD;
#pragma unroll
        for (int r = 0; r < D; ++r) {
            double Pr[D];
            jto_row(A, r, Pr);
#pragma unroll
            for (int c = 0; c < D; ++c) {
                double acc = 0;
#pragma unroll
                for (int k = 0; k < D; ++k) if ((!DIAG || jnz<SP>(k, r)) && jnz<SP>(k, c)) acc += Pr[k] * B[k * D + c];
                mine[flip ? c * D + r : r * D + c] = acc;
            }
        }
    }
    warp_copy_piece_to<DD>(stage, dptr, cross_dst, lane, nvalid);
    // ---- vertex(1) side
    side_piece(B);
    if constexpr (NS + D >= 32) warp_copy_piece<NS + D>(stage, rec0 + (NS + D), STRIDE, lane, nvalid);
    else warp_copy_piece_small<NS + D>(stage, rec0 + (NS + D), STRIDE, lane, nvalid);
}

void launch_linearize(const GraphDev &g, int jac_mode, double h, double *scratch, const int32_t *e_blk,
                      const int32_t *blk_src, double *Hdirect, cudaStream_t st) {
    if (g.ne == 0) return;
    constexpr int NT = 64;
    const int grid = (g.ne + NT - 1) / NT;
    const bool diag = g.info == nullptr || g.info_diag;
#define S3O_LIN(KIND)                                                                                  \
    if (jac_mode == S3O_JAC_ANALYTIC) {                                                                \
        if (diag) linearize_kernel<KIND, S3O_JAC_ANALYTIC, NT, true><<<grid, NT, 0, st>>>(g, h, scratch, e_blk, blk_src, Hdirect);   \
        else linearize_kernel<KIND, S3O_JAC_ANALYTIC, NT, false><<<grid, NT, 0, st>>>(g, h, scratch, e_blk, blk_src, Hdirect);      \
    } else {                                                                                           \
        if (diag) linearize_kernel<KIND, S3O_JAC_NUMERIC, NT, true><<<grid, NT, 0, st>>>(g, h, scratch, e_blk, blk_src, Hdirect);    \
        else linearize_kernel<KIND, S3O_JAC_NUMERIC, NT, false><<<grid, NT, 0, st>>>(g, h, scratch, e_blk, blk_src, Hdirect);       \
    }
    switch (g.kind) {
    case S3O_KIND_SIM3: S3O_LIN(S3O_KIND_SIM3) break;
    case S3O_KIND_SCALE_TRANS: S3O_LIN(S3O_KIND_SCALE_TRANS) break;
    case S3O_KIND_SCALE: S3O_LIN(S3O_KIND_SCALE) break;
    }
#undef S3O_LIN
}

// ======================================================================================
// assemble: scratch records -> BSR-upper blocks and b (fixed order, no atomics)
// ======================================================================================
template <int D>
__global__ void assemble_kernel(GraphDev g, StructDev s, const double *__restrict__ scratch, double *__restrict__ H,
                                double *__restrict__ b) {
    constexpr int DD = D * D, NS = packed_size(D), SIDE = NS + D;
    // work items: SIDE per diagonal block (one per PACKED entry of the symmetric block, which it writes to both
    // triangles, and one per entry of b), then D*D per off-diagonal block fed by more than one edge; single-edge
    // off-diagonal blocks were written in place by linearize_kernel
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long n_diag = (long long)g.nf * SIDE;
    if (tid < n_diag) {
        const int row = (int)(tid / SIDE), f = (int)(tid - (long long)row * SIDE);
        const double *src = scratch + f;
        double acc = 0;
        const int ib = s.inc_ptr[row], ie = s.inc_ptr[row + 1];
        int n = ib;
        for (; n + 8 <= ie; n += 8) {     // eight independent loads in flight, summed in list order
            double v[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) v[q] = src[(size_t)s.inc_ent[n + q] * SIDE];
#pragma unroll
            for (int q = 0; q < 8; ++q) acc += v[q];
        }
        for (; n + 2 <= ie; n += 2) {
            const double v0 = src[(size_t)s.inc_ent[n] * SIDE], v1 = src[(size_t)s.inc_ent[n + 1] * SIDE];
            acc += v0; acc += v1;
        }
        if (n < ie) acc += src[(size_t)s.inc_ent[n] * SIDE];
        if (f < NS) {
            int r = 0, c = f;           // packed upper triangle, row-major: row r holds D - r entries
            while (c >= D - r) { c -= D - r; ++r; }
            c += r;
            double *blk = H + (size_t)s.rowptr[row] * DD;
            blk[r * D + c] = acc;
            if (r != c) blk[c * D + r] = acc;
        } else {
            b[(size_t)row * D + (f - NS)] = acc;
        }
        return;
    }
    const long long m = tid - n_diag;
    const long long w = m / DD;
    if (w >= s.n_multi) return;
    const int el = (int)(m - w * DD);
    const int k = s.multi_blk[w];
    const int r = el / D, c = el - r * D;
    double acc = 0;
    const int eb = s.blk_ebeg[k], ee = s.blk_eend[k];
    const double *cross = scratch + (size_t)g.ne_pad * (2 * SIDE);
    for (int t = eb; t < ee; ++t) {
        // stored block is (min,max); when vertex(0) is the max side the edge's A^T O' B is its transpose
        const bool transposed = g.hidx[g.sv0[t]] > g.hidx[g.sv1[t]];
        acc += cross[(size_t)t * DD + (transposed ? c * D + r : r * D + c)];
    }
    H[(size_t)k * DD + el] = acc;
}

void launch_assemble(const GraphDev &g, const StructDev &s, const double *scratch, double *H, double *b,
                     cudaStream_t st) {
    if (g.nb == 0) return;
    const long long total = (long long)g.nf * (packed_size(g.d) + g.d) + (long long)s.n_multi * g.d * g.d;
    const int grid = (int)((total + 255) / 256);
    switch (g.d) {
    case 7: assemble_kernel<7><<<grid, 256, 0, st>>>(g, s, scratch, H, b); break;
    case 4: assemble_kernel<4><<<grid, 256, 0, st>>>(g, s, scratch, H, b); break;
    case 1: assemble_kernel<1><<<grid, 256, 0, st>>>(g, s, scratch, H, b); break;
    }
}

// ======================================================================================
// retraction
// ======================================================================================
template <int KIND>
__global__ void retract_kernel(GraphDev g, const double *__restrict__ x, double *__restrict__ est_out) {
    constexpr int D = Model<KIND>::D, EST = Model<KIND>::EST;
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= g.nv) return;
    double xs[EST];
    load_planes<EST>(g.est, g.nv_pad, v, xs);
    const int hcol = g.ghidx ? g.ghidx[v] : g.hidx[v];
    if (hcol >= 0) {
        double delta[D];
#pragma unroll
        for (int k = 0; k < D; ++k) delta[k] = x[(size_t)hcol * D + k];
        model_oplus<KIND>(xs, delta, g.model_flags);
    }
#pragma unroll
    for (int k = 0; k < EST; ++k) est_out[(size_t)k * g.nv_pad + v] = xs[k];
}

void launch_retract(const GraphDev &g, const double *x, double *est_out, cudaStream_t st) {
    if (g.nv == 0) return;
    const int grid = (g.nv + 127) / 128;
    switch (g.kind) {
    case S3O_KIND_SIM3: retract_kernel<S3O_KIND_SIM3><<<grid, 128, 0, st>>>(g, x, est_out); break;
    case S3O_KIND_SCALE_TRANS: retract_kernel<S3O_KIND_SCALE_TRANS><<<grid, 128, 0, st>>>(g, x, est_out); break;
    case S3O_KIND_SCALE: retract_kernel<S3O_KIND_SCALE><<<grid, 128, 0, st>>>(g, x, est_out); break;
    }
}

// ======================================================================================
// max diagonal, computeScale
// ======================================================================================
template <int D, int NT>
__global__ void maxdiag_kernel(const double *__restrict__ H, const int32_t *__restrict__ rowptr, int nf,
                               double *__restrict__ partials, DevScalars *sc) {
    __shared__ double sh[32];
    double local = 0;
    for (int t = blockIdx.x * NT + threadIdx.x; t < nf * D; t += gridDim.x * NT) {
        const int i = t / D, j = t - i * D;
        local = fmax(local, fabs(H[(size_t)rowptr[i] * D * D + j * D + j]));
    }
    const double bm = block_max<NT>(local, sh);
    if (threadIdx.x == 0) partials[blockIdx.x] = bm;
    if (last_block(&sc->counters[1])) {
        double v = 0;
        for (int i = threadIdx.x; i < (int)gridDim.x; i += NT) v = fmax(v, __ldcg(partials + i));
        v = block_max<NT>(v, sh);
        if (threadIdx.x == 0) sc->maxdiag = v;
    }
}

void launch_maxdiag(int d, const double *H, const int32_t *rowptr, int nf, double *partials, DevScalars *sc,
                    cudaStream_t st) {
    constexpr int NT = 256;
    const int grid = reduce_grid(nf * d, NT);
    switch (d) {
    case 7: maxdiag_kernel<7, NT><<<grid, NT, 0, st>>>(H, rowptr, nf, partials, sc); break;
    case 4: maxdiag_kernel<4, NT><<<grid, NT, 0, st>>>(H, rowptr, nf, partials, sc); break;
    case 6: maxdiag_kernel<6, NT><<<grid, NT, 0, st>>>(H, rowptr, nf, partials, sc); break;
    case 1: maxdiag_kernel<1, NT><<<grid, NT, 0, st>>>(H, rowptr, nf, partials, sc); break;
    }
}

template <int NT>
__global__ void scale_kernel(int n, const double *__restrict__ x, const double *__restrict__ b, double lambda,
                             double *__restrict__ partials, DevScalars *sc) {
    __shared__ double sh[32];
    double local = 0, lmax = 0;
    for (int t = blockIdx.x * NT + threadIdx.x; t < n; t += gridDim.x * NT) {
        const double xv = x[t];
        local += xv * (lambda * xv + b[t]);
        lmax = fmax(lmax, fabs(xv));
    }
    const double bs = block_sum<NT>(local, sh);
    const double bm = block_max<NT>(lmax, sh);
    if (threadIdx.x == 0) { partials[blockIdx.x] = bs; partials[kMaxPartials + blockIdx.x] = bm; }
    if (last_block(&sc->counters[2])) {
        const double tot = sum_partials<NT>(partials, gridDim.x, sh);
        double v = 0;
        for (int i = threadIdx.x; i < (int)gridDim.x; i += NT) v = fmax(v, __ldcg(partials + kMaxPartials + i));
        v = block_max<NT>(v, sh);
        if (threadIdx.x == 0) { sc->scale = tot; sc->xmax = v; }
    }
}

void launch_scale(int n, const double *x, const double *b, double lambda, double *partials, DevScalars *sc,
                  cudaStream_t st) {
    constexpr int NT = 256;
    scale_kernel<NT><<<reduce_grid(n, NT), NT, 0, st>>>(n, x, b, lambda, partials, sc);
}

// ======================================================================================
// block-Jacobi preconditioner: Minv_i = (H_ii + lambda I)^-1 by Cholesky, stored as its packed upper triangle
// ======================================================================================
template <int D>
__global__ void precond_kernel(const double *__restrict__ H, const int32_t *__restrict__ rowptr, int nf, double lambda,
                               double *__restrict__ Minv, DevScalars *sc) {
    constexpr int DD = D * D;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nf) return;
    double L[DD], Li[DD];
    const double *Hd = H + (size_t)rowptr[i] * DD;
#pragma unroll
    for (int k = 0; k < DD; ++k) L[k] = Hd[k];
#pragma unroll
    for (int k = 0; k < D; ++k) L[k * D + k] += lambda;
    bool ok = true;
    // in-place lower Cholesky
#pragma unroll
    for (int j = 0; j < D; ++j) {
        double djj = L[j * D + j];
#pragma unroll
        for (int k = 0; k < j; ++k) djj -= L[j * D + k] * L[j * D + k];
        if (!(djj > 0)) { ok = false; djj = 1; }
        const double ljj = sqrt(djj);
        L[j * D + j] = ljj;
        const double inv = 1.0 / ljj;
#pragma unroll
        for (int r = j + 1; r < D; ++r) {
            double v = L[r * D + j];
#pragma unroll
            for (int k = 0; k < j; ++k) v -= L[r * D + k] * L[j * D + k];
            L[r * D + j] = v * inv;
        }
    }
    // Li = L^-1 (lower)
#pragma unroll
    for (int c = 0; c < D; ++c) {
#pragma unroll
        for (int r = 0; r < D; ++r) {
            if (r < c) { Li[r * D + c] = 0; continue; }
            double v = (r == c) ? 1.0 : 0.0;
#pragma unroll
            for (int k = c; k < r; ++k) v -= L[r * D + k] * Li[k * D + c];
            Li[r * D + c] = v / L[r * D + r];
        }
    }
    // Minv = Li^T Li, packed upper triangle (sym_off)
    double *out = Minv + (size_t)i * sym_size<D>();
    int f = 0;
#pragma unroll
    for (int r = 0; r < D; ++r)
#pragma unroll
        for (int c = r; c < D; ++c) {
            double v = 0;
#pragma unroll
            for (int k = c; k < D; ++k) v += Li[k * D + r] * Li[k * D + c];
            out[f++] = ok ? v : (r == c ? 1.0 : 0.0);
        }
    if (!ok) sc->precond_fail = 1;
}

void launch_precond(int d, const double *H, const int32_t *rowptr, int nf, double lambda, double *Minv,
                    DevScalars *sc, cudaStream_t st) {
    if (nf == 0) return;
    const int grid = (nf + 127) / 128;
    switch (d) {
    case 7: precond_kernel<7><<<grid, 128, 0, st>>>(H, rowptr, nf, lambda, Minv, sc); break;
    case 4: precond_kernel<4><<<grid, 128, 0, st>>>(H, rowptr, nf, lambda, Minv, sc); break;
    case 6: precond_kernel<6><<<grid, 128, 0, st>>>(H, rowptr, nf, lambda, Minv, sc); break;
    case 1: precond_kernel<1><<<grid, 128, 0, st>>>(H, rowptr, nf, lambda, Minv, sc); break;
    }
}

// ======================================================================================
// symmetric BSR-upper SpMV:  q = (H + lambda I) p  using every stored block once
// ======================================================================================
// A group of GL lanes owns one block row.  The CTA's rows cover a contiguous range of the block
// array, which is staged through shared memory in coalesced tiles.  For an off-diagonal block
// (i,j) the group accumulates H_ij p_j into its own row and writes the transposed product
// t = H_ij^T p_i to T[k]; the column owner adds its T entries in fixed order (finish_q /
// pcg_update).  p.q is formed here as sum_i p_i.(diag_i + 2 off_i), so no second pass over q
// is needed before alpha.

template <int D, int NT, int TB>
__global__ void __launch_bounds__(NT) spmv_kernel(const double *__restrict__ H, StructDev s, int nf, double lambda,
                                                  const double *__restrict__ p, double *__restrict__ q1,
                                                  double *__restrict__ T, double *__restrict__ partials,
                                                  DevScalars *sc, int pcg_mode) {
    constexpr int GL = GroupLanes<D>::value, DD = D * D, RPC = NT / GL;
    __shared__ double tile[TB * DD];
    __shared__ double sh[32];
    if (pcg_mode && sc->done) return;
    const int g = threadIdx.x / GL, l = threadIdx.x % GL;
    const int row0 = blockIdx.x * RPC;
    const int row1 = min(row0 + RPC, nf);
    const int i = row0 + g;
    const bool active = i < nf;
    const int kb = active ? s.rowptr[i] : 0, ke = active ? s.rowptr[i + 1] : 0;
    const int kbeg = s.rowptr[row0], kend = s.rowptr[row1];
    double pi[D];
#pragma unroll
    for (int c = 0; c < D; ++c) pi[c] = active ? p[(size_t)i * D + c] : 0.0;
    double y1 = 0, y2 = 0;
    for (int sub = kbeg; sub < kend; sub += TB) {
        const int cnt = min(TB, kend - sub);
        const double *src = H + (size_t)sub * DD;
        for (int idx = threadIdx.x; idx < cnt * DD; idx += NT) tile[idx] = __ldcs(src + idx);
        __syncthreads();
        const int a = max(kb, sub), bnd = min(ke, sub + cnt);
        for (int k = a; k < bnd; ++k) {
            const int j = s.colidx[k];
            const double *Hs = tile + (k - sub) * DD;
            if (j == i) {
                if (l < D) {
                    double acc = lambda * pi[l];
#pragma unroll
                    for (int c = 0; c < D; ++c) acc += Hs[l * D + c] * pi[c];
                    y1 += acc;
                }
            } else {
                double pj[D];
#pragma unroll
                for (int c = 0; c < D; ++c) pj[c] = p[(size_t)j * D + c];
                if (l < D) {
                    double acc = 0, t = 0;
#pragma unroll
                    for (int c = 0; c < D; ++c) {
                        acc += Hs[l * D + c] * pj[c];
                        t += Hs[c * D + l] * pi[c];
                    }
                    y2 += acc;
                    T[(size_t)k * D + l] = t;
                }
            }
        }
        __syncthreads();
    }
    double local = 0;
    if (active && l < D) {
        q1[(size_t)i * D + l] = y1 + y2;
        local = pi[l] * (y1 + 2.0 * y2);
    }
    if (!pcg_mode) return;
    const double bs = block_sum<NT>(local, sh);
    if (threadIdx.x == 0) partials[blockIdx.x] = bs;
    if (last_block(&sc->counters[3])) {
        const double pq = sum_partials<NT>(partials, gridDim.x, sh);
        if (threadIdx.x == 0) {
            sc->pq = pq;
            fin_spmv(sc);
        }
    }
}

template <int D> struct SpmvCfg { static constexpr int NT = 256; static constexpr int TB = D >= 6 ? 64 : (D == 4 ? 128 : 512); };

void launch_spmv(int d, const double *H, const StructDev &s, int nf, double lambda, const double *p, double *q1,
                 double *T, double *partials, DevScalars *sc, int pcg_mode, cudaStream_t st) {
    if (nf == 0) return;
#define S3O_SPMV(D)                                                                                      \
    {                                                                                                    \
        constexpr int NT = SpmvCfg<D>::NT, TB = SpmvCfg<D>::TB, RPC = NT / GroupLanes<D>::value;         \
        const int grid = (nf + RPC - 1) / RPC;                                                           \
        spmv_kernel<D, NT, TB><<<grid, NT, 0, st>>>(H, s, nf, lambda, p, q1, T, partials, sc, pcg_mode); \
    }
    switch (d) {
    case 7: S3O_SPMV(7) break;
    case 4: S3O_SPMV(4) break;
    case 6: S3O_SPMV(6) break;
    case 1: S3O_SPMV(1) break;
    }
#undef S3O_SPMV
}

// q = q1 + sum of the transposed products addressed to each column (stand-alone SpMV only)
template <int D>
__global__ void finish_q_kernel(StructDev s, int nf, const double *__restrict__ q1, const double *__restrict__ T,
                                double *__restrict__ q) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nf * D) return;
    const int i = t / D, l = t - i * D;
    double acc = q1[t];
    for (int n = s.colT_ptr[i]; n < s.colT_ptr[i + 1]; ++n) acc += T[(size_t)s.colT_blk[n] * D + l];
    q[t] = acc;
}
void launch_finish_q(int d, const StructDev &s, int nf, const double *q1, const double *T, double *q, cudaStream_t st) {
    if (nf == 0) return;
    const int grid = (nf * d + 255) / 256;
    switch (d) {
    case 7: finish_q_kernel<7><<<grid, 256, 0, st>>>(s, nf, q1, T, q); break;
    case 4: finish_q_kernel<4><<<grid, 256, 0, st>>>(s, nf, q1, T, q); break;
    case 6: finish_q_kernel<6><<<grid, 256, 0, st>>>(s, nf, q1, T, q); break;
    case 1: finish_q_kernel<1><<<grid, 256, 0, st>>>(s, nf, q1, T, q); break;
    }
}

// ======================================================================================
// PCG vector kernels
// ======================================================================================
template <int D, int NT>
__global__ void __launch_bounds__(NT) pcg_init_kernel(int nf, const double *__restrict__ b, const double *__restrict__ Minv,
                                                      double *__restrict__ x, double *__restrict__ r,
                                                      double *__restrict__ z, double *__restrict__ p,
                                                      double *__restrict__ partials, DevScalars *sc, double tol,
                                                      int max_iter, int dist) {
    constexpr int GL = GroupLanes<D>::value, DD = D * D, RPC = NT / GL;
    __shared__ double sh[32];
    const int g = threadIdx.x / GL, l = threadIdx.x % GL;
    double lrz = 0, lrr = 0;
    for (int base = blockIdx.x * RPC; base < nf; base += gridDim.x * RPC) {
        // the whole CTA walks the same number of row batches, so the full-mask shuffles converge
        const int i = base + g;
        const bool act = i < nf && l < D;
        const double rl = act ? b[(size_t)i * D + l] : 0.0;
        double zl = 0;
#pragma unroll
        for (int c = 0; c < D; ++c) {
            const double rc = __shfl_sync(0xffffffffu, rl, c, GL);
            if (act) zl += Minv[(size_t)i * sym_size<D>() + sym_off<D>(l, c)] * rc;
        }
        if (act) {
            x[(size_t)i * D + l] = 0;
            r[(size_t)i * D + l] = rl;
            z[(size_t)i * D + l] = zl;
            p[(size_t)i * D + l] = zl;
            lrz += rl * zl;
            lrr += rl * rl;
        }
    }
    const double s1 = block_sum<NT>(lrz, sh);
    const double s2 = block_sum<NT>(lrr, sh);
    if (threadIdx.x == 0) { partials[blockIdx.x] = s1; partials[kMaxPartials + blockIdx.x] = s2; }
    if (last_block(&sc->counters[4])) {
        const double rz = sum_partials<NT>(partials, gridDim.x, sh);
        const double rr = sum_partials<NT>(partials + kMaxPartials, gridDim.x, sh);
        if (threadIdx.x == 0) {
            sc->rz_new = rz; sc->rr = rr;
            if (!dist) fin_init(sc, tol, max_iter);
        }
    }
}

template <int D, int NT>
__global__ void __launch_bounds__(NT) pcg_update_kernel(StructDev s, int nf, const double *__restrict__ q1,
                                                        const double *__restrict__ T, const double *__restrict__ Minv,
                                                        const double *__restrict__ p, double *__restrict__ x,
                                                        double *__restrict__ r, double *__restrict__ z,
                                                        double *__restrict__ partials, DevScalars *sc, int dist) {
    constexpr int GL = GroupLanes<D>::value, DD = D * D, RPC = NT / GL;
    __shared__ double sh[32];
    if (sc->done) return;
    const double alpha = sc->alpha;
    const int g = threadIdx.x / GL, l = threadIdx.x % GL;
    double lrz = 0, lrr = 0;
    for (int base = blockIdx.x * RPC; base < nf; base += gridDim.x * RPC) {
        const int i = base + g;
        const bool act = i < nf && l < D;
        double rl = 0;
        if (act) {
            double q = q1[(size_t)i * D + l];
            for (int n = s.colT_ptr[i]; n < s.colT_ptr[i + 1]; ++n) q += T[(size_t)s.colT_blk[n] * D + l];
            x[(size_t)i * D + l] += alpha * p[(size_t)i * D + l];
            rl = r[(size_t)i * D + l] - alpha * q;
            r[(size_t)i * D + l] = rl;
        }
        double zl = 0;
#pragma unroll
        for (int c = 0; c < D; ++c) {
            const double rc = __shfl_sync(0xffffffffu, rl, c, GL);
            if (act) zl += Minv[(size_t)i * sym_size<D>() + sym_off<D>(l, c)] * rc;
        }
        if (act) {
            z[(size_t)i * D + l] = zl;
            lrz += rl * zl;
            lrr += rl * rl;
        }
    }
    const double s1 = block_sum<NT>(lrz, sh);
    const double s2 = block_sum<NT>(lrr, sh);
    if (threadIdx.x == 0) { partials[blockIdx.x] = s1; partials[kMaxPartials + blockIdx.x] = s2; }
    if (last_block(&sc->counters[5])) {
        const double rz = sum_partials<NT>(partials, gridDim.x, sh);
        const double rr = sum_partials<NT>(partials + kMaxPartials, gridDim.x, sh);
        if (threadIdx.x == 0) {
            sc->rz_new = rz;
            sc->rr = rr;
            if (!dist) fin_update(sc);
        }
    }
}

__global__ void pcg_pupdate_kernel(int n, const double *__restrict__ z, double *__restrict__ p, const DevScalars *sc) {
    if (sc->done) return;
    const double beta = sc->beta;
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < n; t += gridDim.x * blockDim.x)
        p[t] = z[t] + beta * p[t];
}

static int vec_grid(int nf, int rpc) {
    int g = (nf + rpc - 1) / rpc;
    if (g > 148 * 8) g = 148 * 8;
    if (g < 1) g = 1;
    return g;
}

void launch_pcg_init(int d, int nf, const double *b, const double *Minv, double *x, double *r, double *z, double *p,
                     double *partials, DevScalars *sc, double tol, int max_iter, int dist, cudaStream_t st) {
    constexpr int NT = 256;
    switch (d) {
    case 7: pcg_init_kernel<7, NT><<<vec_grid(nf, NT / 8), NT, 0, st>>>(nf, b, Minv, x, r, z, p, partials, sc, tol, max_iter, dist); break;
    case 4: pcg_init_kernel<4, NT><<<vec_grid(nf, NT / 4), NT, 0, st>>>(nf, b, Minv, x, r, z, p, partials, sc, tol, max_iter, dist); break;
    case 6: pcg_init_kernel<6, NT><<<vec_grid(nf, NT / 8), NT, 0, st>>>(nf, b, Minv, x, r, z, p, partials, sc, tol, max_iter, dist); break;
    case 1: pcg_init_kernel<1, NT><<<vec_grid(nf, NT), NT, 0, st>>>(nf, b, Minv, x, r, z, p, partials, sc, tol, max_iter, dist); break;
    }
}

void launch_pcg_update(int d, const StructDev &s, int nf, const double *q1, const double *T, const double *Minv,
                       const double *p, double *x, double *r, double *z, double *partials, DevScalars *sc,
                       int dist, cudaStream_t st) {
    constexpr int NT = 256;
    switch (d) {
    case 7: pcg_update_kernel<7, NT><<<vec_grid(nf, NT / 8), NT, 0, st>>>(s, nf, q1, T, Minv, p, x, r, z, partials, sc, dist); break;
    case 4: pcg_update_kernel<4, NT><<<vec_grid(nf, NT / 4), NT, 0, st>>>(s, nf, q1, T, Minv, p, x, r, z, partials, sc, dist); break;
    case 6: pcg_update_kernel<6, NT><<<vec_grid(nf, NT / 8), NT, 0, st>>>(s, nf, q1, T, Minv, p, x, r, z, partials, sc, dist); break;
    case 1: pcg_update_kernel<1, NT><<<vec_grid(nf, NT), NT, 0, st>>>(s, nf, q1, T, Minv, p, x, r, z, partials, sc, dist); break;
    }
}

void launch_pcg_pupdate(int d, int nf, const double *z, double *p, const DevScalars *sc, cudaStream_t st) {
    const int n = nf * d;
    pcg_pupdate_kernel<<<reduce_grid(n, 256), 256, 0, st>>>(n, z, p, sc);
}

int launches_per_pcg_iter() { return 3; }

// ---- peer-to-peer halo flags (partitioned solve) -------------------------------------------------
// Every rank owns one epoch counter in device memory that its neighbours map through CUDA IPC.  Before a
// product the rank publishes the epoch (its p is complete: the kernels that wrote it precede this one on the
// stream) and waits until every neighbour whose entries it reads has published the same epoch.  Overwriting
// p for the next product is safe without a second flag: it happens after the all-reduce of p.q and the
// all-gather of the same iteration, which every neighbour enters only after its product has finished.
__global__ void halo_signal_kernel(long long *own_flag, long long epoch) {
    *reinterpret_cast<volatile long long *>(own_flag) = epoch;
    __threadfence_system();
}
__global__ void halo_wait_kernel(long long *const *peer_flags, int n_peers, long long epoch, DevScalars *sc) {
    const int t = threadIdx.x;
    if (t >= n_peers) return;
    const volatile long long *f = peer_flags[t];
    long long spins = 0;
    while (*f < epoch) {
        // ~1 minute: a peer died.  Do not leave the iteration on this rank alone (the peers would hang in the next
        // collective): flag it, the SpMV poisons p.q and the all-reduce makes every rank break down together.
        if (++spins > (1ll << 25)) { sc->halo_fail = 1; break; }
    }
    __threadfence_system();
}
void launch_halo_signal(long long *own_flag, long long epoch, cudaStream_t st) { halo_signal_kernel<<<1, 1, 0, st>>>(own_flag, epoch); }
void launch_halo_wait(long long *const *peer_flags, int n_peers, long long epoch, DevScalars *sc, cudaStream_t st) {
    if (n_peers > 0) halo_wait_kernel<<<1, 32, 0, st>>>(peer_flags, n_peers, epoch, sc);
}

// small vector helpers of s3o_smallest_eigenvector
__global__ void scale_vec_kernel(int n, const double *__restrict__ in, double s, double *__restrict__ out) {
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < n; t += gridDim.x * blockDim.x) out[t] = in[t] * s;
}
__global__ void fill_kernel(int n, double a, double b, double *__restrict__ out) {   // a, b, a, b, ...
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < n; t += gridDim.x * blockDim.x) out[t] = (t & 1) ? b : a;
}
void launch_scale_vec(int n, const double *in, double s, double *out, cudaStream_t st) {
    scale_vec_kernel<<<reduce_grid(n, 256), 256, 0, st>>>(n, in, s, out);
}
void launch_fill_const(int n, double v, double *out, cudaStream_t st) { fill_kernel<<<reduce_grid(n, 256), 256, 0, st>>>(n, v, v, out); }
void launch_fill_alternating(int n, double *out, cudaStream_t st) {
    const double v = 1.0 / sqrt((double)(n > 0 ? n : 1));
    fill_kernel<<<reduce_grid(n, 256), 256, 0, st>>>(n, v, -v, out);
}

__global__ void pcg_fin_init_kernel(DevScalars *sc, double tol, int max_iter) { fin_init(sc, tol, max_iter); }
__global__ void pcg_fin_spmv_kernel(DevScalars *sc) { if (!sc->done) fin_spmv(sc); }
__global__ void pcg_fin_update_kernel(DevScalars *sc) { if (!sc->done) fin_update(sc); }
void launch_pcg_fin_init(DevScalars *sc, double tol, int max_iter, cudaStream_t st) { pcg_fin_init_kernel<<<1, 1, 0, st>>>(sc, tol, max_iter); }
void launch_pcg_fin_spmv(DevScalars *sc, cudaStream_t st) { pcg_fin_spmv_kernel<<<1, 1, 0, st>>>(sc); }
void launch_pcg_fin_update(DevScalars *sc, cudaStream_t st) { pcg_fin_update_kernel<<<1, 1, 0, st>>>(sc); }

// gathers the rows a peer needs (halo send buffer): out[n][d] = vec[idx[n]][d]
__global__ void pack_rows_kernel(int d, const double *__restrict__ vec, const int32_t *__restrict__ idx, int n,
                                 double *__restrict__ out, const DevScalars *sc) {
    if (sc->done) return;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * d) return;
    const int k = t / d, c = t - k * d;
    out[t] = vec[(size_t)idx[k] * d + c];
}
void launch_pack_rows(int d, const double *vec, const int32_t *idx, int n, double *out, const DevScalars *sc,
                      cudaStream_t st) {
    if (n == 0) return;
    pack_rows_kernel<<<(n * d + 255) / 256, 256, 0, st>>>(d, vec, idx, n, out, sc);
}

}  // namespace s3o
