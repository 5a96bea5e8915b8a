// ba.cu -- bundle adjustment on the device (kind S3O_KIND_BA): the reference's ba_demo path.
//
// Replaces, for the graph bal_example.cpp:98-194 builds (SE3 cameras ids 0..C-1, marginalised XYZ
// points, EdgeProjectXYZ2UV observations with vertex(0) = point and vertex(1) = camera, Huber
// delta 2.5, one CameraParameters), the g2o work behind optimizer.optimize() (bal_example.cpp:213):
//   computeActiveErrors / activeRobustChi2        -> ba_chi2_kernel
//   EdgeProjectXYZ2UV::linearizeOplus (analytic)  -> ba_linearize_kernel (one thread per observation)
//   constructQuadraticForm                        -> per-observation records, gathered in fixed order by
//                                                    ba_assemble_points_kernel / ba_assemble_cameras_kernel
//   BlockSolver_6_3::solve, Schur branch          -> point-block inverses, Y = Hpl Hll^-1, the
//                                                    block-sparse contraction S = Hpp - sum Y Hpl^T
//                                                    (ba_schur_kernel, fixed-order gather per S block),
//                                                    block-Jacobi PCG on S (the BSR SpMV of spmv.cu with
//                                                    6x6 blocks), back-substitution of the points
//   VertexSE3Expmap / VertexSBAPointXYZ oplus     -> ba_retract_kernel
// All arithmetic fp64; every reduction has a fixed summation order (no floating-point atomics).
// The Schur complement lives in the problem's generic linear-system slots (p->S, p->d_H, p->d_b,
// p->d_x), so the PCG driver (do_solve) is shared with the pose-graph kinds.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "direct.h"
#include "problem.h"
#include "reduce.cuh"
#include "sim3_math.cuh"

namespace s3o {

struct BaState {
    int nc = 0, np = 0, no = 0, nc_pad = 0, np_pad = 0, no_pad = 0;
    int ncf = 0, npf = 0;
    size_t ncon = 0;
    std::vector<uint8_t> cfix, pfix;
    std::vector<int32_t> ocam, opt;         // caller order
    std::vector<double> uv, info;           // caller order; info empty = identity
    std::vector<double> cam0, pt0;          // estimates as last set by the caller (AoS)
    double f = 0, cx = 0, cy = 0;
    std::vector<int32_t> perm;              // sorted position -> caller observation index
    std::vector<int32_t> chidx, phidx;
    // device
    double *d_cam[2] = { nullptr, nullptr }, *d_pt[2] = { nullptr, nullptr };   // SoA [7][nc_pad], [3][np_pad]
    int32_t *d_chidx = nullptr, *d_phidx = nullptr, *d_ocam = nullptr, *d_opt = nullptr;
    int32_t *d_pt_ptr = nullptr, *d_cam_ptr = nullptr, *d_cam_obs = nullptr, *d_con_ptr = nullptr;
    int2 *d_con = nullptr;
    double *d_uv = nullptr, *d_info = nullptr;                                  // SoA [2][no_pad], [3][no_pad]
    double *d_scr = nullptr;                                                    // SoA [36][no_pad]
    double *d_Hpl = nullptr, *d_Y = nullptr;                                    // AoS [no][18]
    double *d_Hpp = nullptr, *d_bp = nullptr, *d_Hll = nullptr, *d_bl = nullptr;
    double *d_Dinv = nullptr, *d_dl = nullptr, *d_xl = nullptr;
    double *d_cam_snap = nullptr, *d_pt_snap = nullptr;
    // marginal covariances (s3o_ba_compute_marginals)
    std::vector<int32_t> pt_ptr, socam;     // observations sorted by point: per-point ranges and their cameras
    int marg_check = -1;                    // host checks of this structure: -1 not run, else their return code
    std::string marg_msg;
    bool marg_lists = false;                // point gather lists below built, on the plan numbered marg_serial
    uint64_t marg_serial = 0;
    int32_t *d_mo_ptr = nullptr, *d_mo_obs = nullptr, *d_mp_sig = nullptr;
    int64_t *d_mp_ptr = nullptr;
    // per call: requested points, camera-point slots, output map, staging and result
    int32_t *d_mrq = nullptr, *d_mcl_ptr = nullptr, *d_mcl_a = nullptr, *d_msrc = nullptr;
    int64_t *d_mdst = nullptr;
    double *d_mpt = nullptr, *d_mout = nullptr;
    int *d_mflag = nullptr;
    size_t cap_mrq = 0, cap_mcl_ptr = 0, cap_mcl_a = 0, cap_msrc = 0, cap_mdst = 0, cap_mpt = 0, cap_mout = 0;
};

namespace {

constexpr int kScr = 36;   // per-observation record: Hcc upper 21 | bc 6 | Hll upper 6 | bl 3

struct BaDev {
    int nc, np, no, nc_pad, np_pad, no_pad, ncf, npf;
    const double *cam, *pt;
    const int32_t *chidx, *phidx, *ocam, *opt;
    const double *uv, *info;
    double f, cx, cy;
    int robust_kind;
    double robust_param;
};

BaDev ba_view(const s3o_problem *p, int which) {
    const BaState &B = *p->ba;
    BaDev v{};
    v.nc = B.nc; v.np = B.np; v.no = B.no; v.nc_pad = B.nc_pad; v.np_pad = B.np_pad; v.no_pad = B.no_pad;
    v.ncf = B.ncf; v.npf = B.npf;
    v.cam = B.d_cam[which]; v.pt = B.d_pt[which];
    v.chidx = B.d_chidx; v.phidx = B.d_phidx; v.ocam = B.d_ocam; v.opt = B.d_opt;
    v.uv = B.d_uv; v.info = B.d_info;
    v.f = B.f; v.cx = B.cx; v.cy = B.cy;
    v.robust_kind = p->robust_kind; v.robust_param = p->robust_param;
    return v;
}

// g2o RobustKernelHuber (rows a13); the PTAM kernels are pose-graph only
__device__ __forceinline__ void ba_robustify(int kind, double delta, double e2, double &rho0, double &rho1) {
    if (kind == S3O_ROBUST_HUBER) {
        const double dsqr = delta * delta;
        if (e2 <= dsqr) { rho0 = e2; rho1 = 1; }
        else { const double sq = sqrt(e2); rho0 = 2 * sq * delta - dsqr; rho1 = delta / sq; }
    } else { rho0 = e2; rho1 = 1; }
}

struct ObsGeom { double e[2], xc[3], R[9]; };

// EdgeProjectXYZ2UV::computeError: e = z - (f (x/z, y/z) + pp), x = T.map(p)
__device__ __forceinline__ void ba_error(const BaDev &g, int k, ObsGeom &o) {
    const int c = g.ocam[k], l = g.opt[k];
    const double qx = g.cam[c], qy = g.cam[g.nc_pad + c], qz = g.cam[2 * g.nc_pad + c], qw = g.cam[3 * g.nc_pad + c];
    quat_to_rot(qx, qy, qz, qw, o.R);
    const double X = g.pt[l], Y = g.pt[g.np_pad + l], Z = g.pt[2 * g.np_pad + l];
    o.xc[0] = o.R[0] * X + o.R[1] * Y + o.R[2] * Z + g.cam[4 * g.nc_pad + c];
    o.xc[1] = o.R[3] * X + o.R[4] * Y + o.R[5] * Z + g.cam[5 * g.nc_pad + c];
    o.xc[2] = o.R[6] * X + o.R[7] * Y + o.R[8] * Z + g.cam[6 * g.nc_pad + c];
    o.e[0] = g.uv[k] - (g.f * o.xc[0] / o.xc[2] + g.cx);
    o.e[1] = g.uv[g.no_pad + k] - (g.f * o.xc[1] / o.xc[2] + g.cy);
}

__device__ __forceinline__ void ba_info(const BaDev &g, int k, double &o00, double &o01, double &o11) {
    if (g.info) { o00 = g.info[k]; o01 = g.info[g.no_pad + k]; o11 = g.info[2 * g.no_pad + k]; }
    else { o00 = 1; o01 = 0; o11 = 1; }
}

template <int NT>
__global__ void __launch_bounds__(NT) ba_chi2_kernel(BaDev g, double *__restrict__ partials, DevScalars *sc) {
    __shared__ double sh[32];
    double local = 0;
    for (int k = blockIdx.x * NT + threadIdx.x; k < g.no; k += gridDim.x * NT) {
        ObsGeom o;
        ba_error(g, k, o);
        double o00, o01, o11;
        ba_info(g, k, o00, o01, o11);
        const double c = o00 * o.e[0] * o.e[0] + 2 * o01 * o.e[0] * o.e[1] + o11 * o.e[1] * o.e[1];
        double r0, r1;
        ba_robustify(g.robust_kind, g.robust_param, c, r0, r1);
        local += r0;
    }
    const double bs = block_sum<NT>(local, sh);
    if (threadIdx.x == 0) partials[blockIdx.x] = bs;
    if (last_block(&sc->counters[0])) {
        const double tot = sum_partials<NT>(partials, gridDim.x, sh);
        if (threadIdx.x == 0) sc->chi2 = tot;
    }
}

__global__ void ba_edge_errors_kernel(BaDev g, double *__restrict__ err) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= g.no) return;
    ObsGeom o;
    ba_error(g, k, o);
    err[2 * k] = o.e[0];
    err[2 * k + 1] = o.e[1];
}

// One thread per observation: analytic Jacobians (g2o types_six_dof_expmap.cpp) and the
// quadratic-form products  Jc^T O' Jc, -Jc^T O' e, Jp^T O' Jp, -Jp^T O' e, Jc^T O' Jp.
__global__ void __launch_bounds__(128) ba_linearize_kernel(BaDev g, double *__restrict__ scr, double *__restrict__ Hpl) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= g.no) return;
    ObsGeom o;
    ba_error(g, k, o);
    const bool cfree = g.chidx[g.ocam[k]] >= 0, pfree = g.phidx[g.opt[k]] >= 0;
    const double x = o.xc[0], y = o.xc[1], z = o.xc[2], z2 = z * z, f = g.f;
    double Jp[6], Jc[12];
    {
        const double t0 = f, t2 = -x / z * f, t4 = f, t5 = -y / z * f, iz = -1.0 / z;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            Jp[c] = iz * (t0 * o.R[c] + t2 * o.R[6 + c]);
            Jp[3 + c] = iz * (t4 * o.R[3 + c] + t5 * o.R[6 + c]);
        }
    }
    Jc[0] = x * y / z2 * f; Jc[1] = -(1 + (x * x / z2)) * f; Jc[2] = y / z * f;
    Jc[3] = -1.0 / z * f;   Jc[4] = 0;                        Jc[5] = x / z2 * f;
    Jc[6] = (1 + y * y / z2) * f; Jc[7] = -x * y / z2 * f;    Jc[8] = -x / z * f;
    Jc[9] = 0;              Jc[10] = -1.0 / z * f;            Jc[11] = y / z2 * f;
    double o00, o01, o11;
    ba_info(g, k, o00, o01, o11);
    double r0, r1;
    ba_robustify(g.robust_kind, g.robust_param, o00 * o.e[0] * o.e[0] + 2 * o01 * o.e[0] * o.e[1] + o11 * o.e[1] * o.e[1], r0, r1);
    o00 *= r1; o01 *= r1; o11 *= r1;
    const double Oe0 = o00 * o.e[0] + o01 * o.e[1], Oe1 = o01 * o.e[0] + o11 * o.e[1];
    double JcO[12], JpO[6];   // J^T O' as [dim][2]
#pragma unroll
    for (int a = 0; a < 6; ++a) { JcO[a * 2] = Jc[a] * o00 + Jc[6 + a] * o01; JcO[a * 2 + 1] = Jc[a] * o01 + Jc[6 + a] * o11; }
#pragma unroll
    for (int a = 0; a < 3; ++a) { JpO[a * 2] = Jp[a] * o00 + Jp[3 + a] * o01; JpO[a * 2 + 1] = Jp[a] * o01 + Jp[3 + a] * o11; }
    int fidx = 0;
#pragma unroll
    for (int a = 0; a < 6; ++a)
#pragma unroll
        for (int c = a; c < 6; ++c)
            scr[(size_t)(fidx++) * g.no_pad + k] = cfree ? JcO[a * 2] * Jc[c] + JcO[a * 2 + 1] * Jc[6 + c] : 0.0;
#pragma unroll
    for (int a = 0; a < 6; ++a) scr[(size_t)(21 + a) * g.no_pad + k] = cfree ? -(Jc[a] * Oe0 + Jc[6 + a] * Oe1) : 0.0;
    fidx = 27;
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int c = a; c < 3; ++c)
            scr[(size_t)(fidx++) * g.no_pad + k] = pfree ? JpO[a * 2] * Jp[c] + JpO[a * 2 + 1] * Jp[3 + c] : 0.0;
#pragma unroll
    for (int a = 0; a < 3; ++a) scr[(size_t)(33 + a) * g.no_pad + k] = pfree ? -(Jp[a] * Oe0 + Jp[3 + a] * Oe1) : 0.0;
    double *W = Hpl + (size_t)k * 18;
#pragma unroll
    for (int a = 0; a < 6; ++a)
#pragma unroll
        for (int c = 0; c < 3; ++c)
            W[a * 3 + c] = (cfree && pfree) ? JcO[a * 2] * Jp[c] + JcO[a * 2 + 1] * Jp[3 + c] : 0.0;
}

// One thread per point: H_ll and b_l from the point's (contiguous) observation range, in order.
__global__ void ba_assemble_points_kernel(BaDev g, const int32_t *__restrict__ pt_ptr, const double *__restrict__ scr,
                                          double *__restrict__ Hll, double *__restrict__ bl) {
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= g.np) return;
    const int li = g.phidx[l];
    if (li < 0) return;
    double acc[9];
#pragma unroll
    for (int a = 0; a < 9; ++a) acc[a] = 0;
    for (int k = pt_ptr[l]; k < pt_ptr[l + 1]; ++k)
#pragma unroll
        for (int a = 0; a < 9; ++a) acc[a] += scr[(size_t)(27 + a) * g.no_pad + k];
    double *H = Hll + (size_t)li * 9;
    H[0] = acc[0]; H[1] = acc[1]; H[2] = acc[2];
    H[3] = acc[1]; H[4] = acc[3]; H[5] = acc[4];
    H[6] = acc[2]; H[7] = acc[4]; H[8] = acc[5];
    bl[(size_t)li * 3] = acc[6]; bl[(size_t)li * 3 + 1] = acc[7]; bl[(size_t)li * 3 + 2] = acc[8];
}

// One CTA per camera: H_pp and b_p from the camera's observation list.  27 record elements x 8
// strided groups; the 8 partial sums are added in group order (fixed summation order).
constexpr int kCamGroups = 8;
__global__ void __launch_bounds__(27 * kCamGroups) ba_assemble_cameras_kernel(BaDev g, const int32_t *__restrict__ cam_ptr,
                                                                               const int32_t *__restrict__ cam_obs,
                                                                               const double *__restrict__ scr,
                                                                               double *__restrict__ Hpp, double *__restrict__ bp) {
    __shared__ double part[kCamGroups][27];
    const int c = blockIdx.x;
    const int ci = g.chidx[c];
    if (ci < 0) return;
    const int el = threadIdx.x % 27, grp = threadIdx.x / 27;
    double acc = 0;
    for (int n = cam_ptr[c] + grp; n < cam_ptr[c + 1]; n += kCamGroups) acc += scr[(size_t)el * g.no_pad + cam_obs[n]];
    part[grp][el] = acc;
    __syncthreads();
    if (threadIdx.x < 27) {
        double s = 0;
#pragma unroll
        for (int q = 0; q < kCamGroups; ++q) s += part[q][el];
        part[0][el] = s;
    }
    __syncthreads();
    if (threadIdx.x < 36) {
        const int r = threadIdx.x / 6, cc = threadIdx.x % 6;
        const int lo = r < cc ? r : cc, hi = r < cc ? cc : r;
        Hpp[(size_t)ci * 36 + threadIdx.x] = part[0][lo * 6 - (lo * (lo - 1)) / 2 + (hi - lo)];
    } else if (threadIdx.x < 42) {
        bp[(size_t)ci * 6 + (threadIdx.x - 36)] = part[0][21 + (threadIdx.x - 36)];
    }
}

template <int NT>
__global__ void ba_maxdiag_kernel(const double *__restrict__ Hpp, int ncf, const double *__restrict__ Hll, int npf,
                                  double *__restrict__ partials, DevScalars *sc) {
    __shared__ double sh[32];
    double local = 0;
    const int n1 = ncf * 6, n = n1 + npf * 3;
    for (int t = blockIdx.x * NT + threadIdx.x; t < n; t += gridDim.x * NT) {
        if (t < n1) { const int i = t / 6, j = t - i * 6; local = fmax(local, fabs(Hpp[(size_t)i * 36 + j * 7])); }
        else { const int u = t - n1, i = u / 3, j = u - i * 3; local = fmax(local, fabs(Hll[(size_t)i * 9 + j * 4])); }
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

// (H_ll + lambda I)^-1 by the adjugate, and dl = Dinv b_l
__global__ void ba_point_inverse_kernel(int npf, const double *__restrict__ Hll, const double *__restrict__ bl, double lambda,
                                        double *__restrict__ Dinv, double *__restrict__ dl, DevScalars *sc) {
    const int li = blockIdx.x * blockDim.x + threadIdx.x;
    if (li >= npf) return;
    const double *A = Hll + (size_t)li * 9;
    const double a = A[0] + lambda, b = A[1], c = A[2], d = A[4] + lambda, e = A[5], f = A[8] + lambda;
    const double c00 = d * f - e * e, c01 = c * e - b * f, c02 = b * e - c * d;
    const double det = a * c00 + b * c01 + c * c02;
    double I[9];
    if (!(fabs(det) > 0) || !isfinite(det)) {
        sc->precond_fail = 1;
#pragma unroll
        for (int q = 0; q < 9; ++q) I[q] = 0;
    } else {
        const double id = 1.0 / det;
        I[0] = c00 * id; I[1] = c01 * id; I[2] = c02 * id;
        I[3] = I[1];     I[4] = (a * f - c * c) * id; I[5] = (b * c - a * e) * id;
        I[6] = I[2];     I[7] = I[5]; I[8] = (a * d - b * b) * id;
    }
    double *O = Dinv + (size_t)li * 9;
#pragma unroll
    for (int q = 0; q < 9; ++q) O[q] = I[q];
    const double b0 = bl[(size_t)li * 3], b1 = bl[(size_t)li * 3 + 1], b2 = bl[(size_t)li * 3 + 2];
#pragma unroll
    for (int q = 0; q < 3; ++q) dl[(size_t)li * 3 + q] = I[q * 3] * b0 + I[q * 3 + 1] * b1 + I[q * 3 + 2] * b2;
}

// Y_k = Hpl_k Dinv_l  (6x3), one thread per observation
__global__ void ba_y_kernel(BaDev g, const double *__restrict__ Hpl, const double *__restrict__ Dinv, double *__restrict__ Y) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= g.no) return;
    const int li = g.phidx[g.opt[k]];
    double *out = Y + (size_t)k * 18;
    if (li < 0) {
#pragma unroll
        for (int q = 0; q < 18; ++q) out[q] = 0;
        return;
    }
    const double *W = Hpl + (size_t)k * 18, *D = Dinv + (size_t)li * 9;
#pragma unroll
    for (int r = 0; r < 6; ++r)
#pragma unroll
        for (int c = 0; c < 3; ++c) out[r * 3 + c] = W[r * 3] * D[c] + W[r * 3 + 1] * D[3 + c] + W[r * 3 + 2] * D[6 + c];
}

// S block (BSR-upper order) = [diagonal: Hpp + lambda I] - sum over its contribution list of
// Y_a Hpl_b^T, one thread per block element, contributions in list order.
__global__ void ba_schur_kernel(int nb, const int32_t *__restrict__ blk_row, const int32_t *__restrict__ colidx,
                                const int32_t *__restrict__ con_ptr, const int2 *__restrict__ con,
                                const double *__restrict__ Y, const double *__restrict__ Hpl, const double *__restrict__ Hpp,
                                double lambda, double *__restrict__ S) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long blk64 = t / 36;
    if (blk64 >= nb) return;
    const int blk = (int)blk64, el = (int)(t - blk64 * 36), r = el / 6, c = el - r * 6;
    double acc = 0;
    for (int n = con_ptr[blk]; n < con_ptr[blk + 1]; ++n) {
        const int2 ab = con[n];
        const double *ya = Y + (size_t)ab.x * 18 + r * 3, *wb = Hpl + (size_t)ab.y * 18 + c * 3;
        acc += ya[0] * wb[0] + ya[1] * wb[1] + ya[2] * wb[2];
    }
    const int row = blk_row[blk];
    double base = 0;
    if (colidx[blk] == row) base = Hpp[(size_t)row * 36 + el] + (r == c ? lambda : 0.0);
    S[(size_t)blk * 36 + el] = base - acc;
}

// bs_c = bp_c - sum over the camera's observations of Hpl_k dl_l; one CTA per camera (6 rows x 32 groups)
constexpr int kBsGroups = 32;
__global__ void __launch_bounds__(6 * kBsGroups) ba_schur_rhs_kernel(BaDev g, const int32_t *__restrict__ cam_ptr,
                                                                      const int32_t *__restrict__ cam_obs,
                                                                      const double *__restrict__ Hpl, const double *__restrict__ dl,
                                                                      const double *__restrict__ bp, double *__restrict__ bs) {
    __shared__ double part[kBsGroups][6];
    const int c = blockIdx.x;
    const int ci = g.chidx[c];
    if (ci < 0) return;
    const int r = threadIdx.x % 6, grp = threadIdx.x / 6;
    double acc = 0;
    for (int n = cam_ptr[c] + grp; n < cam_ptr[c + 1]; n += kBsGroups) {
        const int k = cam_obs[n];
        const int li = g.phidx[g.opt[k]];
        if (li < 0) continue;
        const double *W = Hpl + (size_t)k * 18 + r * 3, *d = dl + (size_t)li * 3;
        acc += W[0] * d[0] + W[1] * d[1] + W[2] * d[2];
    }
    part[grp][r] = acc;
    __syncthreads();
    if (threadIdx.x < 6) {
        double s = 0;
#pragma unroll
        for (int q = 0; q < kBsGroups; ++q) s += part[q][r];
        bs[(size_t)ci * 6 + r] = bp[(size_t)ci * 6 + r] - s;
    }
}

// x_l = Dinv (b_l - sum Hpl^T x_c) = dl - Dinv sum Hpl^T x_c, one thread per point
__global__ void ba_backsub_kernel(BaDev g, const int32_t *__restrict__ pt_ptr, const double *__restrict__ Hpl,
                                  const double *__restrict__ Dinv, const double *__restrict__ dl,
                                  const double *__restrict__ xc, double *__restrict__ xl) {
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= g.np) return;
    const int li = g.phidx[l];
    if (li < 0) return;
    double r0 = 0, r1 = 0, r2 = 0;
    for (int k = pt_ptr[l]; k < pt_ptr[l + 1]; ++k) {
        const int ci = g.chidx[g.ocam[k]];
        if (ci < 0) continue;
        const double *W = Hpl + (size_t)k * 18, *x = xc + (size_t)ci * 6;
#pragma unroll
        for (int q = 0; q < 6; ++q) { r0 += W[q * 3] * x[q]; r1 += W[q * 3 + 1] * x[q]; r2 += W[q * 3 + 2] * x[q]; }
    }
    const double *D = Dinv + (size_t)li * 9;
#pragma unroll
    for (int q = 0; q < 3; ++q) xl[(size_t)li * 3 + q] = dl[(size_t)li * 3 + q] - (D[q * 3] * r0 + D[q * 3 + 1] * r1 + D[q * 3 + 2] * r2);
}

// SE3Quat::exp (g2o se3quat.h: theta < 1e-5 -> R = I + Om + Om^2, V = R) and
// VertexSE3Expmap::oplusImpl  T <- exp(delta) * T  with normalizeRotation(); points p += delta
__global__ void ba_retract_kernel(BaDev g, const double *__restrict__ xc, const double *__restrict__ xl,
                                  double *__restrict__ cam_out, double *__restrict__ pt_out) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < g.nc) {
        const int c = t, ci = g.chidx[c];
        double T[7];
#pragma unroll
        for (int q = 0; q < 7; ++q) T[q] = g.cam[(size_t)q * g.nc_pad + c];
        if (ci >= 0) {
            const double *d = xc + (size_t)ci * 6;
            const double wx = d[0], wy = d[1], wz = d[2];
            const double theta = sqrt(wx * wx + wy * wy + wz * wz);
            double Om[9], Om2[9], R[9], V[9];
            skew3(wx, wy, wz, Om);
            mat3_mul(Om, Om, Om2);
            if (theta < 0.00001) {
#pragma unroll
                for (int q = 0; q < 9; ++q) R[q] = Om[q] + Om2[q];
                R[0] += 1; R[4] += 1; R[8] += 1;
#pragma unroll
                for (int q = 0; q < 9; ++q) V[q] = R[q];
            } else {
                const double k1 = sin(theta) / theta, k2 = (1 - cos(theta)) / (theta * theta);
                const double k3 = (theta - sin(theta)) / (theta * theta * theta);
#pragma unroll
                for (int q = 0; q < 9; ++q) { R[q] = k1 * Om[q] + k2 * Om2[q]; V[q] = k2 * Om[q] + k3 * Om2[q]; }
                R[0] += 1; R[4] += 1; R[8] += 1;
                V[0] += 1; V[4] += 1; V[8] += 1;
            }
            double ux, uy, uz, uw;
            rot_to_quat(R, ux, uy, uz, uw);
            const double tx = V[0] * d[3] + V[1] * d[4] + V[2] * d[5];
            const double ty = V[3] * d[3] + V[4] * d[4] + V[5] * d[5];
            const double tz = V[6] * d[3] + V[7] * d[4] + V[8] * d[5];
            // SE3Quat::operator*: t = t1 + r1 t2, r = r1 r2, normalizeRotation()
            double rx, ry, rz;
            quat_rotate(ux, uy, uz, uw, T[4], T[5], T[6], rx, ry, rz);
            const double ax = ux, ay = uy, az = uz, aw = uw, bx = T[0], by = T[1], bz = T[2], bw = T[3];
            double qw = aw * bw - ax * bx - ay * by - az * bz;
            double qx = aw * bx + ax * bw + ay * bz - az * by;
            double qy = aw * by + ay * bw + az * bx - ax * bz;
            double qz = aw * bz + az * bw + ax * by - ay * bx;
            if (qw < 0) { qx = -qx; qy = -qy; qz = -qz; qw = -qw; }
            const double n = sqrt(qx * qx + qy * qy + qz * qz + qw * qw);
            T[0] = qx / n; T[1] = qy / n; T[2] = qz / n; T[3] = qw / n;
            T[4] = tx + rx; T[5] = ty + ry; T[6] = tz + rz;
        }
#pragma unroll
        for (int q = 0; q < 7; ++q) cam_out[(size_t)q * g.nc_pad + c] = T[q];
    }
    if (t < g.np) {
        const int l = t, li = g.phidx[l];
#pragma unroll
        for (int q = 0; q < 3; ++q) {
            double v = g.pt[(size_t)q * g.np_pad + l];
            if (li >= 0) v += xl[(size_t)li * 3 + q];
            pt_out[(size_t)q * g.np_pad + l] = v;
        }
    }
}

// computeScale over cameras and points: sum x_j (lambda x_j + b_j)
template <int NT>
__global__ void ba_scale_kernel(int n1, const double *__restrict__ xc, const double *__restrict__ bp, int n2,
                                const double *__restrict__ xl, const double *__restrict__ bl, double lambda,
                                double *__restrict__ partials, DevScalars *sc) {
    __shared__ double sh[32];
    double local = 0;
    for (int t = blockIdx.x * NT + threadIdx.x; t < n1 + n2; t += gridDim.x * NT) {
        const double xv = t < n1 ? xc[t] : xl[t - n1];
        const double bv = t < n1 ? bp[t] : bl[t - n1];
        local += xv * (lambda * xv + bv);
    }
    const double bs = block_sum<NT>(local, sh);
    if (threadIdx.x == 0) partials[blockIdx.x] = bs;
    if (last_block(&sc->counters[2])) {
        const double tot = sum_partials<NT>(partials, gridDim.x, sh);
        if (threadIdx.x == 0) sc->scale = tot;
    }
}

// ---- marginal covariances: the point phase --------------------------------------------------------------------
// For a free point l with observations O(l) by free cameras, Y_a = Hpl_a Hll^-1 and Sigma_cc = S^-1 (selected inverse):
//   Z_a = sum_{b in O(l)} Sigma_cc(c_a, c_b) Y_b,   Sigma(c_a, l) = -Z_a,   Sigma(l, l) = Hll^-1 + sum_a Y_a^T Z_a.
// One warp per requested point; a group of 6 lanes per observation a (5 groups a warp), lane r of the group owns row r
// of Z_a and sums over b in list order.  Each lane adds its rows' share of Y_a^T Z_a to a lower triangle, which a
// butterfly over the warp reduces (fixed lanes, fixed order: bitwise reproducible); lane 0 adds Hll^-1 and writes the
// triangle mirrored, so Sigma(l, l) is exactly symmetric.  The observation lists: mo_ptr / mo_obs (sorted observation
// index of each free-camera observation, in order); the Sigma_cc operands: mp_sig[mp_ptr[l] + a |O(l)| + b] = (block
// of the selected inverse << 1) | transposed.  Camera-point blocks: cl_a[q] (q in cl_ptr[s] .. cl_ptr[s+1]) is the
// observation whose -Z_a goes to slot q.  A first grid-stride pass flags every free point whose det(Hll) is not > 0.
constexpr int kMargNT = 256;
__global__ void __launch_bounds__(kMargNT) ba_marginal_points_kernel(
    int npf, int nrq, const int32_t *__restrict__ rq, const int32_t *__restrict__ mo_ptr, const int32_t *__restrict__ mo_obs,
    const int64_t *__restrict__ mp_ptr, const int32_t *__restrict__ mp_sig, const double *__restrict__ Sig,
    const double *__restrict__ Y, const double *__restrict__ Dinv, const double *__restrict__ Hll,
    const int32_t *__restrict__ cl_ptr, const int32_t *__restrict__ cl_a, double *__restrict__ pdiag,
    double *__restrict__ pcl, int *fail) {
    const int gtid = blockIdx.x * kMargNT + threadIdx.x, gthreads = gridDim.x * kMargNT;
    for (int li = gtid; li < npf; li += gthreads) {      // the determinant as ba_point_inverse_kernel forms it
        const double *A = Hll + (size_t)li * 9;
        const double a = A[0], b = A[1], c = A[2], d = A[4], e = A[5], f = A[8];
        const double det = a * (d * f - e * e) + b * (c * e - b * f) + c * (b * e - c * d);
        if (!(det > 0) || !isfinite(det)) *fail = 1;
    }
    const int lane = threadIdx.x & 31, g = lane / 6, r = lane - 6 * g;
    for (int s = gtid >> 5; s < nrq; s += gthreads >> 5) {
        const int li = rq ? rq[s] : s;
        const int o0 = mo_ptr[li], nO = mo_ptr[li + 1] - o0;
        const int32_t *sig = mp_sig + mp_ptr[li];
        double P[6] = { 0, 0, 0, 0, 0, 0 };      // (0,0) (1,0) (1,1) (2,0) (2,1) (2,2)
        for (int a0 = 0; a0 < nO; a0 += 5) {
            const int a = a0 + g;
            if (g >= 5 || a >= nO) continue;
            double z0 = 0, z1 = 0, z2 = 0;
            const int32_t *sg = sig + (size_t)a * nO;
            for (int b = 0; b < nO; ++b) {
                const int t = sg[b];
                const double *blk = Sig + (size_t)(t >> 1) * 36;
                const double *yb = Y + (size_t)mo_obs[o0 + b] * 18;
                double v[6];
                if (t & 1) {
#pragma unroll
                    for (int m = 0; m < 6; ++m) v[m] = blk[m * 6 + r];
                } else {
#pragma unroll
                    for (int m = 0; m < 6; ++m) v[m] = blk[r * 6 + m];
                }
#pragma unroll
                for (int m = 0; m < 6; ++m) { z0 += v[m] * yb[m * 3]; z1 += v[m] * yb[m * 3 + 1]; z2 += v[m] * yb[m * 3 + 2]; }
            }
            const double *ya = Y + (size_t)mo_obs[o0 + a] * 18 + r * 3;
            P[0] += ya[0] * z0; P[1] += ya[1] * z0; P[2] += ya[1] * z1;
            P[3] += ya[2] * z0; P[4] += ya[2] * z1; P[5] += ya[2] * z2;
            if (cl_ptr)
                for (int q = cl_ptr[s]; q < cl_ptr[s + 1]; ++q)
                    if (cl_a[q] == a) { double *o = pcl + (size_t)q * 18 + r * 3; o[0] = -z0; o[1] = -z1; o[2] = -z2; }
        }
#pragma unroll
        for (int k = 0; k < 6; ++k)
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) P[k] += __shfl_xor_sync(0xffffffffu, P[k], off);
        if (lane == 0) {
            const double *D = Dinv + (size_t)li * 9;
            const double v00 = D[0] + P[0], v10 = D[3] + P[1], v11 = D[4] + P[2], v20 = D[6] + P[3], v21 = D[7] + P[4], v22 = D[8] + P[5];
            double *o = pdiag + (size_t)s * 9;
            o[0] = v00; o[1] = v10; o[2] = v20;
            o[3] = v10; o[4] = v11; o[5] = v21;
            o[6] = v20; o[7] = v21; o[8] = v22;
        }
    }
}

// The requested blocks, back to back: src[k] = (index << 2) | kind, kind 0 camera-camera (cc, 6x6), 1 point diagonal
// (pdiag, 3x3), 2 camera-point (pcl, 6x3), 3 point-camera (pcl transposed, 3x6); dst[k] = offset in out.
// flag[1] = the factorisation's pivot flag (dfail, may be nullptr).
__global__ void ba_marginal_gather_kernel(int n_pairs, const int32_t *__restrict__ src, const int64_t *__restrict__ dst,
                                          const double *__restrict__ cc, const double *__restrict__ pdiag,
                                          const double *__restrict__ pcl, const int *dfail, int *flag, double *__restrict__ out) {
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (tid == 0) flag[1] = dfail ? *dfail : 0;
    for (long long item = tid; item < (long long)n_pairs * 36; item += (long long)gridDim.x * blockDim.x) {
        const int k = (int)(item / 36), e = (int)(item - (long long)k * 36);
        const int kind = src[k] & 3, idx = src[k] >> 2;
        double *o = out + dst[k];
        if (kind == 0) o[e] = cc[(size_t)idx * 36 + e];
        else if (kind == 1) { if (e < 9) o[e] = pdiag[(size_t)idx * 9 + e]; }
        else if (e < 18) {
            if (kind == 2) o[e] = pcl[(size_t)idx * 18 + e];
            else { const int a = e / 6, b = e - 6 * a; o[e] = pcl[(size_t)idx * 18 + b * 3 + a]; }
        }
    }
}

__global__ void ba_pack_kernel(const double *__restrict__ aos, int n, int n_pad, int dim, double *__restrict__ soa) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * dim) return;
    soa[(size_t)(t % dim) * n_pad + t / dim] = aos[t];
}
__global__ void ba_unpack_kernel(const double *__restrict__ soa, int n, int n_pad, int dim, double *__restrict__ aos) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * dim) return;
    aos[t] = soa[(size_t)(t % dim) * n_pad + t / dim];
}

int grid_cap(long long n, int nt) {
    long long g = (n + nt - 1) / nt;
    if (g > 148 * 8) g = 148 * 8;
    if (g < 1) g = 1;
    return (int)g;
}

void ba_free_device(BaState &B) {
    dev_free(B.d_cam[0]); dev_free(B.d_cam[1]); dev_free(B.d_pt[0]); dev_free(B.d_pt[1]);
    dev_free(B.d_chidx); dev_free(B.d_phidx); dev_free(B.d_ocam); dev_free(B.d_opt);
    dev_free(B.d_pt_ptr); dev_free(B.d_cam_ptr); dev_free(B.d_cam_obs); dev_free(B.d_con_ptr); dev_free(B.d_con);
    dev_free(B.d_uv); dev_free(B.d_info); dev_free(B.d_scr); dev_free(B.d_Hpl); dev_free(B.d_Y);
    dev_free(B.d_Hpp); dev_free(B.d_bp); dev_free(B.d_Hll); dev_free(B.d_bl);
    dev_free(B.d_Dinv); dev_free(B.d_dl); dev_free(B.d_xl);
    dev_free(B.d_cam_snap); dev_free(B.d_pt_snap);
    dev_free(B.d_mo_ptr); dev_free(B.d_mo_obs); dev_free(B.d_mp_sig); dev_free(B.d_mp_ptr);
    dev_free(B.d_mrq); dev_free(B.d_mcl_ptr); dev_free(B.d_mcl_a); dev_free(B.d_msrc); dev_free(B.d_mdst);
    dev_free(B.d_mpt); dev_free(B.d_mout); dev_free(B.d_mflag);
    B.cap_mrq = B.cap_mcl_ptr = B.cap_mcl_a = B.cap_msrc = B.cap_mdst = B.cap_mpt = B.cap_mout = 0;
    B.marg_lists = false;
    B.marg_check = -1;
}

int upload_soa(s3o_problem *p, const std::vector<double> &aos, int n, int n_pad, int dim, double *soa) {
    if (n == 0) return S3O_OK;
    double *tmp = nullptr;
    int rc = dev_alloc(&tmp, aos.size());
    if (rc) return rc;
    cudaError_t e = cudaMemcpyAsync(tmp, aos.data(), aos.size() * sizeof(double), cudaMemcpyHostToDevice, p->stream);
    if (e == cudaSuccess) {
        ba_pack_kernel<<<(n * dim + 255) / 256, 256, 0, p->stream>>>(tmp, n, n_pad, dim, soa);
        e = cudaStreamSynchronize(p->stream);
    }
    cudaFree(tmp);
    if (e != cudaSuccess) { set_error("ba upload: %s", cudaGetErrorString(e)); return S3O_ERR_CUDA; }
    p->stats.h2d_bytes += (int64_t)(aos.size() * sizeof(double));
    p->stats.kernel_launches += 1;
    return S3O_OK;
}

}  // namespace

// ======================================================================================
// hooks called from problem.cu
// ======================================================================================
void ba_destroy(s3o_problem *p) {
    if (!p->ba) return;
    ba_free_device(*p->ba);
    delete p->ba;
    p->ba = nullptr;
}

BaState *ba_state(s3o_problem *p) {
    if (!p->ba) p->ba = new BaState();
    return p->ba;
}

void ba_invalidate(s3o_problem *p) {
    if (p->ba) ba_free_device(*p->ba);
    free_structure(p);
}

// initializeOptimization + BlockSolver::buildStructure for the BA graph: free cameras numbered in
// id order, then the (marginalised) points; H_schur pattern = diagonal + co-observing camera pairs.
int ba_build_structure(s3o_problem *p) {
    BaState &B = *ba_state(p);
    if (B.nc == 0 || B.np == 0) { set_error("s3o_build_structure(BA): set cameras, points and observations first"); return S3O_ERR_INVALID; }
    ba_invalidate(p);
    B.nc_pad = pad32(B.nc); B.np_pad = pad32(B.np); B.no_pad = pad32(B.no);
    B.chidx.assign(B.nc, -1); B.phidx.assign(B.np, -1);
    B.ncf = B.npf = 0;
    for (int c = 0; c < B.nc; ++c) if (!B.cfix[c]) B.chidx[c] = B.ncf++;
    for (int l = 0; l < B.np; ++l) if (!B.pfix[l]) B.phidx[l] = B.npf++;
    // observations sorted by point (stable: ties keep the caller's order)
    std::vector<int32_t> pt_ptr(B.np + 1, 0);
    for (int k = 0; k < B.no; ++k) pt_ptr[B.opt[k] + 1]++;
    for (int l = 0; l < B.np; ++l) pt_ptr[l + 1] += pt_ptr[l];
    B.perm.resize(B.no);
    {
        std::vector<int32_t> fill(pt_ptr.begin(), pt_ptr.end() - 1);
        for (int k = 0; k < B.no; ++k) B.perm[fill[B.opt[k]]++] = k;
    }
    std::vector<int32_t> socam(B.no), sopt(B.no);
    std::vector<double> suv((size_t)B.no * 2), sinfo;
    if (!B.info.empty()) sinfo.resize((size_t)B.no * 3);
    for (int t = 0; t < B.no; ++t) {
        const int k = B.perm[t];
        socam[t] = B.ocam[k]; sopt[t] = B.opt[k];
        suv[(size_t)t * 2] = B.uv[(size_t)k * 2]; suv[(size_t)t * 2 + 1] = B.uv[(size_t)k * 2 + 1];
        if (!B.info.empty()) for (int q = 0; q < 3; ++q) sinfo[(size_t)t * 3 + q] = B.info[(size_t)k * 3 + q];
    }
    std::vector<int32_t> cam_ptr(B.nc + 1, 0), cam_obs(B.no);
    for (int t = 0; t < B.no; ++t) cam_ptr[socam[t] + 1]++;
    for (int c = 0; c < B.nc; ++c) cam_ptr[c + 1] += cam_ptr[c];
    {
        std::vector<int32_t> fill(cam_ptr.begin(), cam_ptr.end() - 1);
        for (int t = 0; t < B.no; ++t) cam_obs[fill[socam[t]]++] = t;
    }
    // camera pairs that co-observe a free point -> the "edges" of the Schur-complement pattern
    std::vector<uint64_t> keys;
    for (int l = 0; l < B.np; ++l) {
        if (B.phidx[l] < 0) continue;
        for (int a = pt_ptr[l]; a < pt_ptr[l + 1]; ++a)
            for (int b = a + 1; b < pt_ptr[l + 1]; ++b) {
                int c1 = socam[a], c2 = socam[b];
                if (c1 == c2 || B.chidx[c1] < 0 || B.chidx[c2] < 0) continue;
                if (c1 > c2) std::swap(c1, c2);
                keys.push_back(((uint64_t)(uint32_t)c1 << 32) | (uint32_t)c2);
            }
        if (keys.size() > (size_t)64 << 20) {      // bound the host buffer: compact as we go
            std::sort(keys.begin(), keys.end());
            keys.erase(std::unique(keys.begin(), keys.end()), keys.end());
        }
    }
    std::sort(keys.begin(), keys.end());
    keys.erase(std::unique(keys.begin(), keys.end()), keys.end());
    std::vector<int32_t> v0(keys.size()), v1(keys.size());
    for (size_t i = 0; i < keys.size(); ++i) { v0[i] = (int32_t)(keys[i] >> 32); v1[i] = (int32_t)(keys[i] & 0xffffffffu); }
    HostStructure &S = p->S;
    build_structure_host(B.nc, B.cfix.data(), (int)keys.size(), v0.data(), v1.data(), S);
    p->nv = B.nc;
    p->ne = (int)keys.size();
    // contribution lists per BSR block: ordered observation pairs (a, b) of one point with
    // row = camera(a) <= col = camera(b) (both free)
    auto find_block = [&](int r, int c) -> int {
        int lo = S.rowptr[r], hi = S.rowptr[r + 1];
        if (r == c) return lo;                      // diagonal block is first in its row
        ++lo;
        const int32_t *beg = S.colidx.data() + lo, *end = S.colidx.data() + hi;
        const int32_t *it = std::lower_bound(beg, end, c);
        return (it != end && *it == c) ? (int)(it - S.colidx.data()) : -1;
    };
    std::vector<int32_t> con_ptr(S.nb + 1, 0);
    std::vector<int2> con;
    for (int pass = 0; pass < 2; ++pass) {
        std::vector<int32_t> fill;
        if (pass == 1) {
            for (int k = 0; k < S.nb; ++k) con_ptr[k + 1] += con_ptr[k];
            con.resize((size_t)con_ptr[S.nb]);
            fill.assign(con_ptr.begin(), con_ptr.end() - 1);
        }
        for (int l = 0; l < B.np; ++l) {
            if (B.phidx[l] < 0) continue;
            for (int a = pt_ptr[l]; a < pt_ptr[l + 1]; ++a) {
                const int r = B.chidx[socam[a]];
                if (r < 0) continue;
                for (int b = pt_ptr[l]; b < pt_ptr[l + 1]; ++b) {
                    const int c = B.chidx[socam[b]];
                    if (c < r) continue;
                    const int blk = find_block(r, c);
                    if (blk < 0) { set_error("ba_build_structure: internal error (missing Schur block)"); return S3O_ERR_INVALID; }
                    if (pass == 0) con_ptr[blk + 1]++;
                    else con[(size_t)fill[blk]++] = make_int2(a, b);
                }
            }
        }
    }
    B.ncon = con.size();
    B.pt_ptr = pt_ptr;
    B.socam = socam;
    // ---- device ---------------------------------------------------------------------------
    int rc = 0;
    rc = rc ? rc : upload_structure_arrays(p, S.nf);
    rc = rc ? rc : alloc_linear_system(p);
    rc = rc ? rc : upload(p, &B.d_chidx, B.chidx);
    rc = rc ? rc : upload(p, &B.d_phidx, B.phidx);
    rc = rc ? rc : upload(p, &B.d_ocam, socam);
    rc = rc ? rc : upload(p, &B.d_opt, sopt);
    rc = rc ? rc : upload(p, &B.d_pt_ptr, pt_ptr);
    rc = rc ? rc : upload(p, &B.d_cam_ptr, cam_ptr);
    rc = rc ? rc : upload(p, &B.d_cam_obs, cam_obs);
    rc = rc ? rc : upload(p, &B.d_con_ptr, con_ptr);
    rc = rc ? rc : dev_alloc(&B.d_con, con.size());
    if (!rc && !con.empty()) {
        S3O_CUDA(cudaMemcpyAsync(B.d_con, con.data(), con.size() * sizeof(int2), cudaMemcpyHostToDevice, p->stream));
        p->stats.h2d_bytes += (int64_t)(con.size() * sizeof(int2));
    }
    for (int w = 0; w < 2; ++w) {
        rc = rc ? rc : dev_alloc(&B.d_cam[w], (size_t)B.nc_pad * 7);
        rc = rc ? rc : dev_alloc(&B.d_pt[w], (size_t)B.np_pad * 3);
    }
    rc = rc ? rc : dev_alloc(&B.d_uv, (size_t)B.no_pad * 2);
    if (!B.info.empty()) rc = rc ? rc : dev_alloc(&B.d_info, (size_t)B.no_pad * 3);
    rc = rc ? rc : dev_alloc(&B.d_scr, (size_t)B.no_pad * kScr);
    rc = rc ? rc : dev_alloc(&B.d_Hpl, (size_t)B.no * 18);
    rc = rc ? rc : dev_alloc(&B.d_Y, (size_t)B.no * 18);
    rc = rc ? rc : dev_alloc(&B.d_Hpp, (size_t)B.ncf * 36);
    rc = rc ? rc : dev_alloc(&B.d_bp, (size_t)B.ncf * 6);
    rc = rc ? rc : dev_alloc(&B.d_Hll, (size_t)B.npf * 9);
    rc = rc ? rc : dev_alloc(&B.d_bl, (size_t)B.npf * 3);
    rc = rc ? rc : dev_alloc(&B.d_Dinv, (size_t)B.npf * 9);
    rc = rc ? rc : dev_alloc(&B.d_dl, (size_t)B.npf * 3);
    rc = rc ? rc : dev_alloc(&B.d_xl, (size_t)B.npf * 3);
    if (rc) { ba_invalidate(p); return rc; }
    for (int w = 0; w < 2; ++w) {
        cudaMemsetAsync(B.d_cam[w], 0, (size_t)B.nc_pad * 7 * sizeof(double), p->stream);
        cudaMemsetAsync(B.d_pt[w], 0, (size_t)B.np_pad * 3 * sizeof(double), p->stream);
    }
    cudaMemsetAsync(B.d_uv, 0, (size_t)B.no_pad * 2 * sizeof(double), p->stream);
    cudaMemsetAsync(B.d_xl, 0, (size_t)B.npf * 3 * sizeof(double), p->stream);     // (no free point / camera: 0 bytes)
    cudaMemsetAsync(p->d_x, 0, (size_t)S.nf * 6 * sizeof(double), p->stream);
    p->cur = 0;
    rc = rc ? rc : upload_soa(p, B.cam0, B.nc, B.nc_pad, 7, B.d_cam[0]);
    rc = rc ? rc : upload_soa(p, B.pt0, B.np, B.np_pad, 3, B.d_pt[0]);
    rc = rc ? rc : upload_soa(p, suv, B.no, B.no_pad, 2, B.d_uv);
    if (!B.info.empty()) rc = rc ? rc : upload_soa(p, sinfo, B.no, B.no_pad, 3, B.d_info);
    if (rc) { ba_invalidate(p); return rc; }
    S3O_CUDA(cudaStreamSynchronize(p->stream));
    p->built = true;
    p->stats.n_free = S.nf; p->stats.n_blocks = S.nb;
    return S3O_OK;
}

int ba_chi2(s3o_problem *p, int which) {
    BaState &B = *p->ba;
    if (B.no == 0) { S3O_CUDA(cudaMemsetAsync(&p->d_sc->chi2, 0, sizeof(double), p->stream)); return S3O_OK; }
    constexpr int NT = 128;
    ba_chi2_kernel<NT><<<grid_cap(B.no, NT), NT, 0, p->stream>>>(ba_view(p, which), p->d_partials, p->d_sc);
    return check_launch(p, 1);
}

int ba_linearize(s3o_problem *p) {
    BaState &B = *p->ba;
    const BaDev g = ba_view(p, p->cur);
    if (B.no > 0) ba_linearize_kernel<<<(B.no + 127) / 128, 128, 0, p->stream>>>(g, B.d_scr, B.d_Hpl);
    ba_assemble_points_kernel<<<(B.np + 127) / 128, 128, 0, p->stream>>>(g, B.d_pt_ptr, B.d_scr, B.d_Hll, B.d_bl);
    ba_assemble_cameras_kernel<<<B.nc, 27 * kCamGroups, 0, p->stream>>>(g, B.d_cam_ptr, B.d_cam_obs, B.d_scr, B.d_Hpp, B.d_bp);
    p->linearized = true;
    return check_launch(p, 3);
}

int ba_max_diag(s3o_problem *p) {
    BaState &B = *p->ba;
    constexpr int NT = 256;
    ba_maxdiag_kernel<NT><<<grid_cap((long long)B.ncf * 6 + (long long)B.npf * 3, NT), NT, 0, p->stream>>>(
        B.d_Hpp, B.ncf, B.d_Hll, B.npf, p->d_partials, p->d_sc);
    return check_launch(p, 1);
}

// Forms the damped Schur system in p->d_H / p->d_b (launches only)
int ba_form_schur(s3o_problem *p, double lambda) {
    BaState &B = *p->ba;
    const BaDev g = ba_view(p, p->cur);
    if (B.npf > 0) ba_point_inverse_kernel<<<(B.npf + 127) / 128, 128, 0, p->stream>>>(B.npf, B.d_Hll, B.d_bl, lambda, B.d_Dinv, B.d_dl, p->d_sc);
    if (B.no > 0) ba_y_kernel<<<(B.no + 127) / 128, 128, 0, p->stream>>>(g, B.d_Hpl, B.d_Dinv, B.d_Y);
    const long long tot = (long long)p->S.nb * 36;
    if (tot > 0)
        ba_schur_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, p->stream>>>(p->S.nb, p->d_blk_row, p->d_colidx, B.d_con_ptr, B.d_con,
                                                                            B.d_Y, B.d_Hpl, B.d_Hpp, lambda, p->d_H);
    ba_schur_rhs_kernel<<<B.nc, 6 * kBsGroups, 0, p->stream>>>(g, B.d_cam_ptr, B.d_cam_obs, B.d_Hpl, B.d_dl, B.d_bp, p->d_b);
    return check_launch(p, 4);
}

int ba_solve(s3o_problem *p, double lambda, int *status, int *iters, double *rel_res) {
    BaState &B = *p->ba;
    int rc = ba_form_schur(p, lambda);
    if (rc) return rc;
    if ((rc = do_solve(p, 0.0, status, iters, rel_res))) return rc;       // lambda is inside S
    ba_backsub_kernel<<<(B.np + 127) / 128, 128, 0, p->stream>>>(ba_view(p, p->cur), B.d_pt_ptr, B.d_Hpl, B.d_Dinv, B.d_dl, p->d_x, B.d_xl);
    return check_launch(p, 1);
}

int ba_retract_and_scale(s3o_problem *p, double lambda, int trial) {
    BaState &B = *p->ba;
    const int n = std::max(B.nc, B.np);
    ba_retract_kernel<<<(n + 127) / 128, 128, 0, p->stream>>>(ba_view(p, p->cur), p->d_x, B.d_xl, B.d_cam[trial], B.d_pt[trial]);
    constexpr int NT = 256;
    ba_scale_kernel<NT><<<grid_cap((long long)B.ncf * 6 + (long long)B.npf * 3, NT), NT, 0, p->stream>>>(
        B.ncf * 6, p->d_x, B.d_bp, B.npf * 3, B.d_xl, B.d_bl, lambda, p->d_partials, p->d_sc);
    return check_launch(p, 2);
}

int ba_upload_step(s3o_problem *p, const double *x) {
    BaState &B = *p->ba;
    S3O_CUDA(cudaMemcpyAsync(p->d_x, x, (size_t)B.ncf * 6 * sizeof(double), cudaMemcpyHostToDevice, p->stream));
    S3O_CUDA(cudaMemcpyAsync(B.d_xl, x + (size_t)B.ncf * 6, (size_t)B.npf * 3 * sizeof(double), cudaMemcpyHostToDevice, p->stream));
    p->stats.h2d_bytes += (int64_t)(B.ncf * 6 + B.npf * 3) * 8;
    return S3O_OK;
}

int ba_download_step(s3o_problem *p, double *x) {
    BaState &B = *p->ba;
    S3O_CUDA(cudaMemcpyAsync(x, p->d_x, (size_t)B.ncf * 6 * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    S3O_CUDA(cudaMemcpyAsync(x + (size_t)B.ncf * 6, B.d_xl, (size_t)B.npf * 3 * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    S3O_CUDA(cudaStreamSynchronize(p->stream));
    p->stats.d2h_bytes += (int64_t)(B.ncf * 6 + B.npf * 3) * 8;
    return S3O_OK;
}

// device-side copy of the current cameras and points (restore = 0) or its restore (restore = 1)
int ba_snapshot(s3o_problem *p, int restore) {
    BaState &B = *p->ba;
    const size_t cb = (size_t)B.nc_pad * 7 * sizeof(double), pb = (size_t)B.np_pad * 3 * sizeof(double);
    if (!restore) {
        int rc = 0;
        if (!B.d_cam_snap) rc = dev_alloc(&B.d_cam_snap, (size_t)B.nc_pad * 7);
        if (!rc && !B.d_pt_snap) rc = dev_alloc(&B.d_pt_snap, (size_t)B.np_pad * 3);
        if (rc) return rc;
        S3O_CUDA(cudaMemcpyAsync(B.d_cam_snap, B.d_cam[p->cur], cb, cudaMemcpyDeviceToDevice, p->stream));
        S3O_CUDA(cudaMemcpyAsync(B.d_pt_snap, B.d_pt[p->cur], pb, cudaMemcpyDeviceToDevice, p->stream));
        return S3O_OK;
    }
    if (!B.d_cam_snap || !B.d_pt_snap) { set_error("s3o_restore_estimates: no snapshot"); return S3O_ERR_INVALID; }
    S3O_CUDA(cudaMemcpyAsync(B.d_cam[p->cur], B.d_cam_snap, cb, cudaMemcpyDeviceToDevice, p->stream));
    S3O_CUDA(cudaMemcpyAsync(B.d_pt[p->cur], B.d_pt_snap, pb, cudaMemcpyDeviceToDevice, p->stream));
    return S3O_OK;
}

namespace {

// Host checks of s3o_ba_compute_marginals, once per structure (B.marg_check / B.marg_msg).  H is singular when
//  - a connected component of the camera-point observation graph holding a free vertex fixes neither a camera and one
//    more vertex nor three points: the monocular 7-DoF gauge (scale included) is free;
//  - a free point is seen by fewer than two distinct cameras: its Hll has rank <= 2.
int ba_marginal_checks(BaState &B) {
    if (B.marg_check >= 0) {
        if (B.marg_check) set_error("%s", B.marg_msg.c_str());
        return B.marg_check;
    }
    char msg[256] = "";
    const int nv = B.nc + B.np;
    std::vector<int32_t> root(nv);
    for (int v = 0; v < nv; ++v) root[v] = v;
    auto find = [&](int v) { while (root[v] != v) v = root[v] = root[root[v]]; return v; };
    for (int k = 0; k < B.no; ++k) {
        const int a = find(B.ocam[k]), b = find(B.nc + B.opt[k]);
        if (a != b) root[std::max(a, b)] = std::min(a, b);
    }
    std::vector<int32_t> fcam(nv, 0), fpt(nv, 0);
    for (int c = 0; c < B.nc; ++c) if (B.cfix[c]) fcam[find(c)]++;
    for (int l = 0; l < B.np; ++l) if (B.pfix[l]) fpt[find(B.nc + l)]++;
    for (int v = 0; v < nv && !msg[0]; ++v) {
        const bool is_cam = v < B.nc;
        if (is_cam ? B.cfix[v] : B.pfix[v - B.nc]) continue;
        const int r = find(v);
        if ((fcam[r] >= 1 && fcam[r] + fpt[r] >= 2) || fpt[r] >= 3) continue;
        snprintf(msg, sizeof msg, "s3o_ba_compute_marginals: the Hessian is singular: the connected component of %s %d "
                 "fixes %d camera(s) and %d point(s), not a camera and one more vertex or three points (its 7-DoF gauge is free)",
                 is_cam ? "camera" : "point", is_cam ? v : v - B.nc, fcam[r], fpt[r]);
    }
    std::vector<int32_t> cams;
    for (int l = 0; l < B.np && !msg[0]; ++l) {
        if (B.pfix[l]) continue;
        cams.assign(B.socam.begin() + B.pt_ptr[l], B.socam.begin() + B.pt_ptr[l + 1]);
        std::sort(cams.begin(), cams.end());
        const int distinct = (int)(std::unique(cams.begin(), cams.end()) - cams.begin());
        if (distinct < 2)
            snprintf(msg, sizeof msg, "s3o_ba_compute_marginals: the Hessian is singular: free point %d is seen by %d distinct "
                     "camera(s); a free point needs two", l, distinct);
    }
    B.marg_msg = msg;
    B.marg_check = msg[0] ? S3O_ERR_SOLVE : S3O_OK;
    if (B.marg_check) set_error("%s", msg);
    return B.marg_check;
}

// Point gather lists on the plan of the selected inverse (plan == nullptr: no free camera, empty lists), in point
// order, then a-major over the point's free-camera observations: mo_ptr / mo_obs / mp_ptr / mp_sig of
// ba_marginal_points_kernel.  Every pair of cameras co-observing a free point is a block of S, hence of L.
int ba_marginal_lists(s3o_problem *p, BaState &B, const DirectPlan *plan, uint64_t serial) {
    if (B.marg_lists && B.marg_serial == serial) return S3O_OK;
    dev_free(B.d_mo_ptr); dev_free(B.d_mo_obs); dev_free(B.d_mp_sig); dev_free(B.d_mp_ptr);
    B.marg_lists = false;
    std::vector<int32_t> ipos(plan ? plan->n : 0);
    for (int k = 0; plan && k < plan->n; ++k) ipos[plan->perm[k]] = k;
    std::vector<int32_t> mo_ptr(B.npf + 1, 0), mo_obs, mp_sig, pos;
    std::vector<int64_t> mp_ptr(B.npf + 1, 0);
    for (int l = 0; l < B.np; ++l) {
        const int li = B.phidx[l];
        if (li < 0) continue;
        pos.clear();
        for (int t = B.pt_ptr[l]; t < B.pt_ptr[l + 1]; ++t) {
            const int ci = B.chidx[B.socam[t]];
            if (ci < 0) continue;
            mo_obs.push_back(t);
            pos.push_back(ipos[ci]);
        }
        const int nO = (int)pos.size();
        mo_ptr[li + 1] = (int32_t)mo_obs.size();
        mp_ptr[li + 1] = mp_ptr[li] + (int64_t)nO * nO;
        const size_t base = mp_sig.size();
        mp_sig.resize(base + (size_t)nO * nO);
        for (int a = 0; a < nO; ++a)
            for (int b = 0; b <= a; ++b) {
                const int32_t t = direct_find_block(*plan, std::min(pos[a], pos[b]), std::max(pos[a], pos[b]));
                if (t < 0) { set_error("s3o_ba_compute_marginals: internal error (co-observing cameras without a block of L)"); return S3O_ERR_INVALID; }
                mp_sig[base + (size_t)a * nO + b] = (t << 1) | (pos[a] < pos[b] ? 1 : 0);
                mp_sig[base + (size_t)b * nO + a] = (t << 1) | (pos[b] < pos[a] ? 1 : 0);
            }
    }
    int rc = upload(p, &B.d_mo_ptr, mo_ptr);
    rc = rc ? rc : upload(p, &B.d_mo_obs, mo_obs);
    rc = rc ? rc : upload(p, &B.d_mp_ptr, mp_ptr);
    rc = rc ? rc : upload(p, &B.d_mp_sig, mp_sig);
    if (!rc && cudaStreamSynchronize(p->stream) != cudaSuccess) rc = S3O_ERR_CUDA;
    if (rc) { set_error("s3o_ba_compute_marginals: device allocation failed"); return rc; }
    B.marg_lists = true;
    B.marg_serial = serial;
    return S3O_OK;
}

// device buffer of at least `need` elements (kept between calls)
template <class T>
int ensure_cap(T **ptr, size_t *cap, size_t need) {
    if (*ptr && need <= *cap) return S3O_OK;
    dev_free(*ptr);
    *cap = 0;
    const int rc = dev_alloc(ptr, need);
    if (!rc) *cap = need;
    return rc;
}

template <class T>
int h2d(s3o_problem *p, T *dst, const std::vector<T> &v) {
    if (v.empty()) return S3O_OK;
    S3O_CUDA(cudaMemcpyAsync(dst, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, p->stream));
    p->stats.h2d_bytes += (int64_t)(v.size() * sizeof(T));
    return S3O_OK;
}

}  // namespace

}  // namespace s3o

// ======================================================================================
// BA-specific C ABI
// ======================================================================================
using namespace s3o;

extern "C" {

int s3o_ba_set_cameras(s3o_problem *p, int n, const double *est, const uint8_t *fixed) {
    if (!p || p->kind != S3O_KIND_BA || n < 0 || (n > 0 && !est)) { set_error("s3o_ba_set_cameras: bad arguments (kind must be S3O_KIND_BA)"); return S3O_ERR_INVALID; }
    cudaSetDevice(p->device);
    BaState &B = *ba_state(p);
    ba_invalidate(p);
    B.nc = n;
    B.cam0.assign(est, est + (size_t)n * 7);
    B.cfix.assign(n, 0);
    if (fixed) memcpy(B.cfix.data(), fixed, n);
    B.ocam.clear(); B.opt.clear(); B.uv.clear(); B.info.clear(); B.no = 0;
    p->lm_valid = false;
    return S3O_OK;
}

int s3o_ba_set_points(s3o_problem *p, int n, const double *xyz, const uint8_t *fixed) {
    if (!p || p->kind != S3O_KIND_BA || n < 0 || (n > 0 && !xyz)) { set_error("s3o_ba_set_points: bad arguments (kind must be S3O_KIND_BA)"); return S3O_ERR_INVALID; }
    cudaSetDevice(p->device);
    BaState &B = *ba_state(p);
    ba_invalidate(p);
    B.np = n;
    B.pt0.assign(xyz, xyz + (size_t)n * 3);
    B.pfix.assign(n, 0);
    if (fixed) memcpy(B.pfix.data(), fixed, n);
    B.ocam.clear(); B.opt.clear(); B.uv.clear(); B.info.clear(); B.no = 0;
    p->lm_valid = false;
    return S3O_OK;
}

int s3o_ba_set_observations(s3o_problem *p, int n, const int32_t *cam_idx, const int32_t *point_idx, const double *uv,
                            const double *info) {
    if (!p || p->kind != S3O_KIND_BA || n < 0 || (n > 0 && (!cam_idx || !point_idx || !uv))) { set_error("s3o_ba_set_observations: bad arguments"); return S3O_ERR_INVALID; }
    BaState &B = *ba_state(p);
    for (int k = 0; k < n; ++k)
        if (cam_idx[k] < 0 || cam_idx[k] >= B.nc || point_idx[k] < 0 || point_idx[k] >= B.np) {
            set_error("s3o_ba_set_observations: observation %d refers to camera %d / point %d (have %d / %d)", k, cam_idx[k], point_idx[k], B.nc, B.np);
            return S3O_ERR_INVALID;
        }
    cudaSetDevice(p->device);
    ba_invalidate(p);
    B.no = n;
    B.ocam.assign(cam_idx, cam_idx + n);
    B.opt.assign(point_idx, point_idx + n);
    B.uv.assign(uv, uv + (size_t)n * 2);
    if (info) B.info.assign(info, info + (size_t)n * 3); else B.info.clear();
    p->stats.n_edges = n;
    return S3O_OK;
}

int s3o_ba_set_intrinsics(s3o_problem *p, double focal, double cx, double cy) {
    if (!p || p->kind != S3O_KIND_BA) { set_error("s3o_ba_set_intrinsics: kind must be S3O_KIND_BA"); return S3O_ERR_INVALID; }
    BaState &B = *ba_state(p);
    B.f = focal; B.cx = cx; B.cy = cy;
    p->linearized = false;
    return S3O_OK;
}

// overwrite the current estimates (either pointer may be NULL to keep that part); structure is kept
int s3o_ba_set_estimates(s3o_problem *p, const double *cams, const double *points) {
    if (!p || p->kind != S3O_KIND_BA || !p->ba) { set_error("s3o_ba_set_estimates: no BA graph"); return S3O_ERR_INVALID; }
    cudaSetDevice(p->device);
    BaState &B = *p->ba;
    if (cams) B.cam0.assign(cams, cams + (size_t)B.nc * 7);
    if (points) B.pt0.assign(points, points + (size_t)B.np * 3);
    p->linearized = false;
    if (p->lm_resume != 2) p->lm_valid = false;
    if (!p->built) return S3O_OK;
    int rc = 0;
    if (cams) rc = upload_soa(p, B.cam0, B.nc, B.nc_pad, 7, B.d_cam[p->cur]);
    if (!rc && points) rc = upload_soa(p, B.pt0, B.np, B.np_pad, 3, B.d_pt[p->cur]);
    return rc;
}

static int ba_download(s3o_problem *p, const double *soa, int n, int n_pad, int dim, double *out) {
    if (n == 0) return S3O_OK;
    double *tmp = nullptr;
    int rc = dev_alloc(&tmp, (size_t)n * dim);
    if (rc) return rc;
    ba_unpack_kernel<<<(n * dim + 255) / 256, 256, 0, p->stream>>>(soa, n, n_pad, dim, tmp);
    cudaError_t e = cudaMemcpyAsync(out, tmp, (size_t)n * dim * sizeof(double), cudaMemcpyDeviceToHost, p->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(p->stream);
    cudaFree(tmp);
    if (e != cudaSuccess) { set_error("ba download: %s", cudaGetErrorString(e)); return S3O_ERR_CUDA; }
    p->stats.d2h_bytes += (int64_t)n * dim * 8;
    p->stats.kernel_launches += 1;
    return S3O_OK;
}

int s3o_ba_get_cameras(s3o_problem *p, double *est) {
    if (!p || p->kind != S3O_KIND_BA || !p->ba || !est) { set_error("s3o_ba_get_cameras: no BA graph"); return S3O_ERR_INVALID; }
    cudaSetDevice(p->device);
    BaState &B = *p->ba;
    if (!p->built) { memcpy(est, B.cam0.data(), B.cam0.size() * sizeof(double)); return S3O_OK; }
    return ba_download(p, B.d_cam[p->cur], B.nc, B.nc_pad, 7, est);
}

int s3o_ba_get_points(s3o_problem *p, double *xyz) {
    if (!p || p->kind != S3O_KIND_BA || !p->ba || !xyz) { set_error("s3o_ba_get_points: no BA graph"); return S3O_ERR_INVALID; }
    cudaSetDevice(p->device);
    BaState &B = *p->ba;
    if (!p->built) { memcpy(xyz, B.pt0.data(), B.pt0.size() * sizeof(double)); return S3O_OK; }
    return ba_download(p, B.d_pt[p->cur], B.np, B.np_pad, 3, xyz);
}

int s3o_ba_get_sizes(s3o_problem *p, int *n_free_cameras, int *n_free_points, int *n_schur_blocks, int64_t *n_contributions) {
    if (!p || p->kind != S3O_KIND_BA || !p->ba || !p->built) { set_error("s3o_ba_get_sizes: structure not built"); return S3O_ERR_INVALID; }
    if (n_free_cameras) *n_free_cameras = p->ba->ncf;
    if (n_free_points) *n_free_points = p->ba->npf;
    if (n_schur_blocks) *n_schur_blocks = p->S.nb;
    if (n_contributions) *n_contributions = (int64_t)p->ba->ncon;
    return S3O_OK;
}

// lock-step read-outs (caller's observation order for Hpl and errors)
int s3o_ba_edge_errors(s3o_problem *p, double *err) {
    if (!p || p->kind != S3O_KIND_BA || !err) return S3O_ERR_INVALID;
    cudaSetDevice(p->device);
    int rc = p->built ? S3O_OK : s3o_build_structure(p, nullptr, nullptr);
    if (rc) return rc;
    BaState &B = *p->ba;
    double *d_err = nullptr;
    if ((rc = dev_alloc(&d_err, (size_t)B.no * 2))) return rc;
    if (B.no > 0) ba_edge_errors_kernel<<<(B.no + 127) / 128, 128, 0, p->stream>>>(ba_view(p, p->cur), d_err);
    std::vector<double> tmp((size_t)B.no * 2);
    cudaError_t e = cudaMemcpyAsync(tmp.data(), d_err, tmp.size() * sizeof(double), cudaMemcpyDeviceToHost, p->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(p->stream);
    cudaFree(d_err);
    if (e != cudaSuccess) { set_error("s3o_ba_edge_errors: %s", cudaGetErrorString(e)); return S3O_ERR_CUDA; }
    for (int t = 0; t < B.no; ++t) { err[(size_t)B.perm[t] * 2] = tmp[(size_t)t * 2]; err[(size_t)B.perm[t] * 2 + 1] = tmp[(size_t)t * 2 + 1]; }
    p->stats.kernel_launches += 1;
    return S3O_OK;
}

int s3o_ba_get_system(s3o_problem *p, double *Hpp, double *Hll, double *Hpl, double *b) {
    if (!p || p->kind != S3O_KIND_BA || !p->built || !p->linearized) { set_error("s3o_ba_get_system: call s3o_linearize first"); return S3O_ERR_INVALID; }
    cudaSetDevice(p->device);
    BaState &B = *p->ba;
    if (Hpp) S3O_CUDA(cudaMemcpyAsync(Hpp, B.d_Hpp, (size_t)B.ncf * 36 * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    if (Hll) S3O_CUDA(cudaMemcpyAsync(Hll, B.d_Hll, (size_t)B.npf * 9 * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    if (b) {
        S3O_CUDA(cudaMemcpyAsync(b, B.d_bp, (size_t)B.ncf * 6 * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
        S3O_CUDA(cudaMemcpyAsync(b + (size_t)B.ncf * 6, B.d_bl, (size_t)B.npf * 3 * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    }
    std::vector<double> tmp;
    if (Hpl) {
        tmp.resize((size_t)B.no * 18);
        S3O_CUDA(cudaMemcpyAsync(tmp.data(), B.d_Hpl, tmp.size() * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    }
    S3O_CUDA(cudaStreamSynchronize(p->stream));
    if (Hpl) for (int t = 0; t < B.no; ++t) memcpy(Hpl + (size_t)B.perm[t] * 18, tmp.data() + (size_t)t * 18, 18 * sizeof(double));
    return S3O_OK;
}

// damped Schur complement: blocks in the g2o CCS order of s3o_get_structure, bs: 6 * n_free_cameras
int s3o_ba_get_schur(s3o_problem *p, double lambda, double *blocks, double *bs) {
    if (!p || p->kind != S3O_KIND_BA || !p->built || !p->linearized) { set_error("s3o_ba_get_schur: call s3o_linearize first"); return S3O_ERR_INVALID; }
    cudaSetDevice(p->device);
    int rc = ba_form_schur(p, lambda);
    if (rc) return rc;
    if (blocks) {
        std::vector<double> tmp((size_t)p->S.nb * 36);
        S3O_CUDA(cudaMemcpyAsync(tmp.data(), p->d_H, tmp.size() * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
        S3O_CUDA(cudaStreamSynchronize(p->stream));
        for (int c = 0; c < p->S.nb; ++c) memcpy(blocks + (size_t)c * 36, tmp.data() + (size_t)p->S.ccs2bsr[c] * 36, 36 * sizeof(double));
    }
    if (bs) {
        S3O_CUDA(cudaMemcpyAsync(bs, p->d_b, (size_t)p->S.nf * 6 * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
        S3O_CUDA(cudaStreamSynchronize(p->stream));
    }
    return S3O_OK;
}

// Marginal covariances of bundle adjustment: blocks of H^-1 for the undamped H = [[Hpp, Hpl], [Hpl^T, Hll]] at the
// current estimates, from the selected inverse of the Schur complement (direct.cu) and the point phase above.
int s3o_ba_compute_marginals(s3o_problem *p, int n_pairs, const int32_t *rows, const int32_t *cols, double *out) {
    if (!p || p->kind != S3O_KIND_BA || n_pairs < 0 || (!rows != !cols) || (n_pairs > 0 && !out)) {
        set_error("s3o_ba_compute_marginals: bad arguments (the problem must be of kind S3O_KIND_BA)");
        return S3O_ERR_INVALID;
    }
    if (p->dist) { set_error("s3o_ba_compute_marginals: not available with the partitioned solve"); return S3O_ERR_UNSUPPORTED; }
    cudaSetDevice(p->device);
    int rc = p->built ? S3O_OK : s3o_build_structure(p, nullptr, nullptr);
    if (rc) return rc;
    BaState &B = *p->ba;
    const int ncf = B.ncf, npf = B.npf, n = ncf + npf;
    if (n == 0) { set_error("s3o_ba_compute_marginals: 0 free vertices"); return S3O_ERR_INVALID; }
    if (!rows && n_pairs != n) { set_error("s3o_ba_compute_marginals: the diagonal blocks need n_pairs = n_free_cameras + n_free_points = %d", n); return S3O_ERR_INVALID; }
    for (int k = 0; rows && k < n_pairs; ++k)
        if (rows[k] < 0 || rows[k] >= n || cols[k] < 0 || cols[k] >= n) {
            set_error("s3o_ba_compute_marginals: pair %d (%d, %d) is not a pair of Hessian indices in [0, %d) (fixed vertices have none)",
                      k, rows[k], cols[k], n);
            return S3O_ERR_INVALID;
        }
    // ---- the requested pairs: camera-camera to the selected inverse, the rest to the point phase
    std::vector<int32_t> src(n_pairs), cc_r, cc_c, rq, rq_slot, pid;
    std::vector<int64_t> dst(n_pairs);
    std::map<std::pair<int32_t, int32_t>, int32_t> cl;        // (point slot, observation a) -> camera-point slot
    std::vector<std::pair<int32_t, int32_t>> pair_cl(n_pairs);
    int64_t total = 0;
    if (rows) rq_slot.assign(npf, -1);
    auto point_slot = [&](int li) {
        if (rq_slot[li] < 0) { rq_slot[li] = (int32_t)rq.size(); rq.push_back(li); }
        return rq_slot[li];
    };
    for (int k = 0; k < n_pairs; ++k) {
        const int r = rows ? rows[k] : k, c = cols ? cols[k] : k;
        const bool rc_cam = r < ncf, cc_cam = c < ncf;
        dst[k] = total;
        total += (rc_cam ? 6 : 3) * (cc_cam ? 6 : 3);
        if (!rows) { src[k] = k < ncf ? (k << 2) : ((k - ncf) << 2) | 1; continue; }
        if (rc_cam && cc_cam) {
            src[k] = ((int32_t)cc_r.size() << 2);
            cc_r.push_back(r); cc_c.push_back(c);
        } else if (!rc_cam && !cc_cam) {
            if (r != c) { set_error("s3o_ba_compute_marginals: pair %d (%d, %d) joins two distinct points (not supported)", k, r, c); return S3O_ERR_UNSUPPORTED; }
            src[k] = (point_slot(r - ncf) << 2) | 1;
        } else {
            const int ci = rc_cam ? r : c, li = (rc_cam ? c : r) - ncf;
            if (pid.empty()) {
                pid.resize(npf);
                for (int q = 0; q < B.np; ++q) if (B.phidx[q] >= 0) pid[B.phidx[q]] = q;
            }
            const int l = pid[li];
            int a = -1;
            for (int t = B.pt_ptr[l], m = 0; t < B.pt_ptr[l + 1] && a < 0; ++t) {
                const int cf = B.chidx[B.socam[t]];
                if (cf == ci) a = m;
                if (cf >= 0) ++m;
            }
            if (a < 0) {
                set_error("s3o_ba_compute_marginals: pair %d (%d, %d): camera %d does not observe point %d (not supported)", k, r, c, ci, li + ncf);
                return S3O_ERR_UNSUPPORTED;
            }
            pair_cl[k] = { point_slot(li), a };
            cl.emplace(pair_cl[k], 0);
            src[k] = rc_cam ? 2 : 3;
        }
    }
    if ((rc = ba_marginal_checks(B))) return rc;
    // camera-point slots grouped by point slot
    const int nrq = rows ? (int)rq.size() : npf;
    std::vector<int32_t> cl_ptr, cl_a;
    if (!cl.empty()) {
        cl_ptr.assign(nrq + 1, 0);
        for (auto &kv : cl) { kv.second = (int32_t)cl_a.size(); cl_a.push_back(kv.first.second); cl_ptr[kv.first.first + 1]++; }
        for (int s = 0; s < nrq; ++s) cl_ptr[s + 1] += cl_ptr[s];
        for (int k = 0; k < n_pairs; ++k)
            if ((src[k] & 3) >= 2) src[k] |= cl.at(pair_cl[k]) << 2;
    }
    // ---- plan, lists and buffers (host work and uploads, before anything runs)
    MarginalsRun R;
    const int n_cc = rows ? (int)cc_r.size() : ncf;
    if (ncf > 0 && (rc = marginals_open(p, "s3o_ba_compute_marginals", n_cc, rows ? cc_r.data() : nullptr,
                                        rows ? cc_c.data() : nullptr, &R)))
        return rc;
    if ((rc = ba_marginal_lists(p, B, ncf > 0 ? R.plan : nullptr, R.serial))) return rc;
    rc = ensure_cap(&B.d_msrc, &B.cap_msrc, (size_t)n_pairs);
    rc = rc ? rc : ensure_cap(&B.d_mdst, &B.cap_mdst, (size_t)n_pairs);
    rc = rc ? rc : ensure_cap(&B.d_mpt, &B.cap_mpt, (size_t)nrq * 9 + cl_a.size() * 18);
    rc = rc ? rc : ensure_cap(&B.d_mout, &B.cap_mout, (size_t)total);
    if (!rc && !B.d_mflag) rc = dev_alloc(&B.d_mflag, 2);
    if (!rc && rows) rc = ensure_cap(&B.d_mrq, &B.cap_mrq, rq.size());
    if (!rc && !cl_a.empty()) rc = ensure_cap(&B.d_mcl_ptr, &B.cap_mcl_ptr, cl_ptr.size());
    if (!rc && !cl_a.empty()) rc = ensure_cap(&B.d_mcl_a, &B.cap_mcl_a, cl_a.size());
    if (rc) { set_error("s3o_ba_compute_marginals: device allocation failed"); return rc; }
    if ((rc = h2d(p, B.d_msrc, src)) || (rc = h2d(p, B.d_mdst, dst)) || (rc = h2d(p, B.d_mrq, rq)) ||
        (rc = h2d(p, B.d_mcl_ptr, cl_ptr)) || (rc = h2d(p, B.d_mcl_a, cl_a)))
        return rc;
    S3O_CUDA(cudaMemsetAsync(B.d_mflag, 0, 2 * sizeof(int), p->stream));
    // ---- linearize | Schur (lambda = 0) | factor | selected inverse | points | gather
    cudaEvent_t *ev = p->ev;
    cudaEventRecord(ev[0], p->stream);
    if ((rc = ba_linearize(p))) return rc;
    cudaEventRecord(ev[1], p->stream);
    rc = ba_form_schur(p, 0.0);
    p->linearized = false;          // p->d_b holds the undamped Schur right-hand side: the next solve linearises again
    direct_invalidate(p);
    if (rc) return rc;
    cudaEventRecord(ev[2], p->stream);
    if (ncf > 0) {
        if ((rc = marginals_factor(p, R, ev + 3))) return rc;
    } else {
        cudaEventRecord(ev[3], p->stream);
        cudaEventRecord(ev[4], p->stream);
    }
    int launches = 1;
    if (npf > 0) {
        const int grid = (int)std::max<long long>(1, std::min<long long>(148 * 8, ((long long)std::max(nrq, npf) * 32 + kMargNT - 1) / kMargNT));
        ba_marginal_points_kernel<<<grid, kMargNT, 0, p->stream>>>(
            npf, nrq, rows ? B.d_mrq : nullptr, B.d_mo_ptr, B.d_mo_obs, B.d_mp_ptr, B.d_mp_sig, ncf > 0 ? R.Sig : nullptr,
            B.d_Y, B.d_Dinv, B.d_Hll, cl_a.empty() ? nullptr : B.d_mcl_ptr, B.d_mcl_a, B.d_mpt, B.d_mpt + (size_t)nrq * 9, B.d_mflag);
        ++launches;
    }
    cudaEventRecord(ev[5], p->stream);
    if (ncf > 0 && (rc = marginals_pick(p, R, n_cc))) return rc;
    if (n_pairs > 0)
        ba_marginal_gather_kernel<<<(int)std::min<long long>(1024, ((long long)n_pairs * 36 + 255) / 256), 256, 0, p->stream>>>(
            n_pairs, B.d_msrc, B.d_mdst, ncf > 0 ? R.out : nullptr, B.d_mpt, B.d_mpt + (size_t)nrq * 9, ncf > 0 ? R.fail : nullptr,
            B.d_mflag, B.d_mout);
    cudaEventRecord(ev[6], p->stream);
    if ((rc = check_launch(p, launches))) return rc;
    int flag[2] = { 0, 0 };
    if (total > 0) S3O_CUDA(cudaMemcpyAsync(out, B.d_mout, sizeof(double) * total, cudaMemcpyDeviceToHost, p->stream));
    S3O_CUDA(cudaMemcpyAsync(flag, B.d_mflag, sizeof flag, cudaMemcpyDeviceToHost, p->stream));
    S3O_CUDA(cudaStreamSynchronize(p->stream));
    p->stats.d2h_bytes += total * 8 + (int64_t)sizeof flag;
    if (flag[1]) { set_error("s3o_ba_compute_marginals: the Schur complement is not positive definite (a pivot of its factorisation failed)"); return S3O_ERR_SOLVE; }
    if (flag[0]) { set_error("s3o_ba_compute_marginals: a free point's Hll is not positive definite (det <= 0 or not finite)"); return S3O_ERR_SOLVE; }
    if (getenv("S3O_MARGINALS_TRACE")) {     // per-phase CUDA-event times (tools/marginals_probe.py --ba)
        float ms[6] = {};
        for (int k = 0; k < 6; ++k) cudaEventElapsedTime(&ms[k], ev[k], ev[k + 1]);
        fprintf(stderr, "s3o_ba_compute_marginals: linearize %.4f schur %.4f factor %.4f selinv %.4f points %.4f gather %.4f ms\n",
                ms[0], ms[1], ms[2], ms[3], ms[4], ms[5]);
    }
    return S3O_OK;
}

}  // extern "C"
