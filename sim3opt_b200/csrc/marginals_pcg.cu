// marginals_pcg.cu -- marginal covariances beyond the sparse Cholesky's cap: requested block columns of H^-1 by PCG.
//
// For each distinct column vertex c of the requested pairs, d solves H x = e_(c,m) (m = 0..d-1) without damping run
// through the LM's own PCG (pcg_prepare / pcg_iterate: symmetric BSR SpMV, fused vector update, multilevel K-cycle),
// one right-hand side at a time, with the route's own tolerance and iteration cap.  After every solve the true
// residual r = e - H x is formed from one product at lambda = 0 and, while it is above the tolerance, a correction
// H d = r is solved and added (iterative refinement: the recurrence residual of the PCG drifts from the true one at
// tight tolerances).  Component m of every requested block of column c is written straight into the output; no
// n x d column buffer is held.  All reductions are in fixed order: bitwise reproducible.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

#include "problem.h"
#include "reduce.cuh"

namespace s3o {

namespace {

constexpr int kMargMaxIter = 20000;     // PCG iterations per right-hand side, refinement included
constexpr int kMargMaxRounds = 4;       // correction solves after the first
// Where fp64 cannot resolve S3O_MARGINALS_PCG_TOL (the residual's rounding floor ~ eps |H| |x| is above it on graphs
// with kappa(H) ~ 1e12), refinement stops once a round no longer halves the residual, and the result is accepted if
// its normwise backward error |e - H x| / (|H|_F |x|) is at most kMargBackTol.
constexpr double kMargBackTol = 1e-13;
constexpr int kNT = 256;

int grid_for(long long n) { return (int)std::max<long long>(1, std::min<long long>(kMaxPartials, (n + kNT - 1) / kNT)); }

__global__ void marg_unit_rhs_kernel(double *__restrict__ b, int n, int idx) {
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < n; t += gridDim.x * blockDim.x) b[t] = t == idx ? 1.0 : 0.0;
}

// r = e_idx - H x from the SpMV's row products q1 and transposed products T (the column owner adds its T entries in
// the fixed order of finish_q); r into b, per-CTA sums of r^2 and x^2 into partials[0, grid) and [kMaxPartials, ..)
template <int D>
__global__ void __launch_bounds__(kNT) marg_residual_kernel(StructDev s, int nf, const double *__restrict__ q1,
                                                            const double *__restrict__ T, const double *__restrict__ x,
                                                            int idx, double *__restrict__ r, double *__restrict__ partials) {
    __shared__ double sh[32];
    double acc = 0, xx = 0;
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < nf * D; t += gridDim.x * blockDim.x) {
        const int i = t / D, l = t - i * D;
        double q = q1[t];
        for (int n = s.colT_ptr[i]; n < s.colT_ptr[i + 1]; ++n) q += T[(size_t)s.colT_blk[n] * D + l];
        const double v = (t == idx ? 1.0 : 0.0) - q;
        r[t] = v;
        acc += v * v;
        xx += x[t] * x[t];
    }
    const double b1 = block_sum<kNT>(acc, sh);
    const double b2 = block_sum<kNT>(xx, sh);
    if (threadIdx.x == 0) { partials[blockIdx.x] = b1; partials[kMaxPartials + blockIdx.x] = b2; }
}

// |H|_F^2 of the symmetric H from its stored upper blocks (off-diagonal blocks twice), per-CTA sums into partials
__global__ void __launch_bounds__(kNT) marg_hnorm_kernel(const double *__restrict__ H, const int32_t *__restrict__ colidx,
                                                         const int32_t *__restrict__ blk_row, long long n, int dd,
                                                         double *__restrict__ partials) {
    __shared__ double sh[32];
    double acc = 0;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < n; t += (long long)gridDim.x * blockDim.x) {
        const long long k = t / dd;
        acc += (colidx[k] == blk_row[k] ? 1.0 : 2.0) * H[t] * H[t];
    }
    const double bs = block_sum<kNT>(acc, sh);
    if (threadIdx.x == 0) partials[blockIdx.x] = bs;
}

// out[0] = sum of partials[0, n), out[1] = sum of partials[kMaxPartials, kMaxPartials + n2) (fixed order)
__global__ void __launch_bounds__(kNT) marg_sum_kernel(const double *__restrict__ partials, int n, int n2,
                                                       double *__restrict__ out) {
    __shared__ double sh[32];
    const double v = sum_partials<kNT>(partials, n, sh);
    const double w = sum_partials<kNT>(partials + kMaxPartials, n2, sh);
    if (threadIdx.x == 0) { out[0] = v; out[1] = w; }
}

__global__ void marg_add_kernel(int n, const double *__restrict__ dx, double *__restrict__ x) {
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < n; t += gridDim.x * blockDim.x) x[t] += dx[t];
}

// component m of the requested blocks (row[q], c): out[dst[q]][a][m] = x[row[q] * D + a]
template <int D>
__global__ void marg_pcg_gather_kernel(const double *__restrict__ x, const int32_t *__restrict__ row,
                                       const int32_t *__restrict__ dst, int cnt, int m, double *__restrict__ out) {
    for (int item = blockIdx.x * blockDim.x + threadIdx.x; item < cnt * D; item += gridDim.x * blockDim.x) {
        const int q = item / D, a = item - q * D;
        out[(size_t)dst[q] * D * D + a * D + m] = x[(size_t)row[q] * D + a];
    }
}

// requested diagonal blocks: (X + X^T) / 2, one thread per mirrored pair of entries
template <int D>
__global__ void marg_symmetrize_kernel(const int32_t *__restrict__ dst, int cnt, double *__restrict__ out) {
    for (int item = blockIdx.x * blockDim.x + threadIdx.x; item < cnt * D * D; item += gridDim.x * blockDim.x) {
        const int q = item / (D * D), e = item - q * D * D, a = e / D, b = e - a * D;
        if (a >= b) continue;
        double *B = out + (size_t)dst[q] * D * D;
        const double v = 0.5 * (B[a * D + b] + B[b * D + a]);
        B[a * D + b] = v;
        B[b * D + a] = v;
    }
}

// What the LM carries across calls and the statistics of its solver.  The route runs the LM's PCG on the LM's work
// vectors and scalars; the destructor puts all of this back on every exit path.  (The LM's host state -- lambda, nu,
// chi2, the estimate snapshots -- is not touched by the route at all; the LM linearises again before its next solve,
// so the work vectors d_b, d_x, ... need no restoring.)
struct LmGuard {
    s3o_problem *p;
    DevScalars sc{};
    bool have_sc = false, had_amg;
    int last_pcg_iters, trace_state;
    bool auto_multilevel;
    s3o_stats st;
    int64_t rebuilds = 0, reuses = 0;
    explicit LmGuard(s3o_problem *q) : p(q), had_amg(q->amg != nullptr), last_pcg_iters(q->last_pcg_iters),
                                       trace_state(q->trace_state), auto_multilevel(q->auto_multilevel), st(q->stats) {
        amg_counts(p, &rebuilds, &reuses);
        have_sc = cudaMemcpyAsync(&sc, p->d_sc, sizeof(DevScalars), cudaMemcpyDeviceToHost, p->stream) == cudaSuccess &&
                  cudaStreamSynchronize(p->stream) == cudaSuccess;
        p->trace_state = 0;      // S3O_TRACE times an LM solve, not these
    }
    ~LmGuard() {
        if (have_sc) {
            cudaMemcpyAsync(p->d_sc, &sc, sizeof(DevScalars), cudaMemcpyHostToDevice, p->stream);
            cudaStreamSynchronize(p->stream);
            *p->h_sc = sc;
        }
        if (!had_amg) amg_destroy(p);       // a hierarchy built here only: the LM's preconditioner state as before
        else amg_set_counts(p, rebuilds, reuses);
        p->last_pcg_iters = last_pcg_iters;
        p->auto_multilevel = auto_multilevel;
        p->trace_state = trace_state;
        p->stats.pcg_iterations = st.pcg_iterations;
        p->stats.pcg_unconverged = st.pcg_unconverged;
        p->stats.ms_spmv_sampled = st.ms_spmv_sampled;
        p->stats.n_spmv_sampled = st.n_spmv_sampled;
        p->stats.direct_solves = st.direct_solves;
    }
};

struct DevBuf {     // device allocations of one call
    std::vector<void *> ptrs;
    template <class T> int alloc(T **ptr, size_t count) {
        int rc = dev_alloc(ptr, count);
        if (!rc) ptrs.push_back(*ptr);
        return rc;
    }
    ~DevBuf() { for (void *q : ptrs) cudaFree(q); }
};

template <int D>
int run(s3o_problem *p, int n_pairs, const int32_t *rows, const int32_t *cols, double *out, cudaEvent_t *ev) {
    const char *who = "s3o_compute_marginals";
    if (!rows) {
        set_error("%s: the factor of this graph exceeds the sparse Cholesky's cap of block products, and every diagonal "
                  "block by PCG would take n_free * d = %lld solves; request explicit pairs", who, (long long)p->S.nf * D);
        return S3O_ERR_UNSUPPORTED;
    }
    const int nf = p->S.nf, nd = nf * D;
    // requested pairs by column vertex (ascending), rows in request order; diagonal pairs for the symmetrisation
    std::vector<std::pair<int32_t, int32_t>> byc(n_pairs);
    for (int k = 0; k < n_pairs; ++k) byc[k] = { cols[k], k };
    std::sort(byc.begin(), byc.end());
    std::vector<int32_t> col_ptr, col_id, crow(n_pairs), cdst(n_pairs), diag;
    for (int q = 0; q < n_pairs; ++q) {
        if (q == 0 || byc[q].first != byc[q - 1].first) { col_ptr.push_back(q); col_id.push_back(byc[q].first); }
        crow[q] = rows[byc[q].second];
        cdst[q] = byc[q].second;
        if (rows[byc[q].second] == byc[q].first) diag.push_back(byc[q].second);
    }
    col_ptr.push_back(n_pairs);

    LmGuard guard(p);
    DevBuf buf;
    int32_t *d_crow = nullptr, *d_cdst = nullptr, *d_diag = nullptr;
    double *d_out = nullptr, *d_xt = nullptr, *d_rr = nullptr;
    int rc = 0;
    rc = rc ? rc : buf.alloc(&d_crow, crow.size());
    rc = rc ? rc : buf.alloc(&d_cdst, cdst.size());
    rc = rc ? rc : buf.alloc(&d_diag, diag.size());
    rc = rc ? rc : buf.alloc(&d_out, (size_t)n_pairs * D * D);
    rc = rc ? rc : buf.alloc(&d_xt, (size_t)nd);
    rc = rc ? rc : buf.alloc(&d_rr, 2);
    if (rc) { set_error("%s: device allocation failed", who); return rc; }
    auto h2d = [&](int32_t *dst, const std::vector<int32_t> &v) -> int {
        if (v.empty()) return S3O_OK;
        S3O_CUDA(cudaMemcpyAsync(dst, v.data(), v.size() * sizeof(int32_t), cudaMemcpyHostToDevice, p->stream));
        p->stats.h2d_bytes += (int64_t)(v.size() * sizeof(int32_t));
        return S3O_OK;
    };
    if ((rc = h2d(d_crow, crow)) || (rc = h2d(d_cdst, cdst)) || (rc = h2d(d_diag, diag))) return rc;

    // preconditioner at lambda = 0, once for every solve of the call
    bool amg = false;
    if (p->kind != S3O_KIND_BA && p->scale_model == S3O_SCALE_MODEL_DIFFERENCE) {
        if ((rc = amg_setup(p))) return rc;
        amg = amg_levels(p) > 0;
    }
    if ((rc = pcg_prepare(p, 0.0, amg))) return rc;
    double hnorm = 0;
    {
        const long long nh = (long long)p->S.nb * D * D;
        const int hgrid = grid_for(nh);
        marg_hnorm_kernel<<<hgrid, kNT, 0, p->stream>>>(p->d_H, p->d_colidx, p->d_blk_row, nh, D * D, p->d_partials);
        marg_sum_kernel<<<1, kNT, 0, p->stream>>>(p->d_partials, hgrid, 0, d_rr);
        if ((rc = check_launch(p, 2))) return rc;
        S3O_CUDA(cudaMemcpyAsync(&hnorm, d_rr, sizeof(double), cudaMemcpyDeviceToHost, p->stream));
        S3O_CUDA(cudaStreamSynchronize(p->stream));
        hnorm = std::sqrt(hnorm);
    }
    if (ev) cudaEventRecord(ev[0], p->stream);

    const bool trace = getenv("S3O_MARGINALS_TRACE") != nullptr;
    const StructDev s = struct_view(p);
    const int vgrid = grid_for(nd), rgrid = grid_for(nd);
    const double tol = S3O_MARGINALS_PCG_TOL;
    for (size_t g = 0; g + 1 < col_ptr.size(); ++g) {
        const int c = col_id[g], cnt = col_ptr[g + 1] - col_ptr[g];
        int its[8] = {}, rounds_max = 0;
        double worst = 0, worst_back = 0;
        for (int m = 0; m < D; ++m) {
            const int idx = c * D + m;
            marg_unit_rhs_kernel<<<vgrid, kNT, 0, p->stream>>>(p->d_b, nd, idx);
            if ((rc = check_launch(p, 1))) return rc;
            double pcg_tol = 0.5 * tol, res = 0, prev = 0, back = 0;
            int used = 0, round = 0;
            for (;; ++round) {
                if ((rc = pcg_iterate(p, 0.0, amg, pcg_tol, kMargMaxIter - used))) return rc;
                used += p->h_sc->iters;
                if (p->h_sc->done == 3) {
                    set_error("%s: the PCG solve of column vertex %d (Hessian index %d), component %d broke down after %d "
                              "iterations", who, p->S.free2v[c], c, m, used);
                    return S3O_ERR_SOLVE;
                }
                if (round == 0) S3O_CUDA(cudaMemcpyAsync(d_xt, p->d_x, sizeof(double) * nd, cudaMemcpyDeviceToDevice, p->stream));
                else marg_add_kernel<<<vgrid, kNT, 0, p->stream>>>(nd, p->d_x, d_xt);
                // true residual r = e - H x, also the right-hand side of the next correction
                hessian_product(p, d_xt);
                marg_residual_kernel<D><<<rgrid, kNT, 0, p->stream>>>(s, nf, p->d_q1, p->d_T, d_xt, idx, p->d_b, p->d_partials);
                marg_sum_kernel<<<1, kNT, 0, p->stream>>>(p->d_partials, rgrid, rgrid, d_rr);
                if ((rc = check_launch(p, round ? 4 : 3))) return rc;
                double rr[2] = {};
                S3O_CUDA(cudaMemcpyAsync(rr, d_rr, sizeof rr, cudaMemcpyDeviceToHost, p->stream));
                S3O_CUDA(cudaStreamSynchronize(p->stream));
                p->stats.d2h_bytes += sizeof rr;
                res = std::sqrt(rr[0]);
                back = res / (hnorm * std::sqrt(rr[1]));
                if (res <= tol) break;
                // at the rounding floor: a round that no longer halves the residual, at a backward error of round-off
                if (round > 0 && res > 0.5 * prev && back <= kMargBackTol) break;
                if (!std::isfinite(res) || round == kMargMaxRounds || used >= kMargMaxIter) {
                    set_error("%s: the PCG solve of column vertex %d (Hessian index %d), component %d reached a true residual "
                              "of %.3e (backward error %.2e) after %d iterations and %d refinement rounds (tolerance %.1e)",
                              who, p->S.free2v[c], c, m, res, back, used, round, tol);
                    return S3O_ERR_SOLVE;
                }
                prev = res;
                pcg_tol = std::min(0.5, 0.5 * tol / res);     // the correction's residual relative to r
            }
            marg_pcg_gather_kernel<D><<<std::max(1, std::min(1024, (cnt * D + 255) / 256)), 256, 0, p->stream>>>(
                d_xt, d_crow + col_ptr[g], d_cdst + col_ptr[g], cnt, m, d_out);
            if ((rc = check_launch(p, 1))) return rc;
            its[m] = used;
            rounds_max = std::max(rounds_max, round);
            worst = std::max(worst, res);
            worst_back = std::max(worst_back, back);
        }
        if (trace) {
            fprintf(stderr, "s3o_compute_marginals: column %d (vertex %d): PCG iterations", c, p->S.free2v[c]);
            for (int m = 0; m < D; ++m) fprintf(stderr, " %d", its[m]);
            fprintf(stderr, ", refinement rounds %d, true residual %.3e, backward error %.3e\n", rounds_max, worst, worst_back);
        }
    }
    if (ev) cudaEventRecord(ev[1], p->stream);
    if (!diag.empty()) {
        marg_symmetrize_kernel<D><<<std::min(1024, ((int)diag.size() * D * D + 255) / 256), 256, 0, p->stream>>>(
            d_diag, (int)diag.size(), d_out);
        if ((rc = check_launch(p, 1))) return rc;
    }
    if (ev) cudaEventRecord(ev[2], p->stream);
    if (n_pairs > 0) S3O_CUDA(cudaMemcpyAsync(out, d_out, sizeof(double) * n_pairs * D * D, cudaMemcpyDeviceToHost, p->stream));
    S3O_CUDA(cudaStreamSynchronize(p->stream));
    p->stats.d2h_bytes += (int64_t)n_pairs * D * D * 8;
    return S3O_OK;
}

}  // namespace

int pcg_marginals(s3o_problem *p, int n_pairs, const int32_t *rows, const int32_t *cols, double *out, cudaEvent_t *ev) {
    switch (p->d) {
    case 7: return run<7>(p, n_pairs, rows, cols, out, ev);
    case 4: return run<4>(p, n_pairs, rows, cols, out, ev);
    case 1: return run<1>(p, n_pairs, rows, cols, out, ev);
    }
    set_error("s3o_compute_marginals: block dimension %d", p->d);
    return S3O_ERR_UNSUPPORTED;
}

}  // namespace s3o
