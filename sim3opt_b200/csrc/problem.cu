// problem.cu -- the s3o_problem object, the Levenberg-Marquardt driver and the C ABI.
//
// The driver restates OptimizationAlgorithmLevenberg::solve inside SparseOptimizer::optimize
// [EXT g2o] (SURVEY.md section 3.1; reference call sites kitti_surf.cpp:674-675, :1021-1022,
// :1044-1045) with every numeric step on the device:
//   computeActiveErrors/activeRobustChi2 -> chi2 kernel      buildSystem -> linearize + assemble
//   setLambda/solve/restoreDiagonal      -> precond + PCG (lambda added inside the SpMV)
//   push / update / pop / discardTop     -> retract into the alternate estimate buffer + swap
//   computeScale, computeLambdaInit      -> device reductions
// The host only sees three scalars per trial (chi2, scale, PCG status).
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <memory>
#include <thread>
#include <vector>

#include "problem.h"
#include "amg.h"
#include "direct.h"

namespace s3o {

static thread_local char g_err[512] = "";
void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}

}  // namespace s3o

using namespace s3o;


namespace {
void run_spmv(s3o_problem *p, const StructDev &s, double lambda, const double *x, int pcg_mode);

GraphDev graph_view(const s3o_problem *p, int which) {
    GraphDev g{};
    g.kind = p->kind; g.d = p->d; g.est_dim = p->est_dim; g.ninfo = p->ninfo;
    g.nv = p->nv; g.nv_pad = p->nv_pad; g.ne = p->S.ne_act; g.ne_pad = p->ne_pad; g.nf = p->S.nf; g.nb = p->S.nb;
    g.est = p->d_est[which]; g.aux = p->d_aux; g.hidx = p->d_hidx; g.sv0 = p->d_sv0; g.sv1 = p->d_sv1;
    g.meas = p->d_meas; g.info = p->has_info ? p->d_info : nullptr; g.info_diag = p->info_diag;
    g.robust_kind = p->robust_kind; g.robust_param = p->robust_param;
    g.math_corrected = p->math_mode == S3O_MATH_CORRECTED;
    g.model_flags = (g.math_corrected ? 1 : 0) | (p->scale_model == S3O_SCALE_MODEL_LOGRATIO ? 2 : 0);
    g.primary = p->dist ? p->d_primary : nullptr;
    g.ghidx = p->dist ? p->d_ghidx : nullptr;
    return g;
}

}  // namespace

namespace s3o {

// undo setup_p2p: unmap the peers' memory (free_structure then synchronises the ranks before any exported
// vector is freed)
void close_p2p(s3o_problem *p) {
    for (void *m : p->ipc_mapped) cudaIpcCloseMemHandle(m);
    p->ipc_mapped.clear();
    dev_free(p->d_flag); dev_free(p->d_ghost_src); dev_free(p->d_peer_flags);
    p->p2p = false;
    p->n_peers = 0;
}

StructDev struct_view(const s3o_problem *p) {
    StructDev s{};
    s.rowptr = p->d_rowptr; s.colidx = p->d_colidx; s.blk_row = p->d_blk_row;
    s.blk_ebeg = p->d_blk_ebeg; s.blk_eend = p->d_blk_eend; s.blk_src = p->d_blk_src;
    s.multi_blk = p->d_multi_blk; s.n_multi = (int)p->S.multi_blk.size();
    s.colT_ptr = p->d_colT_ptr; s.colT_blk = p->d_colT_blk;
    s.inc_ptr = p->d_inc_ptr; s.inc_ent = p->d_inc_ent; s.e_blk = p->d_e_blk;
    s.tile_row = p->d_tile_row; s.ntiles = (int)p->S.tile_row.size() - 1;
    s.n_own = p->dist ? p->plan.n_own : p->S.nf;
    s.ghost_src = nullptr;      // set per product by run_spmv when the peer-to-peer halo is active
    return s;
}

void free_structure(s3o_problem *p) {
    // Peer-to-peer halo: unmap the neighbours' vectors FIRST, then meet every rank at a barrier, and only then
    // free the vector the neighbours had mapped (cudaFree of an exported allocation before the importers'
    // cudaIpcCloseMemHandle is undefined behaviour).  free_structure is reached collectively (s3o_set_vertices /
    // s3o_set_edges / s3o_set_comm / s3o_destroy are called by every rank), so the barrier matches.
    if (p->p2p) {
        if (p->stream) cudaStreamSynchronize(p->stream);
        close_p2p(p);
        if (p->dist && p->comm.nccl && p->d_sc) {
            comm_allreduce_max(p->comm, &p->d_sc->maxdiag, 1, p->stream);
            cudaStreamSynchronize(p->stream);
        }
    }
    dev_free(p->d_hidx); dev_free(p->d_sv0); dev_free(p->d_sv1); dev_free(p->d_meas); dev_free(p->d_info);
    dev_free(p->d_rowptr); dev_free(p->d_colidx); dev_free(p->d_blk_row); dev_free(p->d_blk_ebeg);
    dev_free(p->d_blk_eend); dev_free(p->d_colT_ptr); dev_free(p->d_colT_blk); dev_free(p->d_inc_ptr);
    dev_free(p->d_inc_ent); dev_free(p->d_e_blk); dev_free(p->d_tile_row); dev_free(p->d_blk_src); dev_free(p->d_multi_blk);
    dev_free(p->d_ghidx); dev_free(p->d_send_idx); dev_free(p->d_primary); dev_free(p->d_sendbuf); dev_free(p->d_xg);
    dev_free(p->d_H); dev_free(p->d_b); dev_free(p->d_x); dev_free(p->d_r); dev_free(p->d_z); dev_free(p->d_p);
    dev_free(p->d_q1); dev_free(p->d_T); dev_free(p->d_Minv); dev_free(p->d_scratch);
    close_p2p(p);
    amg_destroy(p);
    direct_destroy(p);
    p->last_pcg_iters = 0;
    p->auto_multilevel = false;
    p->built = false;
    p->linearized = false;
}

int check_launch(s3o_problem *p, int n) {
    p->stats.kernel_launches += n;
    S3O_CUDA(cudaGetLastError());
    return S3O_OK;
}

}  // namespace s3o

namespace {

// rows this rank solves for (all free vertices on one GPU)
inline int own_rows(const s3o_problem *p) { return p->dist ? p->plan.n_own : p->S.nf; }

int allreduce_sum(s3o_problem *p, double *field, int count) {
    if (!p->dist) return S3O_OK;
    if (comm_allreduce_sum(p->comm, field, count, p->stream)) { set_error("%s", comm_last_error()); return S3O_ERR_NCCL; }
    return S3O_OK;
}
int allreduce_max(s3o_problem *p, double *field, int count) {
    if (!p->dist) return S3O_OK;
    if (comm_allreduce_max(p->comm, field, count, p->stream)) { set_error("%s", comm_last_error()); return S3O_ERR_NCCL; }
    return S3O_OK;
}

}  // namespace

namespace s3o {
int sync_scalars(s3o_problem *p) {
    S3O_CUDA(cudaMemcpyAsync(p->h_sc, p->d_sc, sizeof(DevScalars), cudaMemcpyDeviceToHost, p->stream));
    unsigned bar[2] = { 0, 0 };
    S3O_CUDA(cudaMemcpyAsync(bar, p->d_gridbar, sizeof bar, cudaMemcpyDeviceToHost, p->stream));
    S3O_CUDA(cudaStreamSynchronize(p->stream));
    p->stats.d2h_bytes += sizeof(DevScalars);
    if (bar[1]) {       // a persistent kernel's grid barrier timed out (gridbar.cuh): its result is not to be used
        cudaMemsetAsync(p->d_gridbar, 0, sizeof bar, p->stream);
        set_error("a persistent kernel's grid barrier timed out (are other kernels holding this GPU's SMs?); S3O_COOP_LAUNCH=1 "
                  "selects cooperative launches");
        return S3O_ERR_CUDA;
    }
    return S3O_OK;
}
}  // namespace s3o

namespace {

int ensure_built(s3o_problem *p) {
    if (p->built) return S3O_OK;
    return s3o_build_structure(p, nullptr, nullptr);
}

bool uses_spmv4(const s3o_problem *p) {
    const int ntiles = (int)p->S.tile_row.size() - 1;
    return p->spmv_version == 4 && p->d == 7 && p->S.max_row_blocks <= p->S.tile_blocks && spmv4_fits(ntiles, p->spmv_grid_cap);
}

void run_spmv(s3o_problem *p, const StructDev &s, double lambda, const double *x, int pcg_mode) {
    if (p->spmv_version == 1 && !p->dist)
        launch_spmv(p->d, p->d_H, s, p->S.nf, lambda, x, p->d_q1, p->d_T, p->d_partials, p->d_sc, pcg_mode, p->stream);
    else if (uses_spmv4(p)) {
        StructDev s4 = s;
        if (p->p2p && x == p->d_p) s4.ghost_src = p->d_ghost_src;      // ghost columns read from the owners' p
        launch_spmv4(p->d_H, s4, own_rows(p), lambda, x, p->d_q1, p->d_T, p->d_partials, p->d_sc, pcg_mode,
                     p->spmv4_cfg, p->spmv_grid_cap, p->dist, p->stream);
    }
    else if (p->spmv_version >= 3 && p->S.max_row_blocks <= p->S.tile_blocks)
        launch_spmv3(p->d, p->d_H, s, own_rows(p), lambda, x, p->d_q1, p->d_T, p->d_partials, p->d_sc, pcg_mode,
                     p->spmv_grid_cap, p->dist, p->stream);
    else
        launch_spmv2(p->d, p->d_H, s, own_rows(p), lambda, x, p->d_q1, p->d_T, p->d_partials, p->d_sc, pcg_mode,
                     p->dist, p->stream);
}

int do_chi2(s3o_problem *p, int which) {
    if (p->kind == S3O_KIND_BA) return ba_chi2(p, which);
    if (p->S.ne_act == 0) {
        S3O_CUDA(cudaMemsetAsync(&p->d_sc->chi2, 0, sizeof(double), p->stream));
        return allreduce_sum(p, &p->d_sc->chi2, 1);
    }
    launch_chi2(graph_view(p, which), p->d_partials, p->d_sc, p->stream);
    int rc = check_launch(p, 1);
    return rc ? rc : allreduce_sum(p, &p->d_sc->chi2, 1);
}

int do_linearize(s3o_problem *p) {
    if (p->kind == S3O_KIND_BA) return ba_linearize(p);
    const GraphDev g = graph_view(p, p->cur);
    launch_linearize(g, p->jac_mode, p->jac_h, p->d_scratch, p->d_e_blk, p->d_blk_src, p->d_H, p->stream);
    launch_assemble(g, struct_view(p), p->d_scratch, p->d_H, p->d_b, p->stream);
    amg_invalidate_frames(p);
    direct_invalidate(p);
    p->linearized = true;
    return check_launch(p, 2);
}

}  // namespace

namespace s3o {
// multilevel preconditioner: Sim3 graphs on one GPU; AUTO switches it on for large graphs
bool wants_multilevel(const s3o_problem *p) {
    const int nf = p->dist ? p->plan.nf_global : p->S.nf;
    // (the coarse space of the scale kinds is built on the additive scale update: not with the log-ratio model)
    return p->kind != S3O_KIND_BA && p->kind != 100 /* solver-only handle: no poses to build the coarse space on */ &&
           p->scale_model == S3O_SCALE_MODEL_DIFFERENCE &&
           (p->precond == S3O_PRECOND_MULTILEVEL || (p->precond == S3O_PRECOND_AUTO && (nf >= 20000 || p->auto_multilevel)));
}

// Solve (H + lambda I) x = b; leaves x in d_x.  Returns the PCG status in *status (1 converged,
// 2 iteration cap, 3 breakdown) and the iteration count.
int do_solve(s3o_problem *p, double lambda, int *status, int *iters, double *rel_res, bool defer_sync) {
    if (p->linsolver != S3O_LINSOLVER_PCG) {       // exact solve when the factor is small (direct.cu)
        int rcd = p->dist ? S3O_OK : direct_setup(p);
        if (rcd) return rcd;
        if (direct_available(p)) {
            if ((rcd = direct_solve(p, lambda, p->reuse_factor))) return rcd;
            if (status) *status = 0;
            if (iters) *iters = 0;
            if (rel_res) *rel_res = 0;
            if (defer_sync) return S3O_OK;
            if ((rcd = sync_scalars(p))) return rcd;
            if (status) *status = p->h_sc->done;
            return S3O_OK;
        }
        if (p->linsolver == S3O_LINSOLVER_DIRECT) {
            set_error("s3o_set_linear_solver(DIRECT): %s", p->dist ? "not available in the partitioned solve"
                                                                   : "the factor of this graph is too large; use PCG");
            return S3O_ERR_UNSUPPORTED;
        }
    }
    bool amg = false;
    int rc;
    if (wants_multilevel(p)) {
        if ((rc = amg_setup(p))) return rc;
        amg = amg_levels(p) > 0;
    }
    if ((rc = pcg_prepare(p, lambda, amg))) return rc;
    if ((rc = pcg_iterate(p, lambda, amg, p->pcg_tol, p->pcg_max_iter))) return rc;
    // AUTO on a small graph: block-Jacobi until a solve turns out to be ill-conditioned (small lambda on
    // a long chain), the multilevel correction from the next solve on
    // (and back once the multilevel solves get so cheap -- large lambda -- that its setup dominates)
    if (p->precond == S3O_PRECOND_AUTO && (p->kind == S3O_KIND_SIM3 || p->kind == S3O_KIND_SCALE_TRANS)) {
        if (!amg && p->h_sc->iters > 256) p->auto_multilevel = true;
        else if (amg && p->auto_multilevel && p->h_sc->iters <= 8) p->auto_multilevel = false;
    }
    if (status) *status = p->h_sc->done ? p->h_sc->done : 2;
    if (iters) *iters = p->h_sc->iters;
    if (rel_res) *rel_res = p->h_sc->rr0 > 0 ? std::sqrt(p->h_sc->rr / p->h_sc->rr0) : 0.0;
    return S3O_OK;
}

void hessian_product(s3o_problem *p, const double *x) { run_spmv(p, struct_view(p), 0.0, x, 0); }

// Block-Jacobi inverses of (H + lambda I) and, with the multilevel correction, its Galerkin operators.
int pcg_prepare(s3o_problem *p, double lambda, bool amg) {
    launch_precond(p->d, p->d_H, p->d_rowptr, own_rows(p), lambda, p->d_Minv, p->d_sc, p->stream);
    int rc = check_launch(p, 1);
    if (!rc && amg) rc = amg_update_values(p, lambda);
    return rc;
}

// PCG on (H + lambda I) x = p->d_b from x = 0, x in p->d_x, to the relative recurrence residual tol or max_iter
// iterations; the verdict in p->h_sc (done, iters, rr, rr0).
int pcg_iterate(s3o_problem *p, double lambda, bool amg, double tol, int max_iter) {
    const int nf = own_rows(p), d = p->d;
    const int dist = p->dist ? 1 : 0;
    const StructDev s = struct_view(p);
    const PartitionPlan &P = p->plan;
    auto halo = [&]() -> int {     // bring the ghost entries of p up to date before the product
        if (!dist) return S3O_OK;
        if (p->p2p) {               // the SpMV reads them from the owners' memory: publish my epoch, wait for theirs
            ++p->halo_epoch;
            launch_halo_signal(p->d_flag, p->halo_epoch, p->stream);
            launch_halo_wait(p->d_peer_flags, p->n_peers, p->halo_epoch, p->d_sc, p->stream);
            p->stats.kernel_launches += 2;
            return S3O_OK;
        }
        launch_pack_rows(d, p->d_p, p->d_send_idx, (int)P.send_idx.size(), p->d_sendbuf, p->d_sc, p->stream);
        p->stats.kernel_launches += 1;
        if (comm_halo(p->comm, p->d_sendbuf, P.send_off.data(), P.send_count.data(), p->d_p + (size_t)P.n_own * d,
                      P.recv_off.data(), P.recv_count.data(), d, p->stream)) {
            set_error("%s", comm_last_error());
            return S3O_ERR_NCCL;
        }
        return S3O_OK;
    };
    int rc;
    // with the multilevel correction the vector kernels leave r.z to amg_apply (like the partitioned
    // solve leaves it to the all-reduce)
    const int defer = dist || amg;
    launch_pcg_init(d, nf, p->d_b, p->d_Minv, p->d_x, p->d_r, p->d_z, p->d_p, p->d_partials, p->d_sc, tol,
                    max_iter, defer, p->stream);
    rc = check_launch(p, 1);
    if (rc) return rc;
    if (amg) {      // restriction, V-cycle, r.z (riding on the r_1 all-gather when partitioned), p = z
        if ((rc = amg_apply(p, 1, tol, max_iter))) return rc;
    } else if (dist) {
        if ((rc = allreduce_sum(p, &p->d_sc->rz_new, 2))) return rc;
        launch_pcg_fin_init(p->d_sc, tol, max_iter, p->stream);
        p->stats.kernel_launches += 1;
    }
    // Iterations are launched in batches between host checks of the convergence flag; an iteration launched after
    // convergence exits at once but still costs ~30 launches (~120 us).  The first batch is sized by what the
    // previous solve needed (consecutive LM iterations need similar counts), later ones grow geometrically.
    int batch = p->last_pcg_iters > 0 ? std::max(2, std::min(64, p->last_pcg_iters - 1)) : 8, launched = 0;
    if (p->trace_state == 1 && p->trace_solve > 0) --p->trace_solve;
    for (;;) {
        for (int k = 0; k < batch; ++k) {
            const bool sample = ((launched + k) & 15) == 7 && p->spmv_ev_used < s3o_problem::kSpmvEvents;
            if (p->trace_state == 1 && p->trace_solve == 0 && launched + k == 4) { p->trace_state = 2; trace_mark(p, "start"); }
            if ((rc = halo())) return rc;
            if (sample) {
                p->spmv_ev_iter[p->spmv_ev_used] = launched + k;
                cudaEventRecord(p->spmv_ev[2 * p->spmv_ev_used], p->stream);
            }
            run_spmv(p, s, lambda, p->d_p, 1);
            trace_mark(p, "spmv");
            if (sample) cudaEventRecord(p->spmv_ev[2 * p->spmv_ev_used++ + 1], p->stream);
            if (dist) {
                if ((rc = allreduce_sum(p, &p->d_sc->pq, 1))) return rc;
                launch_pcg_fin_spmv(p->d_sc, p->stream);
            }
            launch_pcg_update(d, s, nf, p->d_q1, p->d_T, p->d_Minv, p->d_p, p->d_x, p->d_r, p->d_z, p->d_partials,
                              p->d_sc, defer, p->stream);
            trace_mark(p, "pcg_update");
            if (amg) {      // ... r.z, beta and p = z + beta p included
                if ((rc = amg_apply(p, 0, tol, max_iter))) return rc;
                if (p->trace_state == 2) { trace_mark(p, "end"); p->trace_state = 3; }
                continue;
            }
            if (dist) {
                if ((rc = allreduce_sum(p, &p->d_sc->rz_new, 2))) return rc;
                launch_pcg_fin_update(p->d_sc, p->stream);
            }
            launch_pcg_pupdate(d, nf, p->d_z, p->d_p, p->d_sc, p->stream);
        }
        launched += batch;
        rc = check_launch(p, (amg ? (dist ? 3 : 2) : (dist ? 5 : 3)) * batch);
        if (rc) return rc;
        rc = sync_scalars(p);
        if (rc) return rc;
        if (p->trace_state == 3) {
            float tot = 0;
            cudaEventElapsedTime(&tot, p->trace.front().second, p->trace.back().second);
            fprintf(stderr, "S3O_TRACE one PCG iteration: %.1f us\n", tot * 1e3f);
            for (size_t t = 1; t < p->trace.size(); ++t) {
                float ms = 0;
                cudaEventElapsedTime(&ms, p->trace[t - 1].second, p->trace[t].second);
                fprintf(stderr, "  %-28s %8.1f us\n", p->trace[t].first, ms * 1e3f);
            }
            for (auto &t : p->trace) cudaEventDestroy(t.second);
            p->trace.clear();
            p->trace_state = 0;
        }
        // a launch after convergence exits at once: keep only the samples of iterations that ran
        // (launch index < iterations executed)
        for (int e = 0; e < p->spmv_ev_used; ++e) {
            float ms = 0;
            if (cudaEventElapsedTime(&ms, p->spmv_ev[2 * e], p->spmv_ev[2 * e + 1]) == cudaSuccess &&
                (!p->h_sc->done || p->spmv_ev_iter[e] < p->h_sc->iters)) {
                p->stats.ms_spmv_sampled += ms;
                p->stats.n_spmv_sampled += 1;
            }
        }
        p->spmv_ev_used = 0;
        if (p->h_sc->done || launched >= max_iter + batch) break;
        batch = launched < 16 ? std::max(2, launched / 2) : std::min(64, launched);
    }
    p->stats.pcg_iterations += p->h_sc->iters;
    p->last_pcg_iters = p->h_sc->iters;
    if (p->h_sc->done != 1) p->stats.pcg_unconverged += 1;      // iteration cap or breakdown: the step is inexact
    return S3O_OK;
}
}  // namespace s3o

namespace s3o {

// BSR-upper arrays of p->S (rows, columns, block->row, column view, SpMV tiles) -> device
int upload_structure_arrays(s3o_problem *p, int rows_own, bool on_device) {
    HostStructure &S = p->S;
    int rc = 0;
    if (!on_device) {       // (the device build hands its own copies over)
        std::vector<int32_t> blk_row(S.nb);
        for (int r = 0; r < S.nf; ++r)
            for (int k = S.rowptr[r]; k < S.rowptr[r + 1]; ++k) blk_row[k] = r;
        rc = rc ? rc : upload(p, &p->d_rowptr, S.rowptr);
        rc = rc ? rc : upload(p, &p->d_colidx, S.colidx);
        rc = rc ? rc : upload(p, &p->d_blk_row, blk_row);
        rc = rc ? rc : upload(p, &p->d_colT_ptr, S.colT_ptr);
        rc = rc ? rc : upload(p, &p->d_colT_blk, S.colT_blk);
    }
    S.max_row_blocks = 0;
    for (int r = 0; r < rows_own; ++r) S.max_row_blocks = std::max(S.max_row_blocks, S.rowptr[r + 1] - S.rowptr[r]);
    S.tile_blocks = (p->spmv_version == 4 && p->d == 7) ? spmv4_tile_blocks(p->spmv4_cfg)
                    : (p->spmv_version >= 3 ? spmv3_tile_blocks(p->d) : spmv_tile_blocks(p->d));
    build_tiles(S.rowptr, rows_own, S.tile_blocks, S.tile_row);
    rc = rc ? rc : upload(p, &p->d_tile_row, S.tile_row);
    return rc;
}

// H, b and the PCG vectors for p->S; vectors are sized for owned + ghost rows, and x also serves
// as the all-gather send buffer (seg rows) in the partitioned solve
int alloc_linear_system(s3o_problem *p) {
    const HostStructure &S = p->S;
    const size_t nfd = (size_t)std::max(S.nf, p->dist ? p->plan.seg : 0) * p->d, dd = (size_t)p->d * p->d;
    int rc = 0;
    rc = rc ? rc : dev_alloc(&p->d_H, (size_t)S.nb * dd + 2);   // +16 B: the TMA tile copy rounds its size up
    rc = rc ? rc : dev_alloc(&p->d_b, nfd);
    rc = rc ? rc : dev_alloc(&p->d_x, nfd);
    rc = rc ? rc : dev_alloc(&p->d_r, nfd);
    rc = rc ? rc : dev_alloc(&p->d_z, nfd);
    rc = rc ? rc : dev_alloc(&p->d_p, nfd);
    rc = rc ? rc : dev_alloc(&p->d_q1, nfd);
    rc = rc ? rc : dev_alloc(&p->d_T, (size_t)S.nb * p->d);
    rc = rc ? rc : dev_alloc(&p->d_Minv, (size_t)S.nf * dd);
    return rc;
}

}  // namespace s3o

namespace {
// Peer-to-peer halo: every rank exports its p vector and an epoch flag through CUDA IPC, the handles travel by
// one NCCL all-gather, and each rank maps the vectors of the ranks it has ghosts from.  The SpMV then loads
// ghost columns straight from the owner's HBM over NVLink (ghost_src table).  All ranks take the same
// decision: if any mapping fails anywhere, everybody stays on the NCCL send/recv halo.
int setup_p2p(s3o_problem *p) {
    p->want_p2p_setup = false;
    if (getenv("S3O_NO_P2P") || !uses_spmv4(p)) return S3O_OK;
    const PartitionPlan &P = p->plan;
    const int world = P.world, rank = P.rank, d = p->d;
    struct Handles { cudaIpcMemHandle_t vec, flag; };
    int rc = dev_alloc(&p->d_flag, 1);
    if (rc) return rc;
    S3O_CUDA(cudaMemsetAsync(p->d_flag, 0, sizeof(long long), p->stream));
    Handles mine{};
    int ok = cudaIpcGetMemHandle(&mine.vec, p->d_p) == cudaSuccess && cudaIpcGetMemHandle(&mine.flag, p->d_flag) == cudaSuccess;
    cudaGetLastError();
    unsigned char *d_h = nullptr;
    if ((rc = dev_alloc(&d_h, sizeof(Handles) * (size_t)(world + 1)))) return rc;
    S3O_CUDA(cudaMemcpyAsync(d_h + sizeof(Handles) * world, &mine, sizeof(Handles), cudaMemcpyHostToDevice, p->stream));
    if (comm_allgather_bytes(p->comm, d_h + sizeof(Handles) * world, d_h, sizeof(Handles), p->stream)) {
        cudaFree(d_h); set_error("%s", comm_last_error()); return S3O_ERR_NCCL;
    }
    std::vector<Handles> all(world);
    S3O_CUDA(cudaMemcpyAsync(all.data(), d_h, sizeof(Handles) * world, cudaMemcpyDeviceToHost, p->stream));
    S3O_CUDA(cudaStreamSynchronize(p->stream));
    cudaFree(d_h);
    std::vector<double *> peer_vec(world, nullptr);
    std::vector<long long *> flags;
    for (int q = 0; q < world && ok; ++q) {
        if (q == rank || P.recv_count[q] == 0) continue;
        void *v = nullptr, *f = nullptr;
        if (cudaIpcOpenMemHandle(&v, all[q].vec, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { ok = 0; break; }
        p->ipc_mapped.push_back(v);
        if (cudaIpcOpenMemHandle(&f, all[q].flag, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { ok = 0; break; }
        p->ipc_mapped.push_back(f);
        peer_vec[q] = (double *)v;
        flags.push_back((long long *)f);
    }
    cudaGetLastError();
    if (flags.size() > 32) ok = 0;      // halo_wait_kernel polls one flag per lane of one warp
    // collective decision: 1 only if every rank mapped everything it needs
    double *d_ok = nullptr;
    if ((rc = dev_alloc(&d_ok, 1))) return rc;
    const double fail = ok ? 0.0 : 1.0;
    S3O_CUDA(cudaMemcpyAsync(d_ok, &fail, sizeof(double), cudaMemcpyHostToDevice, p->stream));
    if (comm_allreduce_max(p->comm, d_ok, 1, p->stream)) { cudaFree(d_ok); set_error("%s", comm_last_error()); return S3O_ERR_NCCL; }
    double any_fail = 1;
    S3O_CUDA(cudaMemcpyAsync(&any_fail, d_ok, sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    S3O_CUDA(cudaStreamSynchronize(p->stream));
    cudaFree(d_ok);
    if (any_fail != 0.0) { close_p2p(p); return S3O_OK; }       // NCCL halo everywhere
    std::vector<double *> src(P.n_ghost);
    for (int t = 0; t < P.n_ghost; ++t) {
        const int gidx = P.ghosts[t], q = gidx / P.seg;
        src[t] = peer_vec[q] + (size_t)(gidx - q * P.seg) * d;
    }
    rc = upload(p, &p->d_ghost_src, src);
    rc = rc ? rc : upload(p, &p->d_peer_flags, flags);
    if (rc) return rc;
    S3O_CUDA(cudaStreamSynchronize(p->stream));
    p->n_peers = (int)flags.size();
    p->halo_epoch = 0;
    p->p2p = true;
    return S3O_OK;
}
}  // namespace

// ======================================================================================
// C ABI
// ======================================================================================
extern "C" {

const char *s3o_last_error(void) { return g_err; }
int s3o_version(void) { return 100; }

int s3o_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

// kind of the handle behind s3o_linsolver_*: a block system only (no graph, no estimates)
static constexpr int kKindLinear = 100;

static int create_impl(int kind, int linear_dim, int device, s3o_problem **out) {
    if (!out) { set_error("s3o_create: out is NULL"); return S3O_ERR_INVALID; }
    *out = nullptr;
    int d, est_dim;
    switch (kind) {
    case kKindLinear: d = linear_dim; est_dim = 0; break;
    case S3O_KIND_SIM3: d = 7; est_dim = 8; break;
    case S3O_KIND_SCALE_TRANS: d = 4; est_dim = 4; break;
    case S3O_KIND_SCALE: d = 1; est_dim = 1; break;
    case S3O_KIND_BA: d = 6; est_dim = 7; break;     // Schur-complement system: 6x6 camera blocks
    default: set_error("s3o_create: unsupported kind %d", kind); return S3O_ERR_UNSUPPORTED;
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        set_error("s3o_create: no CUDA device available (this library has no CPU path)");
        return S3O_ERR_CUDA;
    }
    if (device < 0 || device >= ndev) { set_error("s3o_create: device %d out of range (%d devices)", device, ndev); return S3O_ERR_INVALID; }
    S3O_CUDA(cudaSetDevice(device));
    s3o_problem *p = new s3o_problem();
    p->kind = kind; p->d = d; p->est_dim = est_dim; p->ninfo = d * (d + 1) / 2; p->device = device;
    cudaError_t e = cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) { set_error("cudaStreamCreate: %s", cudaGetErrorString(e)); delete p; return S3O_ERR_CUDA; }
    p->own_stream = true;
    if (spmv2_configure() != 0) { set_error("s3o_create: cannot configure SpMV shared memory"); delete p; return S3O_ERR_CUDA; }
    if (const char *v = getenv("S3O_TRACE")) { p->trace_state = atoi(v) > 0 ? 1 : 0; p->trace_solve = atoi(v); }    // trace the n-th solve
    if (const char *v = getenv("S3O_SPMV_VERSION")) p->spmv_version = atoi(v);
    if (const char *v = getenv("S3O_SPMV_GRID")) {      // every CTA of the SpMV owns one of the kMaxPartials p.q partials
        const int g = atoi(v);
        if (g >= 1 && g <= kMaxPartials) p->spmv_grid_cap = g;
    }
    if (const char *v = getenv("S3O_SPMV4_CFG")) {
        const int c = atoi(v);
        if (c >= 0 && c <= 2) p->spmv4_cfg = c;
    }
    if (const char *v = getenv("S3O_PRECOND")) {        // experiment switch; s3o_set_preconditioner overrides it
        const int k = atoi(v);
        if (k >= S3O_PRECOND_AUTO && k <= S3O_PRECOND_MULTILEVEL && (k != S3O_PRECOND_MULTILEVEL || kind != S3O_KIND_BA)) p->precond = k;
    }
    for (auto &ev : p->ev) cudaEventCreate(&ev);
    for (auto &ev : p->spmv_ev) cudaEventCreate(&ev);
    if (const char *v = getenv("S3O_COOP_LAUNCH")) p->coop_launch = atoi(v) != 0;
    if (dev_alloc(&p->d_sc, 1) || dev_alloc(&p->d_partials, 3 * kMaxPartials) || dev_alloc(&p->d_gridbar, 2) ||
        cudaMallocHost((void **)&p->h_sc, sizeof(DevScalars)) != cudaSuccess) {
        s3o_destroy(p);
        return S3O_ERR_CUDA;
    }
    cudaMemsetAsync(p->d_sc, 0, sizeof(DevScalars), p->stream);
    cudaMemsetAsync(p->d_gridbar, 0, 2 * sizeof(unsigned), p->stream);
    memset(p->h_sc, 0, sizeof(DevScalars));
    p->stats.dim = d;
    *out = p;
    return S3O_OK;
}

int s3o_create(int kind, int device, s3o_problem **out) {
    if (kind == kKindLinear) { set_error("s3o_create: unsupported kind %d", kind); return S3O_ERR_UNSUPPORTED; }
    return create_impl(kind, 0, device, out);
}

// ---- LinearSolver-level entry (the slot of g2o::LinearSolver<M>::solve(A, x, b), kitti_surf.cpp:553-557) ----
int s3o_linsolver_create(int device, int block_dim, s3o_linsolver **out) {
    if (block_dim != 1 && block_dim != 4 && block_dim != 6 && block_dim != 7) {
        set_error("s3o_linsolver_create: block dimension %d (supported: 1, 4, 6, 7)", block_dim);
        return S3O_ERR_UNSUPPORTED;
    }
    return create_impl(kKindLinear, block_dim, device, out);
}

int s3o_linsolver_destroy(s3o_linsolver *p) { return s3o_destroy(p); }

int s3o_linsolver_solve(s3o_linsolver *p, int n, const int32_t *colptr, const int32_t *rowidx, const double *blocks,
                        int column_major, double lambda, const double *b, double *x, int *method, int *pcg_iterations) {
    if (!p || p->kind != kKindLinear || n < 0 || !colptr || (n > 0 && (!rowidx || !blocks || !b || !x))) { set_error("s3o_linsolver_solve: bad arguments"); return S3O_ERR_INVALID; }
    if (n == 0) return S3O_OK;
    cudaSetDevice(p->device);
    const int d = p->d, dd = d * d, nb = colptr[n];
    // same pattern as the last call (LinearSolver::init() once, solve() per LM trial): keep structure and plan
    bool same = p->built && p->S.nf == n && p->S.nb == nb &&
                memcmp(p->S.ccs_colptr.data(), colptr, sizeof(int32_t) * (n + 1)) == 0 &&
                memcmp(p->S.ccs_rowidx.data(), rowidx, sizeof(int32_t) * nb) == 0;
    if (!same) {
        free_structure(p);
        std::vector<int32_t> v0, v1;
        for (int c = 0; c < n; ++c) {
            bool diag = false;
            for (int k = colptr[c]; k < colptr[c + 1]; ++k) {
                const int r = rowidx[k];
                if (r < 0 || r > c || (k > colptr[c] && r <= rowidx[k - 1])) {
                    set_error("s3o_linsolver_solve: column %d is not an upper block-CCS column (rows ascending, row <= column)", c);
                    return S3O_ERR_INVALID;
                }
                if (r == c) diag = true;
                else { v0.push_back(r); v1.push_back(c); }
            }
            if (!diag) { set_error("s3o_linsolver_solve: column %d has no diagonal block", c); return S3O_ERR_INVALID; }
        }
        p->nv = n;
        p->fixed.assign(n, 0);
        build_structure_host(n, nullptr, (int)v0.size(), v0.data(), v1.data(), p->S);
        if (p->S.nb != nb || memcmp(p->S.ccs_rowidx.data(), rowidx, sizeof(int32_t) * nb) != 0) { set_error("s3o_linsolver_solve: pattern mismatch"); return S3O_ERR_INVALID; }
        int rc = upload_structure_arrays(p, n);
        rc = rc ? rc : alloc_linear_system(p);
        if (rc) { free_structure(p); return rc; }
        p->built = true;
        p->stats.n_free = n; p->stats.n_blocks = nb;
    }
    // blocks into BSR-upper order (row-major d x d)
    std::vector<double> H((size_t)nb * dd);
    for (int c = 0; c < nb; ++c) {
        double *dst = H.data() + (size_t)p->S.ccs2bsr[c] * dd;
        const double *src = blocks + (size_t)c * dd;
        if (!column_major) memcpy(dst, src, sizeof(double) * dd);
        else
            for (int r = 0; r < d; ++r)
                for (int cc = 0; cc < d; ++cc) dst[r * d + cc] = src[cc * d + r];
    }
    S3O_CUDA(cudaMemcpyAsync(p->d_H, H.data(), H.size() * sizeof(double), cudaMemcpyHostToDevice, p->stream));
    S3O_CUDA(cudaMemcpyAsync(p->d_b, b, (size_t)n * d * sizeof(double), cudaMemcpyHostToDevice, p->stream));
    p->stats.h2d_bytes += (int64_t)((H.size() + (size_t)n * d) * sizeof(double));
    p->linearized = true;
    direct_invalidate(p);
    int status = 0, iters = 0;
    int rc = do_solve(p, lambda, &status, &iters, nullptr);
    if (rc) return rc;
    S3O_CUDA(cudaMemcpyAsync(x, p->d_x, (size_t)n * d * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    S3O_CUDA(cudaStreamSynchronize(p->stream));
    p->stats.d2h_bytes += (int64_t)n * d * 8;
    if (method) *method = direct_available(p) && p->linsolver != S3O_LINSOLVER_PCG ? S3O_LINSOLVER_DIRECT : S3O_LINSOLVER_PCG;
    if (pcg_iterations) *pcg_iterations = iters;
    if (status == 3) { set_error("s3o_linsolver_solve: the matrix is not positive definite (pivot / PCG breakdown)"); return S3O_ERR_SOLVE; }
    if (status == 2) { set_error("s3o_linsolver_solve: PCG hit the iteration cap"); return S3O_ERR_SOLVE; }
    return S3O_OK;
}

int s3o_destroy(s3o_problem *p) {
    if (!p) return S3O_OK;
    cudaSetDevice(p->device);
    if (p->stream) cudaStreamSynchronize(p->stream);
    free_structure(p);
    ba_destroy(p);
    dev_free(p->d_meas_aos); dev_free(p->d_info_aos);
    dev_free(p->d_est[0]); dev_free(p->d_est[1]); dev_free(p->d_aux);
    dev_free(p->d_sc); dev_free(p->d_partials); dev_free(p->d_gridbar);
    comm_destroy(p->comm);
    if (p->h_sc) cudaFreeHost(p->h_sc);
    for (auto &ev : p->ev) if (ev) cudaEventDestroy(ev);
    for (auto &ev : p->spmv_ev) if (ev) cudaEventDestroy(ev);
    dev_free(p->d_est_snap);
    dev_free(p->d_stage);
    if (p->own_stream && p->stream) cudaStreamDestroy(p->stream);
    delete p;
    return S3O_OK;
}

int s3o_comm_unique_id(char *id128) {
    if (!id128) return S3O_ERR_INVALID;
    if (comm_unique_id(id128)) { set_error("%s", comm_last_error()); return S3O_ERR_NCCL; }
    return S3O_OK;
}

int s3o_set_comm(s3o_problem *p, int rank, int world, const char *id128) {
    if (!p || world < 1 || rank < 0 || rank >= world || (world > 1 && !id128)) { set_error("s3o_set_comm: bad arguments"); return S3O_ERR_INVALID; }
    if (p->kind == S3O_KIND_BA && world > 1) {
        set_error("s3o_set_comm: bundle adjustment has no partitioned path (replicas only, SURVEY.md 8e)");
        return S3O_ERR_UNSUPPORTED;
    }
    cudaSetDevice(p->device);
    free_structure(p);
    comm_destroy(p->comm);
    p->dist = false;
    if (world == 1) return S3O_OK;
    if (comm_init(p->comm, rank, world, id128)) { set_error("%s", comm_last_error()); return S3O_ERR_NCCL; }
    p->dist = true;
    return S3O_OK;
}

int s3o_set_stream(s3o_problem *p, void *cuda_stream) {
    if (!p) return S3O_ERR_INVALID;
    cudaSetDevice(p->device);
    if (p->stream) cudaStreamSynchronize(p->stream);
    if (p->own_stream && p->stream) cudaStreamDestroy(p->stream);
    p->own_stream = false;
    p->stream = (cudaStream_t)cuda_stream;
    if (!cuda_stream) {
        S3O_CUDA(cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking));
        p->own_stream = true;
    }
    return S3O_OK;
}

// caller-ordered (AoS) staging buffer of the vertex estimates: allocated once per vertex set, so
// the per-step host round trip of the estimates never pays a cudaMalloc / cudaFree (both
// device-synchronising, and measured at up to 0.4 s after a long solve)
static int ensure_stage(s3o_problem *p) {
    if (p->d_stage) return S3O_OK;
    return dev_alloc(&p->d_stage, (size_t)p->nv * p->est_dim);
}

static int upload_estimates(s3o_problem *p, const double *est) {
    const size_t cnt = (size_t)p->nv * p->est_dim;
    int rc = ensure_stage(p);
    if (rc) return rc;
    double *tmp = p->d_stage;
    cudaError_t e = cudaMemcpyAsync(tmp, est, cnt * sizeof(double), cudaMemcpyHostToDevice, p->stream);
    if (e == cudaSuccess) {
        launch_pack_vertices(tmp, p->nv, p->nv_pad, p->est_dim, p->d_est[p->cur], p->stream);
        e = cudaStreamSynchronize(p->stream);
    }
    if (e != cudaSuccess) { set_error("upload_estimates: %s", cudaGetErrorString(e)); return S3O_ERR_CUDA; }
    p->stats.h2d_bytes += (int64_t)(cnt * sizeof(double));
    p->stats.kernel_launches += 1;
    return S3O_OK;
}

int s3o_set_vertices(s3o_problem *p, int n, const double *est, const uint8_t *fixed, const double *aux) {
    if (!p || n < 0 || (n > 0 && !est)) { set_error("s3o_set_vertices: bad arguments"); return S3O_ERR_INVALID; }
    if (p->kind == S3O_KIND_BA) { set_error("s3o_set_vertices: a BA problem takes s3o_ba_set_cameras / s3o_ba_set_points"); return S3O_ERR_INVALID; }
    if (p->kind == S3O_KIND_SCALE_TRANS && !aux && n > 0) { set_error("s3o_set_vertices: SCALE_TRANS needs aux rotations"); return S3O_ERR_INVALID; }
    cudaSetDevice(p->device);
    free_structure(p);
    dev_free(p->d_est[0]); dev_free(p->d_est[1]); dev_free(p->d_aux);
    p->nv = n;
    p->nv_pad = pad32(n);
    p->cur = 0;
    p->lm_valid = false;
    dev_free(p->d_est_snap);
    dev_free(p->d_stage);
    p->fixed.assign(n, 0);
    if (fixed) memcpy(p->fixed.data(), fixed, n);
    int rc;
    if ((rc = dev_alloc(&p->d_est[0], (size_t)p->nv_pad * p->est_dim))) return rc;
    if ((rc = dev_alloc(&p->d_est[1], (size_t)p->nv_pad * p->est_dim))) return rc;
    S3O_CUDA(cudaMemsetAsync(p->d_est[0], 0, (size_t)p->nv_pad * p->est_dim * sizeof(double), p->stream));
    S3O_CUDA(cudaMemsetAsync(p->d_est[1], 0, (size_t)p->nv_pad * p->est_dim * sizeof(double), p->stream));
    if ((rc = upload_estimates(p, est))) return rc;
    p->has_aux = aux != nullptr;
    if (aux) {
        double *tmp = nullptr;
        if ((rc = dev_alloc(&tmp, (size_t)n * 4))) return rc;
        if ((rc = dev_alloc(&p->d_aux, (size_t)p->nv_pad * 4))) { cudaFree(tmp); return rc; }
        cudaError_t e = cudaMemcpyAsync(tmp, aux, (size_t)n * 4 * sizeof(double), cudaMemcpyHostToDevice, p->stream);
        if (e == cudaSuccess) {
            launch_pack_vertices(tmp, n, p->nv_pad, 4, p->d_aux, p->stream);
            e = cudaStreamSynchronize(p->stream);
        }
        cudaFree(tmp);
        if (e != cudaSuccess) { set_error("s3o_set_vertices(aux): %s", cudaGetErrorString(e)); return S3O_ERR_CUDA; }
        p->stats.h2d_bytes += (int64_t)n * 32;
        p->stats.kernel_launches += 1;
    }
    p->stats.n_vertices = n;
    return S3O_OK;
}

int s3o_set_estimates(s3o_problem *p, const double *est) {
    if (p && p->kind == S3O_KIND_BA) { set_error("s3o_set_estimates: a BA problem takes s3o_ba_set_estimates"); return S3O_ERR_INVALID; }
    if (!p || !est || !p->d_est[0]) { set_error("s3o_set_estimates: call s3o_set_vertices first"); return S3O_ERR_INVALID; }
    cudaSetDevice(p->device);
    p->linearized = false;
    if (p->lm_resume != 2) { p->lm_valid = false; p->auto_multilevel = false; }
    return upload_estimates(p, est);
}

// ---- sharded host round trip of the estimates (partitioned solve) -------------------------------
// Every rank keeps ALL estimates on its device (cut edges, retraction), but the host side of a rank only has to move
// its share: the even split of the vertex ids.  Slices are all-gathered over NVLink into the staging buffer.
static void estimate_slice(const s3o_problem *p, int rank, int *first, int *count) {
    const int world = p->dist ? p->comm.world : 1;
    const int per = (p->nv + world - 1) / world;
    const int f = std::min(p->nv, rank * per);
    *first = f;
    *count = std::max(0, std::min(per, p->nv - f));
}

int s3o_estimate_slice(s3o_problem *p, int *first, int *count) {
    if (!p || !first || !count || p->kind == S3O_KIND_BA) { set_error("s3o_estimate_slice: bad arguments"); return S3O_ERR_INVALID; }
    estimate_slice(p, p->dist ? p->comm.rank : 0, first, count);
    return S3O_OK;
}

int s3o_set_estimates_slice(s3o_problem *p, const double *est_slice) {
    if (!p || p->kind == S3O_KIND_BA || !p->d_est[0]) { set_error("s3o_set_estimates_slice: call s3o_set_vertices first"); return S3O_ERR_INVALID; }
    cudaSetDevice(p->device);
    p->linearized = false;
    if (p->lm_resume != 2) { p->lm_valid = false; p->auto_multilevel = false; }
    int rc = ensure_stage(p);
    if (rc) return rc;
    const int world = p->dist ? p->comm.world : 1, rank = p->dist ? p->comm.rank : 0;
    int first = 0, count = 0;
    estimate_slice(p, rank, &first, &count);
    if (count > 0 && !est_slice) { set_error("s3o_set_estimates_slice: null slice"); return S3O_ERR_INVALID; }
    const size_t ed = (size_t)p->est_dim;
    if (count > 0) S3O_CUDA(cudaMemcpyAsync(p->d_stage + first * ed, est_slice, count * ed * sizeof(double), cudaMemcpyHostToDevice, p->stream));
    if (world > 1) {
        std::vector<size_t> off(world), cnt(world);
        for (int q = 0; q < world; ++q) {
            int f = 0, c = 0;
            estimate_slice(p, q, &f, &c);
            off[q] = f * ed;
            cnt[q] = c * ed;
        }
        if (comm_allgatherv(p->comm, p->d_stage, off.data(), cnt.data(), p->stream)) { set_error("%s", comm_last_error()); return S3O_ERR_NCCL; }
    }
    launch_pack_vertices(p->d_stage, p->nv, p->nv_pad, p->est_dim, p->d_est[p->cur], p->stream);
    S3O_CUDA(cudaStreamSynchronize(p->stream));
    p->stats.h2d_bytes += (int64_t)(count * ed * sizeof(double));
    p->stats.kernel_launches += 1;
    return S3O_OK;
}

int s3o_get_vertices_slice(s3o_problem *p, double *est_slice) {
    if (!p || p->kind == S3O_KIND_BA || !p->d_est[0]) { set_error("s3o_get_vertices_slice: no vertices"); return S3O_ERR_INVALID; }
    cudaSetDevice(p->device);
    int rc = ensure_stage(p);
    if (rc) return rc;
    int first = 0, count = 0;
    estimate_slice(p, p->dist ? p->comm.rank : 0, &first, &count);
    if (count > 0 && !est_slice) { set_error("s3o_get_vertices_slice: null slice"); return S3O_ERR_INVALID; }
    const size_t ed = (size_t)p->est_dim;
    launch_unpack_vertices(p->d_est[p->cur], p->nv, p->nv_pad, p->est_dim, p->d_stage, p->stream);
    if (count > 0) S3O_CUDA(cudaMemcpyAsync(est_slice, p->d_stage + first * ed, count * ed * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    S3O_CUDA(cudaStreamSynchronize(p->stream));
    p->stats.d2h_bytes += (int64_t)(count * ed * sizeof(double));
    p->stats.kernel_launches += 1;
    return S3O_OK;
}

int s3o_set_edges(s3o_problem *p, int n, const int32_t *v0, const int32_t *v1, const double *meas, const double *info) {
    if (!p || n < 0 || (n > 0 && (!v0 || !v1 || !meas))) { set_error("s3o_set_edges: bad arguments"); return S3O_ERR_INVALID; }
    if (p->kind == S3O_KIND_BA) { set_error("s3o_set_edges: a BA problem takes s3o_ba_set_observations"); return S3O_ERR_INVALID; }
    for (int k = 0; k < n; ++k)
        if (v0[k] < 0 || v0[k] >= p->nv || v1[k] < 0 || v1[k] >= p->nv || v0[k] == v1[k]) {
            set_error("s3o_set_edges: edge %d has invalid vertices (%d,%d), n_vertices=%d", k, v0[k], v1[k], p->nv);
            return S3O_ERR_INVALID;
        }
    cudaSetDevice(p->device);
    setup_mark(nullptr);
    free_structure(p);
    dev_free(p->d_meas_aos); dev_free(p->d_info_aos);
    p->user_ne = n;
    p->has_info = info != nullptr;
    p->info_diag = false;
    // Diagonal information matrices (the usual case) are kept as their d diagonal entries.  One threaded pass over
    // the caller's matrices checks the off-diagonal entries and extracts the diagonals at the same time (the buffer
    // is left uninitialised so that its pages are first touched by the threads that fill them).
    std::unique_ptr<double[]> info_diag_host;
    if (info && n > 0) {
        const int dd = p->d * p->d, d = p->d;
        const unsigned hw = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
        info_diag_host.reset(new double[(size_t)n * d]);
        double *dst = info_diag_host.get();
        std::vector<char> nondiag(hw, 0);
        std::vector<std::thread> th;
        for (unsigned w = 0; w < hw; ++w)
            th.emplace_back([&, w]() {
                const size_t lo = (size_t)n * w / hw, hi = (size_t)n * (w + 1) / hw;
                for (size_t k = lo; k < hi && !nondiag[w]; ++k) {
                    const double *M = info + k * dd;
                    for (int e = 0; e < dd; ++e) {
                        const int r = e / d, c = e - r * d;
                        if (r == c) dst[k * d + r] = M[e];
                        else if (M[e] != 0.0) { nondiag[w] = 1; break; }
                    }
                }
            });
        for (auto &t : th) t.join();
        p->info_diag = true;
        for (char f : nondiag) if (f) p->info_diag = false;
        if (!p->info_diag) info_diag_host.reset();
    }
    setup_mark("set_edges: info scan");
    std::vector<double> meas_loc, info_loc;
    if (p->dist) {
        // keep only the edges that touch a vertex this rank owns (cut edges live on both sides)
        build_partition_plan(p->nv, p->fixed.data(), n, v0, v1, p->comm.rank, p->comm.world, p->plan);
        const PartitionPlan &P = p->plan;
        p->gv0.assign(v0, v0 + n);
        p->gv1.assign(v1, v1 + n);
        const int nl = (int)P.local_edges.size();
        const int ed = p->est_dim, dd = p->d * p->d;
        p->v0.resize(nl); p->v1.resize(nl);
        meas_loc.resize((size_t)nl * ed);
        // the information matrices of the local edges: their diagonals when all are diagonal, else the full matrices
        const int iw = p->info_diag ? p->d : dd;
        const double *isrc = p->info_diag ? info_diag_host.get() : info;
        if (info) info_loc.resize((size_t)nl * iw);
        for (int t = 0; t < nl; ++t) {
            const size_t k = (size_t)P.local_edges[t];
            p->v0[t] = v0[k]; p->v1[t] = v1[k];
            memcpy(&meas_loc[(size_t)t * ed], meas + k * ed, sizeof(double) * ed);
            if (info) memcpy(&info_loc[(size_t)t * iw], isrc + k * iw, sizeof(double) * iw);
        }
        n = nl;
        meas = meas_loc.data();
        if (info) info = info_loc.data();       // (diagonals only when info_diag)
    } else {
        p->v0.assign(v0, v0 + n);
        p->v1.assign(v1, v1 + n);
    }
    p->ne = n;
    setup_mark("set_edges: index copy");
    int rc;
    const size_t mcount = (size_t)n * p->est_dim;
    if ((rc = dev_alloc(&p->d_meas_aos, mcount))) return rc;
    if (n) S3O_CUDA(cudaMemcpyAsync(p->d_meas_aos, meas, mcount * sizeof(double), cudaMemcpyHostToDevice, p->stream));
    p->stats.h2d_bytes += (int64_t)(mcount * sizeof(double));
    if (info) {
        const int d = p->d, dd = d * d;
        const double *src = info;
        size_t icount = (size_t)n * dd;
        if (p->info_diag) {         // 56 B per edge over PCIe instead of 392 B
            src = p->dist ? info : info_diag_host.get();
            icount = (size_t)n * d;
        }
        if ((rc = dev_alloc(&p->d_info_aos, icount))) return rc;
        if (n) S3O_CUDA(cudaMemcpyAsync(p->d_info_aos, src, icount * sizeof(double), cudaMemcpyHostToDevice, p->stream));
        p->stats.h2d_bytes += (int64_t)(icount * sizeof(double));
    }
    S3O_CUDA(cudaStreamSynchronize(p->stream));
    setup_mark("set_edges: upload");
    p->stats.n_edges = p->user_ne;
    return S3O_OK;
}

int s3o_set_robust(s3o_problem *p, int kind, double param) {
    if (!p || kind < S3O_ROBUST_NONE || kind > S3O_ROBUST_PTAM_LS) { set_error("s3o_set_robust: bad kind"); return S3O_ERR_INVALID; }
    if (kind != S3O_ROBUST_NONE && kind != S3O_ROBUST_PTAM_LS && !(param > 0)) { set_error("s3o_set_robust: param must be > 0"); return S3O_ERR_INVALID; }
    p->robust_kind = kind;
    p->robust_param = param;
    p->linearized = false;
    return S3O_OK;
}

int s3o_set_jacobian_mode(s3o_problem *p, int mode, double h) {
    if (!p || (mode != S3O_JAC_NUMERIC && mode != S3O_JAC_ANALYTIC)) { set_error("s3o_set_jacobian_mode: bad mode"); return S3O_ERR_INVALID; }
    p->jac_mode = mode;
    if (h > 0) p->jac_h = h;
    p->linearized = false;
    return S3O_OK;
}

int s3o_set_math_mode(s3o_problem *p, int mode) {
    if (!p || (mode != S3O_MATH_REFERENCE && mode != S3O_MATH_CORRECTED)) { set_error("s3o_set_math_mode: bad mode"); return S3O_ERR_INVALID; }
    p->math_mode = mode;
    p->linearized = false;
    return S3O_OK;
}

int s3o_set_scale_model(s3o_problem *p, int model) {
    if (!p || (model != S3O_SCALE_MODEL_DIFFERENCE && model != S3O_SCALE_MODEL_LOGRATIO)) { set_error("s3o_set_scale_model: bad model"); return S3O_ERR_INVALID; }
    if (p->kind != S3O_KIND_SCALE && p->kind != S3O_KIND_SCALE_TRANS) { set_error("s3o_set_scale_model: scale / scale-trans problems only"); return S3O_ERR_UNSUPPORTED; }
    p->scale_model = model;
    p->linearized = false;
    return S3O_OK;
}

int s3o_set_lm(s3o_problem *p, double tau, double user_lambda_init, int max_trials) {
    if (!p) return S3O_ERR_INVALID;
    if (tau > 0) p->tau = tau;
    p->user_lambda = user_lambda_init;
    if (max_trials > 0) p->max_trials = max_trials;
    return S3O_OK;
}

int s3o_set_preconditioner(s3o_problem *p, int kind) {
    if (!p) return S3O_ERR_INVALID;
    if (kind != S3O_PRECOND_AUTO && kind != S3O_PRECOND_BLOCK_JACOBI && kind != S3O_PRECOND_MULTILEVEL) {
        set_error("s3o_set_preconditioner: unknown kind %d", kind);
        return S3O_ERR_INVALID;
    }
    if (kind == S3O_PRECOND_MULTILEVEL && p->kind == S3O_KIND_BA) {
        set_error("s3o_set_preconditioner: the multilevel preconditioner is built on the gauge modes of a pose graph (not BA)");
        return S3O_ERR_UNSUPPORTED;
    }
    p->precond = kind;
    // naming a preconditioner asks for the Krylov solver (AUTO leaves the direct / PCG choice to the library)
    if (kind != S3O_PRECOND_AUTO && p->linsolver == S3O_LINSOLVER_AUTO) p->linsolver = S3O_LINSOLVER_PCG;
    return S3O_OK;
}

int s3o_set_linear_solver(s3o_problem *p, int kind) {
    if (!p) return S3O_ERR_INVALID;
    if (kind != S3O_LINSOLVER_AUTO && kind != S3O_LINSOLVER_PCG && kind != S3O_LINSOLVER_DIRECT) {
        set_error("s3o_set_linear_solver: unknown kind %d", kind);
        return S3O_ERR_INVALID;
    }
    if (kind != p->linsolver) direct_destroy(p);     // the AUTO and DIRECT size limits differ: analyse again
    p->linsolver = kind;
    return S3O_OK;
}

int s3o_set_stop_rules(s3o_problem *p, double max_abs_step, double min_rel_predicted_decrease) {
    if (!p || !(max_abs_step >= 0) || !(min_rel_predicted_decrease >= 0)) { set_error("s3o_set_stop_rules: bad arguments"); return S3O_ERR_INVALID; }
    p->stop_step = max_abs_step;
    p->stop_pred = min_rel_predicted_decrease;
    return S3O_OK;
}

int s3o_set_pcg(s3o_problem *p, double rel_tol, int max_iter) {
    if (!p) return S3O_ERR_INVALID;
    if (rel_tol > 0) p->pcg_tol = rel_tol;
    if (max_iter > 0) p->pcg_max_iter = max_iter;
    return S3O_OK;
}

int s3o_build_structure(s3o_problem *p, int *n_free, int *n_blocks) {
    if (!p) return S3O_ERR_INVALID;
    if (p->kind == S3O_KIND_BA) {
        cudaSetDevice(p->device);
        if (!p->built) { int rc = ba_build_structure(p); if (rc) return rc; }
        if (n_free) *n_free = p->S.nf;
        if (n_blocks) *n_blocks = p->S.nb;
        return S3O_OK;
    }
    if (!p->d_est[0]) { set_error("s3o_build_structure: no vertices"); return S3O_ERR_INVALID; }
    cudaSetDevice(p->device);
    if (!p->built) {
        if (p->ne > 0 && !p->d_meas_aos) { set_error("s3o_build_structure: edges were consumed; call s3o_set_edges again"); return S3O_ERR_INVALID; }
        setup_mark(nullptr);
        free_structure(p);
        HostStructure &S = p->S;
        DeviceStructure dev;
        // the index build runs on the device (structure_dev.cu); S3O_STRUCTURE=host selects the host twin
        const char *where = getenv("S3O_STRUCTURE");
        if (where && !strcmp(where, "host")) {
            if (p->dist)
                build_structure_from_hidx(p->nv, p->plan.lhidx.data(), p->plan.n_own + p->plan.n_ghost, p->ne,
                                          p->v0.data(), p->v1.data(), S);
            else
                build_structure_host(p->nv, p->fixed.data(), p->ne, p->v0.data(), p->v1.data(), S);
        } else {
            const int rcs = p->dist ? build_structure_device(p->stream, p->nv, nullptr, p->plan.lhidx.data(), p->plan.n_own + p->plan.n_ghost,
                                                             p->ne, p->v0.data(), p->v1.data(), S, &dev)
                                    : build_structure_device(p->stream, p->nv, p->fixed.data(), nullptr, 0, p->ne, p->v0.data(), p->v1.data(), S, &dev);
            if (rcs) return rcs;
        }
        setup_mark("structure: index build");
        const int rows_own = p->dist ? p->plan.n_own : S.nf;
        p->ne_pad = pad32(S.ne_act);
        int rc = 0;
        int32_t *d_perm = nullptr;
        if (dev.valid) {        // built on the device: the arrays are already where they are needed
            p->d_hidx = dev.hidx; p->d_sv0 = dev.sv0; p->d_sv1 = dev.sv1; p->d_blk_ebeg = dev.blk_ebeg; p->d_blk_eend = dev.blk_eend;
            p->d_blk_src = dev.blk_src; p->d_multi_blk = dev.multi_blk; p->d_inc_ptr = dev.inc_ptr; p->d_inc_ent = dev.inc_ent;
            p->d_e_blk = dev.e_blk; p->d_rowptr = dev.rowptr; p->d_colidx = dev.colidx; p->d_blk_row = dev.blk_row;
            p->d_colT_ptr = dev.colT_ptr; p->d_colT_blk = dev.colT_blk;
            d_perm = dev.perm;
        } else {
            rc = rc ? rc : upload(p, &p->d_hidx, S.hidx);
            rc = rc ? rc : upload(p, &p->d_sv0, S.sv0);
            rc = rc ? rc : upload(p, &p->d_sv1, S.sv1);
            rc = rc ? rc : upload(p, &p->d_blk_ebeg, S.blk_ebeg);
            rc = rc ? rc : upload(p, &p->d_blk_eend, S.blk_eend);
            rc = rc ? rc : upload(p, &p->d_blk_src, S.blk_src);
            rc = rc ? rc : upload(p, &p->d_multi_blk, S.multi_blk);
            rc = rc ? rc : upload(p, &p->d_inc_ptr, S.inc_ptr);
            rc = rc ? rc : upload(p, &p->d_inc_ent, S.inc_ent);
            rc = rc ? rc : upload(p, &p->d_e_blk, S.e_blk);
        }
        setup_mark("  structure: edge-array uploads");
        rc = rc ? rc : upload_structure_arrays(p, rows_own, dev.valid);
        setup_mark("  structure: BSR/tile uploads");
        if (p->dist) {
            const PartitionPlan &P = p->plan;
            std::vector<uint8_t> prim(S.ne_act);
            for (int t = 0; t < S.ne_act; ++t) prim[t] = P.primary[S.perm[t]];
            rc = rc ? rc : upload(p, &p->d_primary, prim);
            rc = rc ? rc : upload(p, &p->d_ghidx, P.ghidx);
            rc = rc ? rc : upload(p, &p->d_send_idx, P.send_idx);
            rc = rc ? rc : dev_alloc(&p->d_sendbuf, P.send_idx.size() * p->d);
            rc = rc ? rc : dev_alloc(&p->d_xg, (size_t)P.world * P.seg * p->d);
        }
        p->want_p2p_setup = p->dist;
        if (!dev.valid) rc = rc ? rc : upload(p, &d_perm, S.perm);
        rc = rc ? rc : dev_alloc(&p->d_meas, (size_t)p->ne_pad * p->est_dim);
        const int info_planes = p->info_diag ? p->d : p->ninfo;
        if (p->has_info) rc = rc ? rc : dev_alloc(&p->d_info, (size_t)p->ne_pad * info_planes);
        rc = rc ? rc : alloc_linear_system(p);
        rc = rc ? rc : dev_alloc(&p->d_scratch, (size_t)p->ne_pad * scratch_stride(p->d));
        setup_mark("  structure: allocations");
        const size_t nfd = (size_t)std::max(S.nf, p->dist ? p->plan.seg : 0) * p->d;
        if (rc) { dev_free(d_perm); free_structure(p); return rc; }
        if (S.ne_act > 0) {
            cudaMemsetAsync(p->d_meas, 0, (size_t)p->ne_pad * p->est_dim * sizeof(double), p->stream);
            if (p->has_info) cudaMemsetAsync(p->d_info, 0, (size_t)p->ne_pad * info_planes * sizeof(double), p->stream);
            launch_pack_edges(p->d_meas_aos, p->has_info ? p->d_info_aos : nullptr, d_perm, S.ne_act, p->ne_pad,
                              p->est_dim, p->d, p->info_diag ? 1 : 0, p->d_meas, p->d_info, p->stream);
            p->stats.kernel_launches += 1;
        }
        cudaMemsetAsync(p->d_x, 0, nfd * sizeof(double), p->stream);
        cudaError_t e = cudaStreamSynchronize(p->stream);
        dev_free(d_perm);
        if (e != cudaSuccess || (e = cudaGetLastError()) != cudaSuccess) {
            set_error("s3o_build_structure: %s", cudaGetErrorString(e));
            free_structure(p);
            return S3O_ERR_CUDA;
        }
        dev_free(p->d_meas_aos);
        dev_free(p->d_info_aos);
        setup_mark("structure: uploads + pack");
        p->built = true;
        p->stats.n_free = S.nf; p->stats.n_blocks = S.nb;
        if (p->want_p2p_setup && (rc = setup_p2p(p))) return rc;
        // the aggregation hierarchy is structure work too: build it here rather than inside the first solve
        if (wants_multilevel(p) && (rc = amg_setup(p))) return rc;
        setup_mark("structure: hierarchy total");
    }
    if (n_free) *n_free = p->S.nf;
    if (n_blocks) *n_blocks = p->S.nb;
    return S3O_OK;
}

int s3o_host_structure(int n_vertices, const uint8_t *fixed, int n_edges, const int32_t *v0, const int32_t *v1,
                       int *n_free, int *n_blocks, int32_t *colptr, int32_t *rowidx, int32_t *hidx) {
    if (n_vertices < 0 || n_edges < 0 || (n_edges > 0 && (!v0 || !v1))) { set_error("s3o_host_structure: bad arguments"); return S3O_ERR_INVALID; }
    for (int k = 0; k < n_edges; ++k)
        if (v0[k] < 0 || v0[k] >= n_vertices || v1[k] < 0 || v1[k] >= n_vertices || v0[k] == v1[k]) {
            set_error("s3o_host_structure: edge %d has invalid vertices", k);
            return S3O_ERR_INVALID;
        }
    HostStructure S;
    build_structure_host(n_vertices, fixed, n_edges, v0, v1, S);
    if (n_free) *n_free = S.nf;
    if (n_blocks) *n_blocks = S.nb;
    if (colptr) memcpy(colptr, S.ccs_colptr.data(), sizeof(int32_t) * (S.nf + 1));
    if (rowidx) memcpy(rowidx, S.ccs_rowidx.data(), sizeof(int32_t) * S.nb);
    if (hidx) memcpy(hidx, S.hidx.data(), sizeof(int32_t) * n_vertices);
    return S3O_OK;
}

int s3o_host_partition(int n_vertices, const uint8_t *fixed, int n_edges, const int32_t *v0, const int32_t *v1,
                       int rank, int world, int32_t *n_own, int32_t *n_ghost, int32_t *n_local_edges,
                       int32_t *n_primary, int32_t *ghosts, int32_t *send_count, int32_t *recv_count,
                       int32_t *send_idx_global) {
    if (n_vertices < 0 || n_edges < 0 || world < 1 || rank < 0 || rank >= world) { set_error("s3o_host_partition: bad arguments"); return S3O_ERR_INVALID; }
    PartitionPlan P;
    build_partition_plan(n_vertices, fixed, n_edges, v0, v1, rank, world, P);
    if (n_own) *n_own = P.n_own;
    if (n_ghost) *n_ghost = P.n_ghost;
    if (n_local_edges) *n_local_edges = (int32_t)P.local_edges.size();
    if (n_primary) { int c = 0; for (uint8_t f : P.primary) c += f; *n_primary = c; }
    if (ghosts) memcpy(ghosts, P.ghosts.data(), sizeof(int32_t) * P.ghosts.size());
    if (send_count) memcpy(send_count, P.send_count.data(), sizeof(int32_t) * world);
    if (recv_count) memcpy(recv_count, P.recv_count.data(), sizeof(int32_t) * world);
    if (send_idx_global) for (size_t k = 0; k < P.send_idx.size(); ++k) send_idx_global[k] = P.send_idx[k] + P.own_lo;
    return S3O_OK;
}

int s3o_host_multilevel(int n_vertices, const uint8_t *fixed, int n_edges, const int32_t *v0, const int32_t *v1,
                        int world, int cap, int *n_levels, int32_t *level_vertices, int32_t *level_blocks,
                        int32_t *aggregate0) {
    if (n_vertices < 0 || n_edges < 0 || (n_edges > 0 && (!v0 || !v1)) || !n_levels || world < 1) { set_error("s3o_host_multilevel: bad arguments"); return S3O_ERR_INVALID; }
    for (int k = 0; k < n_edges; ++k)
        if (v0[k] < 0 || v0[k] >= n_vertices || v1[k] < 0 || v1[k] >= n_vertices || v0[k] == v1[k]) {
            set_error("s3o_host_multilevel: edge %d has invalid vertices", k);
            return S3O_ERR_INVALID;
        }
    HostStructure S;
    build_structure_host(n_vertices, fixed, n_edges, v0, v1, S);
    std::vector<s3o::AmgHostLevel> lv;
    // world > 1: the hierarchy of the partitioned solve (aggregates stay inside the ranks' vertex ranges)
    const int seg = world > 1 ? (S.nf + world - 1) / world : 0;
    s3o::amg_build_hierarchy(S, S.nf >= 20000 ? 128 : 16, 12, lv, seg);      // same rule as amg_setup
    *n_levels = (int)lv.size();
    for (int l = 0; l < (int)lv.size() && l < cap; ++l) {
        if (level_vertices) level_vertices[l] = lv[l].n;
        if (level_blocks) level_blocks[l] = (int32_t)lv[l].colidx.size();
    }
    if (aggregate0 && !lv.empty()) memcpy(aggregate0, lv[0].agg.data(), sizeof(int32_t) * S.nf);
    return S3O_OK;
}

int s3o_host_direct_plan(int n_vertices, const uint8_t *fixed, int n_edges, const int32_t *v0, const int32_t *v1,
                         int64_t max_pairs, int64_t *counts, int32_t *perm, int32_t *lev_ptr, int32_t *cptr,
                         int32_t *brow, int32_t *src, int32_t *upd_ptr, int32_t *upd_a, int32_t *upd_b) {
    if (n_vertices < 0 || n_edges < 0 || (n_edges > 0 && (!v0 || !v1)) || !counts) { set_error("s3o_host_direct_plan: bad arguments"); return S3O_ERR_INVALID; }
    for (int k = 0; k < n_edges; ++k)
        if (v0[k] < 0 || v0[k] >= n_vertices || v1[k] < 0 || v1[k] >= n_vertices || v0[k] == v1[k]) {
            set_error("s3o_host_direct_plan: edge %d has invalid vertices", k);
            return S3O_ERR_INVALID;
        }
    HostStructure S;
    build_structure_host(n_vertices, fixed, n_edges, v0, v1, S);
    s3o::DirectPlan P;
    if (!s3o::direct_analyze(S.nf, S.rowptr, S.colidx, max_pairs > 0 ? max_pairs : (1ll << 62), P)) {
        set_error("s3o_host_direct_plan: the factor needs more than %lld block products", (long long)max_pairs);
        return S3O_ERR_UNSUPPORTED;
    }
    counts[0] = P.n; counts[1] = P.nlev; counts[2] = (int64_t)P.brow.size(); counts[3] = (int64_t)P.upd_a.size();
    counts[4] = P.n_pairs;
    auto put = [](int32_t *dst, const std::vector<int32_t> &v) { if (dst && !v.empty()) memcpy(dst, v.data(), sizeof(int32_t) * v.size()); };
    put(perm, P.perm); put(lev_ptr, P.lev_ptr); put(cptr, P.cptr); put(brow, P.brow); put(src, P.src);
    put(upd_ptr, P.upd_ptr); put(upd_a, P.upd_a); put(upd_b, P.upd_b);
    return S3O_OK;
}

int s3o_get_structure(s3o_problem *p, int32_t *colptr, int32_t *rowidx) {
    if (!p || !p->built) { set_error("s3o_get_structure: structure not built"); return S3O_ERR_INVALID; }
    if (colptr) memcpy(colptr, p->S.ccs_colptr.data(), sizeof(int32_t) * (p->S.nf + 1));
    if (rowidx) memcpy(rowidx, p->S.ccs_rowidx.data(), sizeof(int32_t) * p->S.nb);
    return S3O_OK;
}

int s3o_get_hessian_index(s3o_problem *p, int32_t *hidx) {
    if (!p || !p->built || !hidx) { set_error("s3o_get_hessian_index: structure not built"); return S3O_ERR_INVALID; }
    memcpy(hidx, p->S.hidx.data(), sizeof(int32_t) * p->nv);
    return S3O_OK;
}

int s3o_chi2(s3o_problem *p, double *chi2) {
    if (!p || !chi2) return S3O_ERR_INVALID;
    cudaSetDevice(p->device);
    int rc = ensure_built(p);
    if (rc) return rc;
    if ((rc = do_chi2(p, p->cur))) return rc;
    if ((rc = sync_scalars(p))) return rc;
    *chi2 = p->h_sc->chi2;
    return S3O_OK;
}

int s3o_edge_errors(s3o_problem *p, double *err) {
    if (!p || !err) return S3O_ERR_INVALID;
    if (p->kind == S3O_KIND_BA) return s3o_ba_edge_errors(p, err);
    cudaSetDevice(p->device);
    int rc = ensure_built(p);
    if (rc) return rc;
    const int na = p->S.ne_act, d = p->d;
    double *d_err = nullptr;
    if ((rc = dev_alloc(&d_err, (size_t)na * d))) return rc;
    launch_edge_errors(graph_view(p, p->cur), d_err, nullptr, p->stream);
    std::vector<double> tmp((size_t)na * d);
    cudaError_t e = cudaMemcpyAsync(tmp.data(), d_err, tmp.size() * sizeof(double), cudaMemcpyDeviceToHost, p->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(p->stream);
    cudaFree(d_err);
    if (e != cudaSuccess) { set_error("s3o_edge_errors: %s", cudaGetErrorString(e)); return S3O_ERR_CUDA; }
    p->stats.kernel_launches += 1;
    p->stats.d2h_bytes += (int64_t)(tmp.size() * sizeof(double));
    // caller's edge order; in the partitioned solve only the edges this rank evaluates are filled
    memset(err, 0, sizeof(double) * (size_t)(p->dist ? p->user_ne : p->ne) * d);
    for (int t = 0; t < na; ++t) {
        const size_t user = p->dist ? (size_t)p->plan.local_edges[p->S.perm[t]] : (size_t)p->S.perm[t];
        memcpy(err + user * d, tmp.data() + (size_t)t * d, sizeof(double) * d);
    }
    return S3O_OK;
}

int s3o_linearize(s3o_problem *p) {
    if (!p) return S3O_ERR_INVALID;
    cudaSetDevice(p->device);
    int rc = ensure_built(p);
    if (rc) return rc;
    if ((rc = do_linearize(p))) return rc;
    S3O_CUDA(cudaStreamSynchronize(p->stream));
    return S3O_OK;
}

int s3o_get_hessian(s3o_problem *p, double *blocks, double *b) {
    if (p && p->kind == S3O_KIND_BA) { set_error("s3o_get_hessian: a BA problem exposes s3o_ba_get_system / s3o_ba_get_schur"); return S3O_ERR_INVALID; }
    if (!p || !p->built || !p->linearized) { set_error("s3o_get_hessian: call s3o_linearize first"); return S3O_ERR_INVALID; }
    cudaSetDevice(p->device);
    const size_t dd = (size_t)p->d * p->d;
    if (blocks) {
        std::vector<double> tmp((size_t)p->S.nb * dd);
        S3O_CUDA(cudaMemcpyAsync(tmp.data(), p->d_H, tmp.size() * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
        S3O_CUDA(cudaStreamSynchronize(p->stream));
        p->stats.d2h_bytes += (int64_t)(tmp.size() * sizeof(double));
        for (int c = 0; c < p->S.nb; ++c)
            memcpy(blocks + (size_t)c * dd, tmp.data() + (size_t)p->S.ccs2bsr[c] * dd, dd * sizeof(double));
    }
    if (b) {
        S3O_CUDA(cudaMemcpyAsync(b, p->d_b, (size_t)p->S.nf * p->d * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
        S3O_CUDA(cudaStreamSynchronize(p->stream));
        p->stats.d2h_bytes += (int64_t)p->S.nf * p->d * 8;
    }
    return S3O_OK;
}

int s3o_max_diag(s3o_problem *p, double *max_diag) {
    if (!p || !p->built || !p->linearized || !max_diag) { set_error("s3o_max_diag: call s3o_linearize first"); return S3O_ERR_INVALID; }
    cudaSetDevice(p->device);
    int rc;
    if (p->kind == S3O_KIND_BA) rc = ba_max_diag(p);
    else {
        launch_maxdiag(p->d, p->d_H, p->d_rowptr, own_rows(p), p->d_partials, p->d_sc, p->stream);
        rc = check_launch(p, 1);
    }
    if (rc) return rc;
    if ((rc = allreduce_max(p, &p->d_sc->maxdiag, 1))) return rc;
    if ((rc = sync_scalars(p))) return rc;
    *max_diag = p->h_sc->maxdiag;
    return S3O_OK;
}

int s3o_solve(s3o_problem *p, double lambda, double *x, int *pcg_iters, double *rel_residual) {
    if (!p || !p->built || !p->linearized) { set_error("s3o_solve: call s3o_linearize first"); return S3O_ERR_INVALID; }
    cudaSetDevice(p->device);
    int status = 0;
    if (p->kind == S3O_KIND_BA) {       // x = [cameras 6 n_free_cameras | points 3 n_free_points]
        int rc = ba_solve(p, lambda, &status, pcg_iters, rel_residual);
        if (rc) return rc;
        if (x && (rc = ba_download_step(p, x))) return rc;
        if (status == 3) { set_error("s3o_solve: the Schur system is not positive definite"); return S3O_ERR_SOLVE; }
        return S3O_OK;
    }
    int rc = do_solve(p, lambda, &status, pcg_iters, rel_residual);
    if (rc) return rc;
    if (x) {
        S3O_CUDA(cudaMemcpyAsync(x, p->d_x, (size_t)p->S.nf * p->d * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
        S3O_CUDA(cudaStreamSynchronize(p->stream));
        p->stats.d2h_bytes += (int64_t)p->S.nf * p->d * 8;
    }
    if (status == 3) { set_error("s3o_solve: the damped Hessian is not positive definite (pivot / PCG breakdown)"); return S3O_ERR_SOLVE; }
    return S3O_OK;
}

int s3o_hessian_multiply(s3o_problem *p, double lambda, const double *x, double *y) {
    if (!p || !p->built || !p->linearized || !x || !y) { set_error("s3o_hessian_multiply: call s3o_linearize first"); return S3O_ERR_INVALID; }
    if (p->dist) { set_error("s3o_hessian_multiply: a lock-step getter of the single-GPU problem (the partitioned solve holds owned rows only)"); return S3O_ERR_UNSUPPORTED; }
    cudaSetDevice(p->device);
    const size_t bytes = (size_t)p->S.nf * p->d * sizeof(double);
    S3O_CUDA(cudaMemcpyAsync(p->d_p, x, bytes, cudaMemcpyHostToDevice, p->stream));
    run_spmv(p, struct_view(p), lambda, p->d_p, 0);
    launch_finish_q(p->d, struct_view(p), p->S.nf, p->d_q1, p->d_T, p->d_z, p->stream);
    int rc = check_launch(p, 2);
    if (rc) return rc;
    S3O_CUDA(cudaMemcpyAsync(y, p->d_z, bytes, cudaMemcpyDeviceToHost, p->stream));
    S3O_CUDA(cudaStreamSynchronize(p->stream));
    p->stats.h2d_bytes += (int64_t)bytes;
    p->stats.d2h_bytes += (int64_t)bytes;
    return S3O_OK;
}

int s3o_update(s3o_problem *p, const double *x) {
    if (!p || !x) return S3O_ERR_INVALID;
    cudaSetDevice(p->device);
    int rc = ensure_built(p);
    if (rc) return rc;
    if (p->kind == S3O_KIND_BA) {
        if ((rc = ba_upload_step(p, x))) return rc;
        if ((rc = ba_retract_and_scale(p, 0.0, p->cur ^ 1))) return rc;
        S3O_CUDA(cudaStreamSynchronize(p->stream));
        p->cur ^= 1;
        p->linearized = false;
        return S3O_OK;
    }
    // partitioned solve: x holds this rank's OWNED rows (the first n_own entries of the local numbering); they are
    // all-gathered so that every rank retracts every vertex from the same global step, exactly like s3o_optimize
    const double *xfull = p->d_x;
    const size_t bytes = (size_t)(p->dist ? p->plan.n_own : p->S.nf) * p->d * sizeof(double);
    if (p->dist) S3O_CUDA(cudaMemsetAsync(p->d_x, 0, (size_t)p->plan.seg * p->d * sizeof(double), p->stream));
    S3O_CUDA(cudaMemcpyAsync(p->d_x, x, bytes, cudaMemcpyHostToDevice, p->stream));
    if (p->dist) {
        if (comm_allgather(p->comm, p->d_x, p->d_xg, (size_t)p->plan.seg * p->d, p->stream)) {
            set_error("%s", comm_last_error());
            return S3O_ERR_NCCL;
        }
        xfull = p->d_xg;
    }
    launch_retract(graph_view(p, p->cur), xfull, p->d_est[p->cur ^ 1], p->stream);
    if ((rc = check_launch(p, 1))) return rc;
    S3O_CUDA(cudaStreamSynchronize(p->stream));
    p->cur ^= 1;
    p->linearized = false;
    p->stats.h2d_bytes += (int64_t)bytes;
    return S3O_OK;
}

int s3o_optimize(s3o_problem *p, int max_iter, double stop_rel_gain, int *iterations, double *final_chi2,
                 double *final_lambda, double *hist, int hist_cap) {
    if (!p) return S3O_ERR_INVALID;
    cudaSetDevice(p->device);
    int rc = ensure_built(p);
    if (rc) return rc;
    if (iterations) *iterations = -1;
    // partitioned solve: decided on the GLOBAL count, so that a rank that happens to own no row still takes part
    // in every collective of the loop below (zero-sized local work)
    if (p->dist ? p->plan.nf_global == 0 : p->S.nf == 0) { set_error("s3o_optimize: 0 vertices to optimize"); return S3O_ERR_INVALID; }
    const int nf = own_rows(p), d = p->d;
    const bool resume = p->lm_resume != 0 && p->lm_valid;
    double lambda = resume ? p->lm_lambda : 0, ni = resume ? p->lm_ni : 2, currentChi = resume ? p->lm_chi : 0;
    if (!resume) { p->lm_prev_step = 0; p->lm_est_dist = 0; p->lm_stop_hits = 0; }
    int done = 0;
    p->stats.ms_linearize = p->stats.ms_solve = p->stats.ms_chi2 = p->stats.ms_update = p->stats.ms_total = 0;
    cudaEventRecord(p->ev[0], p->stream);
    int result = S3O_RESULT_OK;
    for (int it = 0; it < max_iter; ++it) {
        if (it == 0 && !resume) {
            if ((rc = do_chi2(p, p->cur))) return rc;
        }
        cudaEventRecord(p->ev[1], p->stream);
        if ((rc = do_linearize(p))) return rc;
        cudaEventRecord(p->ev[2], p->stream);
        if (it == 0 && !resume) {
            if (p->kind == S3O_KIND_BA) { if ((rc = ba_max_diag(p))) return rc; }
            else {
                launch_maxdiag(d, p->d_H, p->d_rowptr, nf, p->d_partials, p->d_sc, p->stream);
                if ((rc = check_launch(p, 1))) return rc;
            }
            if ((rc = allreduce_max(p, &p->d_sc->maxdiag, 1))) return rc;
            if ((rc = sync_scalars(p))) return rc;
            currentChi = p->h_sc->chi2;
            lambda = p->user_lambda > 0 ? p->user_lambda : p->tau * p->h_sc->maxdiag;
            ni = 2;
        }
        const double chi_start = currentChi;
        double rho = 0;
        int qmax = 0, pcg_total = 0;
        bool unresolved = false;
        do {
            cudaEventRecord(p->ev[3], p->stream);
            int status = 0, iters = 0;
            if (p->kind == S3O_KIND_BA) rc = ba_solve(p, lambda, &status, &iters, nullptr);
            else rc = do_solve(p, lambda, &status, &iters, nullptr, true);
            if (rc) return rc;
            pcg_total += iters;
            cudaEventRecord(p->ev[4], p->stream);
            const int trial = p->cur ^ 1;
            const double *xfull = p->d_x;
            if (p->dist) {   // every rank retracts all vertices from the gathered step
                if (comm_allgather(p->comm, p->d_x, p->d_xg, (size_t)p->plan.seg * d, p->stream)) {
                    set_error("%s", comm_last_error());
                    return S3O_ERR_NCCL;
                }
                xfull = p->d_xg;
            }
            if (p->kind == S3O_KIND_BA) {
                if ((rc = ba_retract_and_scale(p, lambda, trial))) return rc;
            } else {
                launch_retract(graph_view(p, p->cur), xfull, p->d_est[trial], p->stream);
                launch_scale(nf * d, p->d_x, p->d_b, lambda, p->d_partials, p->d_sc, p->stream);
                if ((rc = check_launch(p, 2))) return rc;
            }
            if ((rc = allreduce_sum(p, &p->d_sc->scale, 1))) return rc;
            if (p->dist && (rc = allreduce_max(p, &p->d_sc->xmax, 1))) return rc;
            if ((rc = do_chi2(p, trial))) return rc;
            cudaEventRecord(p->ev[5], p->stream);
            if ((rc = sync_scalars(p))) return rc;
            float ms = 0;
            cudaEventElapsedTime(&ms, p->ev[3], p->ev[4]); p->stats.ms_solve += ms; p->stats.sum_ms_solve += ms;
            cudaEventElapsedTime(&ms, p->ev[4], p->ev[5]); p->stats.ms_update += ms; p->stats.sum_ms_update += ms;
            if (status == 0) status = p->h_sc->done;     // exact solve: its verdict arrived with this read-back
            double tempChi = p->h_sc->chi2;
            const bool ok2 = status != 3;
            if (!ok2) tempChi = DBL_MAX;
            rho = currentChi - tempChi;
            double scale = p->h_sc->scale;
            scale += 1e-3;
            rho /= scale;
            // s3o_set_stop_rules: the predicted decrease of this step is below what the fp64 chi2 sums resolve, so
            // g2o's acceptance test would be decided by round-off (and so would that of every further trial).  The
            // quadratic model is exact to that precision here: take the step if chi2 stayed inside the noise band,
            // and stop.
            const bool unresolved_step = p->stop_pred > 0 && ok2 && p->h_sc->scale >= 0 && p->h_sc->scale < p->stop_pred * currentChi;
            if (unresolved_step && std::isfinite(tempChi) && tempChi - currentChi <= 10 * p->stop_pred * currentChi && !(rho > 0)) rho = 1e-300;
            if (rho > 0 && std::isfinite(tempChi)) {
                double alpha = 1. - std::pow((2 * rho - 1), 3);
                alpha = std::min(alpha, 2. / 3.);
                const double scaleFactor = std::max(1. / 3., alpha);
                lambda *= scaleFactor;
                ni = 2;
                currentChi = tempChi;
                p->cur = trial;            // discardTop: keep the updated estimates
                if (p->kind != S3O_KIND_BA) {
                    // distance left to the stationary point, from the linear convergence of the accepted steps:
                    // step_k * rho / (1 - rho) with rho = step_k / step_(k-1) (no estimate until the steps contract)
                    const double step = p->h_sc->xmax, prev = p->lm_prev_step;
                    const double ratio = prev > 0 ? step / prev : 1.0;
                    p->lm_est_dist = ratio < 0.5 ? step * ratio / (1.0 - ratio) : step;
                    p->lm_prev_step = step;
                    p->stats.last_step_inf = step;
                    p->stats.est_distance = p->lm_est_dist;
                }
            } else {
                lambda *= ni;              // pop: the current buffer still holds the old estimates
                ni *= 2;
            }
            qmax++;
            p->stats.lm_trials++;
            // the predicted decrease of this step is below what the chi2 sums can resolve: the acceptance test
            // above was decided by round-off, and so would be that of every further trial
            if (unresolved_step) { unresolved = true; break; }
        } while (rho < 0 && qmax < p->max_trials);
        {
            float ms = 0;
            cudaEventElapsedTime(&ms, p->ev[1], p->ev[2]);
            p->stats.ms_linearize += ms;
            p->stats.sum_ms_linearize += ms;
        }
        done = it + 1;
        p->stats.lm_iterations++;
        if (hist && it < hist_cap) {
            hist[it * 5 + 0] = currentChi; hist[it * 5 + 1] = lambda; hist[it * 5 + 2] = qmax;
            hist[it * 5 + 3] = rho; hist[it * 5 + 4] = pcg_total;
        }
        p->stats.stop_reason = 0;
        if (unresolved) { p->stats.stop_reason = 3; break; }
        if (qmax == p->max_trials || rho == 0) { result = S3O_RESULT_TERMINATE; p->stats.stop_reason = 4; break; }
        if (stop_rel_gain > 0) {
            const double gain = (chi_start - currentChi) / currentChi;
            if (gain >= 0 && gain < stop_rel_gain) { p->stats.stop_reason = 1; break; }
        }
        // step-size rule: the last accepted step moved no tangent component by more than stop_step
        // After an INEXACT solve (PCG forcing tolerance) the step can fall short of the Newton step in the modes the
        // preconditioner resolves worst, and the estimate with it (block-Jacobi at 0.2 stopped 1.3 mm early on the s10k
        // sphere): such solves have to meet the rule in two consecutive iterations.
        if (p->stop_step > 0 && rho > 0 && p->kind != S3O_KIND_BA) {
            const bool exact = (p->linsolver != S3O_LINSOLVER_PCG && !p->dist && direct_available(p)) || p->pcg_tol <= 1e-4;
            p->lm_stop_hits = p->lm_est_dist < p->stop_step ? p->lm_stop_hits + 1 : 0;
            if (p->lm_stop_hits >= (exact ? 1 : 2)) { p->stats.stop_reason = 2; break; }
        }
    }
    cudaEventRecord(p->ev[1], p->stream);
    S3O_CUDA(cudaStreamSynchronize(p->stream));
    {
        float ms = 0;
        cudaEventElapsedTime(&ms, p->ev[0], p->ev[1]);
        p->stats.ms_total = ms;
    }
    p->linearized = false;
    p->lm_valid = true; p->lm_lambda = lambda; p->lm_ni = ni; p->lm_chi = currentChi;
    if (iterations) *iterations = done;
    if (final_chi2) *final_chi2 = currentChi;
    if (final_lambda) *final_lambda = lambda;
    (void)result;
    return S3O_OK;
}

// Eigenvector of the smallest eigenvalue of H (the Gram matrix J^T Omega J at the current
// estimates) by inverse iteration  y = (H + shift I)^-1 x,  x = y / |y|  with the PCG solver, all
// vectors on the device.  This is the stepwise pipeline's scale initialisation
// (kitti_surf.cpp:887-934: last right singular vector of the scale-constraint matrix, whose Gram
// matrix is the Hessian of the 1-DoF scale graph with no vertex fixed).  lambda_max comes from a
// short power iteration and only feeds the reference's conditioning warning.
int s3o_smallest_eigenvector(s3o_problem *p, int max_iter, double tol, double *x, double *lambda_min,
                             double *lambda_max, int *iterations) {
    if (!p || !x) { set_error("s3o_smallest_eigenvector: bad arguments"); return S3O_ERR_INVALID; }
    if (p->dist || p->kind == S3O_KIND_BA) { set_error("s3o_smallest_eigenvector: not available for this problem"); return S3O_ERR_UNSUPPORTED; }
    if (p->scale_model != S3O_SCALE_MODEL_DIFFERENCE) {   // the reference's linear system (kitti_surf.cpp:897-906) is the DIFFERENCE rows
        set_error("s3o_smallest_eigenvector: defined on the S3O_SCALE_MODEL_DIFFERENCE rows");
        return S3O_ERR_UNSUPPORTED;
    }
    cudaSetDevice(p->device);
    int rc = ensure_built(p);
    if (rc) return rc;
    if (p->S.nf == 0) { set_error("s3o_smallest_eigenvector: 0 free vertices"); return S3O_ERR_INVALID; }
    if ((rc = do_linearize(p))) return rc;
    const int n = p->S.nf * p->d;
    const StructDev s = struct_view(p);
    launch_maxdiag(p->d, p->d_H, p->d_rowptr, p->S.nf, p->d_partials, p->d_sc, p->stream);
    if ((rc = check_launch(p, 1)) || (rc = sync_scalars(p))) return rc;
    const double maxdiag = p->h_sc->maxdiag;
    auto dot = [&](const double *a, const double *b, double *out) -> int {   // sum a_j b_j
        launch_scale(n, a, b, 0.0, p->d_partials, p->d_sc, p->stream);
        int r = check_launch(p, 1);
        if (r || (r = sync_scalars(p))) return r;
        *out = p->h_sc->scale;
        return S3O_OK;
    };
    // ---- largest eigenvalue: power iteration from an alternating-sign vector (d_r as x, d_z as y)
    double lmax = 0;
    launch_fill_alternating(n, p->d_r, p->stream);
    for (int it = 0; it < 30; ++it) {
        run_spmv(p, s, 0.0, p->d_r, 0);
        launch_finish_q(p->d, s, p->S.nf, p->d_q1, p->d_T, p->d_z, p->stream);
        if ((rc = check_launch(p, 2))) return rc;
        double yy = 0, xy = 0;
        if ((rc = dot(p->d_z, p->d_z, &yy)) || (rc = dot(p->d_z, p->d_r, &xy))) return rc;
        if (!(yy > 0)) break;
        lmax = xy;                                  // x normalised: Rayleigh quotient x^T H x
        launch_scale_vec(n, p->d_z, 1.0 / std::sqrt(yy), p->d_r, p->stream);
        p->stats.kernel_launches += 1;
    }
    // ---- smallest eigenvalue: inverse iteration (d_b holds the normalised iterate)
    // With the exact solver one factorisation serves every sweep; its shift stays well above the round-off of
    // a Cholesky factor (H itself is singular: the null vector is what is being computed), which still
    // contracts the error by shift / lambda_2 per sweep.
    bool exact = false;
    if (p->linsolver != S3O_LINSOLVER_PCG) {
        if ((rc = direct_setup(p))) return rc;
        exact = direct_available(p);
    }
    const double shift = (exact ? 1e-10 : 1e-13) * maxdiag;
    launch_fill_const(n, 1.0 / std::sqrt((double)n), p->d_b, p->stream);
    double theta = 0, theta_prev = -1;
    int done = 0;
    p->reuse_factor = true;
    for (int it = 0; it < std::max(max_iter, 1); ++it) {
        int status = 0;
        if ((rc = do_solve(p, shift, &status, nullptr, nullptr))) { p->reuse_factor = false; return rc; }
        if (status == 3) {
            p->reuse_factor = false;
            set_error("s3o_smallest_eigenvector: the linear solve of sweep %d broke down", it);
            return S3O_ERR_INVALID;
        }
        double yy = 0, xy = 0;
        if ((rc = dot(p->d_x, p->d_x, &yy)) || (rc = dot(p->d_x, p->d_b, &xy))) { p->reuse_factor = false; return rc; }
        if (!(yy > 0) || !std::isfinite(yy)) { p->reuse_factor = false; set_error("s3o_smallest_eigenvector: inverse iteration broke down"); return S3O_ERR_INVALID; }
        theta = xy / yy - shift;
        launch_scale_vec(n, p->d_x, 1.0 / std::sqrt(yy), p->d_b, p->stream);
        p->stats.kernel_launches += 1;
        done = it + 1;
        // exact sweeps: stop on the change of the Rayleigh quotient measured against the shift (theta itself
        // is ~0 for a null vector, so a relative test on it never settles)
        const double ref = exact ? std::max(std::fabs(theta), shift) : std::fabs(theta);
        if (it > 0 && std::fabs(theta - theta_prev) <= tol * ref) break;
        theta_prev = theta;
    }
    p->reuse_factor = false;
    direct_invalidate(p);
    S3O_CUDA(cudaMemcpyAsync(x, p->d_b, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    S3O_CUDA(cudaStreamSynchronize(p->stream));
    p->stats.d2h_bytes += (int64_t)n * 8;
    p->linearized = false;                          // b was overwritten
    if (lambda_min) *lambda_min = theta;
    if (lambda_max) *lambda_max = lmax;
    if (iterations) *iterations = done;
    return S3O_OK;
}

// Marginal covariances (g2o SparseOptimizer::computeMarginals): H = J^T Omega' J at the current estimates, factorised
// without damping, and its selected inverse (direct.cu).
int s3o_compute_marginals(s3o_problem *p, int n_pairs, const int32_t *rows, const int32_t *cols, double *out) {
    if (!p || n_pairs < 0 || (!rows != !cols) || (n_pairs > 0 && !out)) { set_error("s3o_compute_marginals: bad arguments"); return S3O_ERR_INVALID; }
    if (p->dist || (p->kind != S3O_KIND_SIM3 && p->kind != S3O_KIND_SCALE_TRANS && p->kind != S3O_KIND_SCALE)) {
        set_error("s3o_compute_marginals: pose-graph kinds on one GPU only (not bundle adjustment, the partitioned solve or a linear-solver handle)");
        return S3O_ERR_UNSUPPORTED;
    }
    cudaSetDevice(p->device);
    int rc = ensure_built(p);
    if (rc) return rc;
    const int nf = p->S.nf;
    if (nf == 0) { set_error("s3o_compute_marginals: 0 free vertices"); return S3O_ERR_INVALID; }
    if (!rows && n_pairs != nf) { set_error("s3o_compute_marginals: the diagonal blocks need n_pairs = n_free = %d", nf); return S3O_ERR_INVALID; }
    for (int k = 0; rows && k < n_pairs; ++k)
        if (rows[k] < 0 || rows[k] >= nf || cols[k] < 0 || cols[k] >= nf) {
            set_error("s3o_compute_marginals: pair %d (%d, %d) is not a pair of Hessian indices in [0, %d) (fixed vertices have none)",
                      k, rows[k], cols[k], nf);
            return S3O_ERR_INVALID;
        }
    // H is singular when a connected component holds no fixed vertex (its gauge is free)
    {
        std::vector<int32_t> root(p->nv);
        for (int v = 0; v < p->nv; ++v) root[v] = v;
        auto find = [&](int v) { while (root[v] != v) v = root[v] = root[root[v]]; return v; };
        for (int e = 0; e < p->ne; ++e) {
            const int a = find(p->v0[e]), b = find(p->v1[e]);
            if (a != b) root[std::max(a, b)] = std::min(a, b);
        }
        std::vector<uint8_t> anchored(p->nv, 0);
        for (int v = 0; v < p->nv; ++v) if (p->fixed[v]) anchored[find(v)] = 1;
        for (int v = 0; v < p->nv; ++v)
            if (!anchored[find(v)]) {
                set_error("s3o_compute_marginals: the Hessian is singular: the connected component of vertex %d has no fixed vertex", v);
                return S3O_ERR_SOLVE;
            }
    }
    // the selected inverse of the sparse Cholesky factor, or PCG solves of the requested block columns where that
    // factor exceeds the forced cap (marginals_pcg.cu)
    bool iterative = false;
    if ((rc = marginals_iterative(p, &iterative))) return rc;
    cudaEventRecord(p->ev[0], p->stream);
    if ((rc = do_linearize(p))) return rc;
    cudaEventRecord(p->ev[1], p->stream);
    rc = iterative ? pcg_marginals(p, n_pairs, rows, cols, out, p->ev + 2) : direct_marginals(p, n_pairs, rows, cols, out, p->ev + 2);
    direct_invalidate(p);
    p->linearized = false;          // as after s3o_optimize: the next solve linearises again
    if (rc) return rc;
    if (getenv("S3O_MARGINALS_TRACE")) {     // per-phase CUDA-event times (tools/marginals_probe.py)
        float ms[4] = {};
        for (int k = 0; k < 4; ++k) cudaEventElapsedTime(&ms[k], p->ev[k], p->ev[k + 1]);
        if (iterative)
            fprintf(stderr, "s3o_compute_marginals: linearize %.4f precond %.4f solves %.4f symmetrize %.4f ms\n", ms[0], ms[1], ms[2], ms[3]);
        else
            fprintf(stderr, "s3o_compute_marginals: linearize %.4f factor %.4f selinv %.4f gather %.4f ms\n", ms[0], ms[1], ms[2], ms[3]);
    }
    return S3O_OK;
}

int s3o_get_vertices(s3o_problem *p, double *est) {
    if (p && p->kind == S3O_KIND_BA) { set_error("s3o_get_vertices: a BA problem takes s3o_ba_get_cameras / s3o_ba_get_points"); return S3O_ERR_INVALID; }
    if (!p || !est || !p->d_est[0]) { set_error("s3o_get_vertices: no vertices"); return S3O_ERR_INVALID; }
    cudaSetDevice(p->device);
    const size_t cnt = (size_t)p->nv * p->est_dim;
    int rc = ensure_stage(p);
    if (rc) return rc;
    double *tmp = p->d_stage;
    launch_unpack_vertices(p->d_est[p->cur], p->nv, p->nv_pad, p->est_dim, tmp, p->stream);
    cudaError_t e = cudaMemcpyAsync(est, tmp, cnt * sizeof(double), cudaMemcpyDeviceToHost, p->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(p->stream);
    if (e != cudaSuccess) { set_error("s3o_get_vertices: %s", cudaGetErrorString(e)); return S3O_ERR_CUDA; }
    p->stats.d2h_bytes += (int64_t)(cnt * sizeof(double));
    p->stats.kernel_launches += 1;
    return S3O_OK;
}

int s3o_set_lm_resume(s3o_problem *p, int resume) {
    if (!p) return S3O_ERR_INVALID;
    if (resume < 0 || resume > 2) { set_error("s3o_set_lm_resume: mode must be 0, 1 or 2"); return S3O_ERR_INVALID; }
    p->lm_resume = resume;
    return S3O_OK;
}

int s3o_snapshot_estimates(s3o_problem *p) {
    if (p && p->kind == S3O_KIND_BA) { cudaSetDevice(p->device); int rc = ensure_built(p); return rc ? rc : ba_snapshot(p, 0); }
    if (!p || !p->d_est[0]) { set_error("s3o_snapshot_estimates: no vertices"); return S3O_ERR_INVALID; }
    cudaSetDevice(p->device);
    const size_t cnt = (size_t)p->nv_pad * p->est_dim;
    if (!p->d_est_snap) { int rc = dev_alloc(&p->d_est_snap, cnt); if (rc) return rc; }
    S3O_CUDA(cudaMemcpyAsync(p->d_est_snap, p->d_est[p->cur], cnt * sizeof(double), cudaMemcpyDeviceToDevice, p->stream));
    return S3O_OK;
}

int s3o_restore_estimates(s3o_problem *p) {
    if (p && p->kind == S3O_KIND_BA) {
        cudaSetDevice(p->device);
        p->linearized = false;
        p->lm_valid = false;
        return ba_snapshot(p, 1);
    }
    if (!p || !p->d_est_snap) { set_error("s3o_restore_estimates: no snapshot"); return S3O_ERR_INVALID; }
    cudaSetDevice(p->device);
    const size_t cnt = (size_t)p->nv_pad * p->est_dim;
    S3O_CUDA(cudaMemcpyAsync(p->d_est[p->cur], p->d_est_snap, cnt * sizeof(double), cudaMemcpyDeviceToDevice, p->stream));
    p->linearized = false;
    p->lm_valid = false;
    p->auto_multilevel = false;     // a new solve starts: AUTO decides again (keeps solves reproducible)
    return S3O_OK;
}

int s3o_get_stats(s3o_problem *p, s3o_stats *out) {
    if (!p || !out) return S3O_ERR_INVALID;
    p->stats.n_vertices = p->nv; p->stats.dim = p->d;
    if (p->kind != S3O_KIND_BA) p->stats.n_edges = p->ne;
    p->stats.n_free = p->built ? p->S.nf : 0;
    p->stats.n_blocks = p->built ? p->S.nb : 0;
    p->stats.multilevel_levels = amg_levels(p);
    amg_counts(p, &p->stats.multilevel_rebuilds, &p->stats.multilevel_reuses);
    p->stats.p2p_halo = p->p2p ? 1 : 0;
    *out = p->stats;
    return S3O_OK;
}

int s3o_reset_stats(s3o_problem *p) {
    if (!p) return S3O_ERR_INVALID;
    p->stats = s3o_stats{};
    amg_counts(p, nullptr, nullptr);        // zeroes them
    return S3O_OK;
}

int s3o_estimate_sigma_squared(s3o_problem *p, int robust_kind, double *sigma_squared) {
    if (!p || !sigma_squared) return S3O_ERR_INVALID;
    if (p->kind == S3O_KIND_BA) { set_error("s3o_estimate_sigma_squared: pose-graph kinds only"); return S3O_ERR_UNSUPPORTED; }
    cudaSetDevice(p->device);
    int rc = ensure_built(p);
    if (rc) return rc;
    const int na = p->S.ne_act, d = p->d;
    double *d_err = nullptr, *d_chi = nullptr;
    if ((rc = dev_alloc(&d_err, (size_t)na * d))) return rc;
    if ((rc = dev_alloc(&d_chi, (size_t)na))) { cudaFree(d_err); return rc; }
    launch_edge_errors(graph_view(p, p->cur), d_err, d_chi, p->stream);
    std::vector<double> chi(na);
    cudaError_t e = cudaMemcpyAsync(chi.data(), d_chi, sizeof(double) * na, cudaMemcpyDeviceToHost, p->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(p->stream);
    cudaFree(d_err); cudaFree(d_chi);
    if (e != cudaSuccess) { set_error("s3o_estimate_sigma_squared: %s", cudaGetErrorString(e)); return S3O_ERR_CUDA; }
    p->stats.kernel_launches += 1;
    if (na == 0) { *sigma_squared = 0; return S3O_OK; }
    if (robust_kind == S3O_ROBUST_PTAM_LS) {       // MEstimator.h:190-198
        double sum = 0;
        for (double c : chi) sum += c;
        *sigma_squared = sum / na;
        return S3O_OK;
    }
    // MEstimator.h:79-89 / :113-123 / :157-167: median of the sorted squared errors
    std::nth_element(chi.begin(), chi.begin() + na / 2, chi.end());
    const double med = chi[na / 2];
    double sigma = 1.4826 * (1 + 5.0 / (na * 2 - 6)) * std::sqrt(med);
    sigma *= (robust_kind == S3O_ROBUST_PTAM_HUBER) ? 1.345 : 4.6851;
    *sigma_squared = sigma * sigma;
    return S3O_OK;
}

}  // extern "C"
