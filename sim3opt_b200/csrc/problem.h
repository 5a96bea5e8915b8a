// problem.h -- the s3o_problem object and the host-side helpers shared by problem.cu and ba.cu.
#pragma once
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "comm.h"
#include "internal.h"
#include "kernels.cuh"
#include "gridbar.cuh"

namespace s3o {

template <class T>
int dev_alloc(T **ptr, size_t count) {
    *ptr = nullptr;
    if (count == 0) count = 1;
    S3O_CUDA(cudaMalloc((void **)ptr, count * sizeof(T)));
    return S3O_OK;
}
template <class T>
void dev_free(T *&ptr) {
    if (ptr) cudaFree(ptr);
    ptr = nullptr;
}

struct BaState;   // bundle adjustment (ba.cu)
struct AmgState;  // multilevel preconditioner (amg.cu)
struct DirectState;  // sparse block Cholesky (direct.cu)
struct DirectPlan;   // its symbolic analysis (direct.h)

// kind of the handle behind s3o_linsolver_*: a block system only (no graph, no estimates)
constexpr int kKindLinear = 100;

}  // namespace s3o

using s3o::Comm;
using s3o::DevScalars;
using s3o::HostStructure;
using s3o::PartitionPlan;

struct s3o_problem {
    int kind = 0, d = 0, est_dim = 0, ninfo = 0, device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    // host-side graph description
    int nv = 0, ne = 0;
    std::vector<uint8_t> fixed;
    std::vector<int32_t> v0, v1;
    bool has_info = false, has_aux = false, info_diag = false;
    // caller-ordered staging of the edge records until the structure is built; on a built problem, of the edges
    // appended since (s3o_add_edges), until the next build merges them.  has_info / info_diag describe the staged
    // records and, once merged or built, the whole graph
    double *d_meas_aos = nullptr, *d_info_aos = nullptr;
    // device graph
    int nv_pad = 0, ne_pad = 0;
    double *d_est[2] = { nullptr, nullptr };
    int cur = 0;
    double *d_aux = nullptr;
    int32_t *d_hidx = nullptr, *d_sv0 = nullptr, *d_sv1 = nullptr;
    double *d_meas = nullptr, *d_info = nullptr;
    // structure
    HostStructure S;
    bool built = false;
    int32_t *d_rowptr = nullptr, *d_colidx = nullptr, *d_blk_row = nullptr, *d_blk_ebeg = nullptr, *d_blk_eend = nullptr;
    int32_t *d_colT_ptr = nullptr, *d_colT_blk = nullptr, *d_inc_ptr = nullptr, *d_inc_ent = nullptr, *d_e_blk = nullptr;
    int32_t *d_tile_row = nullptr;
    int32_t *d_blk_src = nullptr, *d_multi_blk = nullptr;
    int32_t *d_perm = nullptr;              // [ne_act] sorted position -> caller edge (read by the merge)
    int built_info_rep = 0;                 // information in d_info: 0 none, 1 diagonal planes, 2 packed triangles
    // partitioned solve (one process per GPU, NCCL): s3o_set_comm
    Comm comm;
    bool dist = false;
    PartitionPlan plan;
    int user_ne = 0;                       // edges passed by the caller (plan.local_edges index into them)
    std::vector<int32_t> gv0, gv1;         // all edges' endpoints (the multilevel hierarchy is built on the global graph)
    int32_t *d_ghidx = nullptr, *d_send_idx = nullptr;
    uint8_t *d_primary = nullptr;
    double *d_sendbuf = nullptr, *d_xg = nullptr;
    // peer-to-peer halo (NVLink loads inside the SpMV instead of pack + NCCL send/recv): CUDA IPC mappings of
    // the neighbours' p vectors and epoch flags
    bool p2p = false, want_p2p_setup = false;
    long long halo_epoch = 0;
    long long *d_flag = nullptr;               // my epoch flag (mapped by the neighbours)
    double **d_ghost_src = nullptr;            // [n_ghost] address of every ghost column inside its owner's p
    long long **d_peer_flags = nullptr;        // [n_peers] the neighbours' flags
    int n_peers = 0;
    std::vector<void *> ipc_mapped;            // to cudaIpcCloseMemHandle
    int spmv_version = 4;       // 1: lane-group rows, 2: tiled thread-per-block, 3: v2 + TMA ring, 4: v3 + prefetch pipeline (d = 7)
    int spmv_grid_cap = 148 * 2;            // persistent SpMV grid; S3O_SPMV_GRID in [1, kMaxPartials]
    int spmv4_cfg = 0;          // v4 tile / ring: 0: TB=112 NS=2, 1: TB=80 NS=3, 2: TB=56 NS=4; fixes the tiles of this problem
    // linear system
    double *d_H = nullptr, *d_b = nullptr, *d_x = nullptr, *d_r = nullptr, *d_z = nullptr, *d_p = nullptr;
    double *d_q1 = nullptr, *d_T = nullptr, *d_Minv = nullptr, *d_scratch = nullptr, *d_partials = nullptr;
    DevScalars *d_sc = nullptr, *h_sc = nullptr;
    unsigned *d_gridbar = nullptr;          // [0] arrival counter of the persistent kernels' grid barrier, [1] abort flag
    bool coop_launch = false;               // S3O_COOP_LAUNCH=1: cudaLaunchCooperativeKernel instead of the counter barrier
    // parameters
    int robust_kind = S3O_ROBUST_NONE;
    double robust_param = 0;
    int math_mode = S3O_MATH_REFERENCE;
    int scale_model = S3O_SCALE_MODEL_DIFFERENCE;      // s3o_set_scale_model
    int jac_mode = S3O_JAC_ANALYTIC;
    double jac_h = 1e-9;
    double tau = 1e-5, user_lambda = 0;
    int max_trials = 10;
    double stop_step = 0, stop_pred = 0;    // s3o_set_stop_rules
    double pcg_tol = 1e-8;
    int pcg_max_iter = 1000;
    int last_pcg_iters = 0;                 // iterations of the previous PCG solve (sizes the first launch batch)
    int precond = S3O_PRECOND_AUTO;         // s3o_set_preconditioner
    bool auto_multilevel = false;           // AUTO: a block-Jacobi solve needed > 256 iterations
    bool linearized = false;
    // LM continuation state (s3o_set_lm_resume)
    int lm_resume = 0;
    bool lm_valid = false;
    double lm_lambda = 0, lm_ni = 2, lm_chi = 0;
    double lm_prev_step = 0, lm_est_dist = 0;   // step-size stop rule: previous accepted step, estimated distance left
    int lm_stop_hits = 0;                       // consecutive accepted iterations that met the step-size rule
    double *d_est_snap = nullptr;
    double *d_stage = nullptr;             // AoS staging of the estimates (upload / download)
    // sampled SpMV timing
    static constexpr int kSpmvEvents = 64;
    cudaEvent_t spmv_ev[2 * kSpmvEvents] = {};
    int spmv_ev_used = 0;
    int spmv_ev_iter[kSpmvEvents] = {};     // PCG iteration (launch index within the solve) of each sample
    // statistics
    s3o_stats stats{};
    cudaEvent_t ev[8] = {};
    // bundle adjustment (kind S3O_KIND_BA): cameras / points / observations live in ba.cu
    s3o::BaState *ba = nullptr;
    // multilevel preconditioner of the pose-graph PCG (amg.cu), built on first use
    s3o::AmgState *amg = nullptr;
    // exact solve: sparse block Cholesky on the device (direct.cu), built on first use
    s3o::DirectState *direct = nullptr;
    int linsolver = S3O_LINSOLVER_AUTO;     // s3o_set_linear_solver
    bool reuse_factor = false;              // repeated solves with one matrix (inverse iteration)
    // S3O_TRACE=1: CUDA-event timeline of ONE PCG iteration (the 5th of a solve), printed to stderr
    std::vector<std::pair<const char *, cudaEvent_t>> trace;
    int trace_state = 0, trace_solve = 0;   // 0 off, 1 armed, 2 recording, 3 done; solves left before recording
};

namespace s3o {

template <class T>
int upload(s3o_problem *p, T **dst, const std::vector<T> &src) {
    int rc = dev_alloc(dst, src.size());
    if (rc) return rc;
    if (!src.empty()) {
        S3O_CUDA(cudaMemcpyAsync(*dst, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice, p->stream));
        p->stats.h2d_bytes += (int64_t)(src.size() * sizeof(T));
    }
    return S3O_OK;
}

StructDev struct_view(const s3o_problem *p);
void free_structure(s3o_problem *p);
void close_p2p(s3o_problem *p);
int check_launch(s3o_problem *p, int n);
int sync_scalars(s3o_problem *p);
int upload_structure_arrays(s3o_problem *p, int rows_own, bool on_device = false);   // BSR / tile arrays of p->S -> device
int alloc_linear_system(s3o_problem *p);                      // H, b, x, r, z, p, q1, T, Minv for p->S
// Solve (H + lambda I) x = b on the system held in p->d_H / p->d_b; x in p->d_x.  Sparse block Cholesky when the
// factor is small (s3o_set_linear_solver), PCG otherwise.  defer_sync: the exact path does not wait for the
// device; *status stays 0 and the caller reads DevScalars::done after its own sync_scalars.
int do_solve(s3o_problem *p, double lambda, int *status, int *iters, double *rel_res, bool defer_sync = false);
// The PCG of do_solve in two steps, shared with the iterative marginals: pcg_prepare forms the block-Jacobi inverses
// of (H + lambda I) and, when amg, the multilevel operators; pcg_iterate solves (H + lambda I) x = p->d_b from x = 0
// into p->d_x, to the relative recurrence residual tol or max_iter iterations, and leaves its verdict in p->h_sc.
int pcg_prepare(s3o_problem *p, double lambda, bool amg);
int pcg_iterate(s3o_problem *p, double lambda, bool amg, double tol, int max_iter);
void hessian_product(s3o_problem *p, const double *x);   // q1 and T of H x (lambda = 0; completed by the column owner)

// ---- sparse block Cholesky (direct.cu, direct_host.cpp) ---------------------------------------
int direct_setup(s3o_problem *p);                     // symbolic analysis + upload, once per structure
bool direct_available(const s3o_problem *p);          // false: the factor would be too large, use PCG
int direct_solve(s3o_problem *p, double lambda, bool reuse_factor);
void direct_invalidate(s3o_problem *p);               // H changed
void direct_destroy(s3o_problem *p);
// read-outs for tests (s3o_direct_schedule, s3o_get_direct_factor): the plan the factorisations run on -- the linear
// solver's, else the marginals' -- and the factor its last numeric factorisation left
int direct_schedule(s3o_problem *p, int32_t *info, int cap);
int direct_read_factor(s3o_problem *p, double *L, double *Linv);
// Marginal covariances: blocks (rows[k], cols[k]) of H^-1 (Hessian indices, validated by the caller) for the H in
// p->d_H, into out (n_pairs x d x d); rows == cols == nullptr: the n_pairs = n_free diagonal blocks.  Factorises H on
// the linear solver's plan, or on a plan under the forced cap kept for the marginals (the choice of the linear solver
// does not change), then runs the selected inverse.  Leaves p->d_b / p->d_x / p->d_sc untouched and no factor held.
// ev (may be nullptr): 3 events recorded after the factorisation, the selected inverse and the gather.  Errors are
// reported as "<who>: ..." (the C-ABI entry that called it).
int direct_marginals(s3o_problem *p, const char *who, int n_pairs, const int32_t *rows, const int32_t *cols, double *out,
                     cudaEvent_t *ev);
// The same call in steps, so that the BA marginals (ba.cu) can run their point phase on the selected inverse:
//   marginals_open    plan choice, first-call buffers and gather lists, the requested pairs' lists (host + upload);
//                     errors are reported as "<who>: ..."
//   marginals_factor  factorisation of p->d_H without damping and the selected inverse (launches; ev: 2 events)
//   marginals_pick    the requested blocks into run.out, [n_pairs][d*d] (launches)
// *fail is set on the device when a pivot fails.  serial identifies the plan: gather lists built on run.plan elsewhere
// stay valid while it does not change.
struct MarginalsRun {
    DirectState *S = nullptr;
    const DirectPlan *plan = nullptr;
    uint64_t serial = 0;
    const double *Sig = nullptr;     // [nL][d*d] selected inverse, laid out like L (elimination order)
    const double *out = nullptr;
    const int *fail = nullptr;
};
int marginals_open(s3o_problem *p, const char *who, int n_pairs, const int32_t *rows, const int32_t *cols, MarginalsRun *run);
int marginals_factor(s3o_problem *p, const MarginalsRun &run, cudaEvent_t *ev);
int marginals_pick(s3o_problem *p, const MarginalsRun &run, int n_pairs);
// Which route serves a pose-graph marginals call: the iterative one (*iterative) when the factor exceeds the forced
// cap, or when S3O_MARGINALS_ROUTE=pcg asks for it.
int marginals_iterative(s3o_problem *p, bool *iterative);
// Iterative route (marginals_pcg.cu): for each distinct column vertex c of the explicit pairs, d PCG solves
// H x = e_(c,m) without damping, refined until the true residual |e - H x| <= S3O_MARGINALS_PCG_TOL.  Reuses the LM's
// PCG work vectors and scalars; puts back what the LM carries across calls and the solver statistics.  ev (may be
// nullptr): 3 events recorded after the preconditioner set-up, the solves and the gather.  Preconditioner: multilevel
// for the pose-graph kinds under the difference scale model, block-Jacobi otherwise (a linear-solver handle has no
// estimates to build a hierarchy on).  Errors are reported as "<who>: ...".
int pcg_marginals(s3o_problem *p, const char *who, int n_pairs, const int32_t *rows, const int32_t *cols, double *out,
                  cudaEvent_t *ev);
// Launches a persistent kernel whose CTAs synchronise through grid_barrier (gridbar.cuh).  The kernel's LAST argument
// is a GridBarrier; args[nargs - 1] must point to a GridBarrier that this call fills.
inline int launch_persistent(s3o_problem *p, const void *func, int grid, int block, void **args, int nargs, size_t smem = 0) {
    GridBarrier *gb = (GridBarrier *)args[nargs - 1];
    gb->counter = p->d_gridbar;
    gb->abort = (int *)(p->d_gridbar + 1);
    gb->cooperative = p->coop_launch ? 1 : 0;
    if (p->coop_launch) {
        S3O_CUDA(cudaLaunchCooperativeKernel(func, dim3(grid), dim3(block), args, smem, p->stream));
        return S3O_OK;
    }
    S3O_CUDA(cudaMemsetAsync(p->d_gridbar, 0, sizeof(unsigned), p->stream));
    S3O_CUDA(cudaLaunchKernel(func, dim3(grid), dim3(block), args, smem, p->stream));
    return S3O_OK;
}
inline void trace_mark(s3o_problem *p, const char *what) {
    if (p->trace_state != 2) return;
    cudaEvent_t e;
    cudaEventCreate(&e);
    cudaEventRecord(e, p->stream);
    p->trace.push_back({ what, e });
}

// ---- multilevel preconditioner (amg.cu) -------------------------------------------------------
bool wants_multilevel(const s3o_problem *p);
int amg_setup(s3o_problem *p);                        // hierarchy for p->S (host build + upload)
void amg_destroy(s3o_problem *p);
int amg_levels(const s3o_problem *p);                 // coarse levels (0: graph too small, block-Jacobi only)
void amg_counts(const s3o_problem *p, int64_t *rebuilds, int64_t *reuses);
void amg_invalidate_frames(s3o_problem *p);           // the linearisation point moved
int amg_update_frames(s3o_problem *p);
int amg_update_values(s3o_problem *p, double lambda); // Galerkin operators for (H + lambda I)
int amg_apply(s3o_problem *p, int init, double tol, int max_iter);   // z += P0 V(P0^T r), r.z and the PCG scalars
void amg_set_counts(s3o_problem *p, int64_t rebuilds, int64_t reuses);
// read-outs for tests (layouts: include/sim3opt_b200.h, s3o_multilevel_prepare and s3o_get_multilevel_*)
int amg_plan_info(const s3o_problem *p, bool active, int32_t *info, int cap);
int amg_read_level(s3o_problem *p, int level, int32_t *agg, int32_t *root_vid, int32_t *rowptr, int32_t *colidx,
                   double *A, double *Dinv, double *rel);
int amg_read_coarsest_inverse(s3o_problem *p, double *inv);

// ---- bundle adjustment hooks (ba.cu), called from the C ABI in problem.cu --------------------
void ba_destroy(s3o_problem *p);
int ba_build_structure(s3o_problem *p);
int ba_chi2(s3o_problem *p, int which);
int ba_linearize(s3o_problem *p);
int ba_max_diag(s3o_problem *p);
int ba_solve(s3o_problem *p, double lambda, int *status, int *iters, double *rel_res);   // full step in ba->d_x
int ba_retract_and_scale(s3o_problem *p, double lambda, int trial);
int ba_upload_step(s3o_problem *p, const double *x);
int ba_download_step(s3o_problem *p, double *x);
int ba_snapshot(s3o_problem *p, int restore);

}  // namespace s3o
