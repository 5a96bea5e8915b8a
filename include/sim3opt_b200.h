/*
 * sim3opt_b200.h -- C ABI of the B200-native Sim3 / SE3 nonlinear least-squares back-end.
 *
 * This is the drop-in boundary (SURVEY.md section 8b): everything the reference does through
 * g2o between "graph is built" and "estimates are read back" goes through these calls.
 *
 *   reference call site (kitti_surf.cpp)                         replacement
 *   ------------------------------------------------------------ ---------------------------
 *   new OptimizationAlgorithmLevenberg(BlockSolverX(LinearSolverEigen))  :552-558,:726-735
 *                                                                 s3o_create / s3o_set_lm / s3o_set_pcg
 *   optimizer.addVertex(VertexSim3Expmap: setEstimate,setFixed)  :597-622   s3o_set_vertices
 *   optimizer.addEdge(EdgeSim3: setVertex,setMeasurement,information) :624-670  s3o_set_edges
 *   optimizer.initializeOptimization()                           :674       s3o_build_structure
 *   optimizer.optimize(100)                                      :675       s3o_optimize
 *   vSim3->estimate()                                            :688-689   s3o_get_vertices
 *   G2oVertexScaleTrans / G2oEdgeScaleTrans graph                :779-884   kind S3O_KIND_SCALE_TRANS
 *   edge->setRobustKernel(RobustKernelHuber, delta)   bal_example.cpp:149-153   s3o_set_robust
 *
 * Conventions
 *   - plain pointers and sizes only; all array arguments are HOST pointers borrowed for the
 *     duration of the call (copied to the device inside); results are copied into caller buffers.
 *   - every function returns 0 on success or a negative s3o_status; s3o_last_error() gives text.
 *     Nothing throws across this boundary.  There is no CPU fallback: without a CUDA device
 *     s3o_create fails with S3O_ERR_CUDA.
 *   - Sim3 state   : 8 doubles [qx qy qz qw tx ty tz s] (g2o::Sim3: x -> s*(R x) + t)
 *     tangent      : 7 doubles [omega upsilon sigma] (g2o order)
 *     scale-trans  : 4 doubles [s tx ty tz], aux = fixed rotation quaternion [qx qy qz qw]
 *     matrices     : row-major
 *   - one host thread per problem; distinct problems are independent (SURVEY.md 8b "Threading").
 */
#ifndef SIM3OPT_B200_H
#define SIM3OPT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct s3o_problem s3o_problem;

enum s3o_status {
    S3O_OK = 0,
    S3O_ERR_INVALID = -1,   /* bad argument / call order */
    S3O_ERR_CUDA = -2,      /* CUDA runtime failure (no device, OOM, launch error) */
    S3O_ERR_NCCL = -3,
    S3O_ERR_IO = -4,
    S3O_ERR_UNSUPPORTED = -5,
    S3O_ERR_SOLVE = -6      /* the linear solve failed: matrix not positive definite (pivot / PCG breakdown) or the PCG
                               hit its iteration cap -- g2o's LinearSolver::solve() == false */
};

enum s3o_kind { S3O_KIND_SIM3 = 0, S3O_KIND_SCALE_TRANS = 1, S3O_KIND_SCALE = 2, S3O_KIND_BA = 3 };
enum s3o_jacobian { S3O_JAC_NUMERIC = 0, S3O_JAC_ANALYTIC = 1 };
/* robust kernels: g2o RobustKernelHuber (param = delta) and the PTAM M-estimators of
 * MEstimator.h:54-198 (param = sigma squared) */
enum s3o_robust { S3O_ROBUST_NONE = 0, S3O_ROBUST_HUBER = 1, S3O_ROBUST_PTAM_TUKEY = 2,
                  S3O_ROBUST_PTAM_CAUCHY = 3, S3O_ROBUST_PTAM_HUBER = 4, S3O_ROBUST_PTAM_LS = 5 };
/* Sim3 exp/log small-angle coefficients.  REFERENCE (default): exactly as written at
 * sim3_rv.h:143-181,:261-303 -- including B = ((sigma^2/2 - sigma + 1) s)/sigma^3 (no "-1") in the
 * theta<eps, |sigma|>=eps branch and R = I + Om + Om^2 -- which is what the reference's pinned g2o
 * computes.  CORRECTED: the consistent Taylor limits (B with "-1", R = I + Om + Om^2/2).  The
 * as-written B is O(1/sigma^3) off, which makes the objective discontinuous whenever a residual
 * rotation drops below 4.5e-3 rad while sigma != 0; graphs that must converge to a minimum
 * (the synthetic configs) are run in CORRECTED mode on both the CPU and the GPU side. */
enum s3o_math_mode { S3O_MATH_REFERENCE = 0, S3O_MATH_CORRECTED = 1 };
/* [EXT vio_g2o] G2oEdgeScale / G2oEdgeScaleTrans (kitti_surf.cpp:827-847, :865-884) are not in the reference tree, and
 * vio_g2o is cloned unpinned (build.sh:92), so their error form and the vertices' oplus are restated from the
 * reference's call sites (SURVEY.md row a18).  Both plausible readings are implemented and selectable:
 *   DIFFERENCE (default): e_s = s_ji s_i - s_j (the rows of the reference's own linear system, :897-906), s <- s + d
 *   LOGRATIO:             e_s = log(s_ji s_i / s_j),                                                      s <- s exp(d)
 * The translation rows t_j - (s_j/s_i) R_j R_i^T t_i - t_ji (:969-985) and t <- t + d are common to both.  The
 * scale null-vector stage (s3o_smallest_eigenvector) is defined on the DIFFERENCE rows. */
enum s3o_scale_model { S3O_SCALE_MODEL_DIFFERENCE = 0, S3O_SCALE_MODEL_LOGRATIO = 1 };
/* Preconditioner of the PCG that stands in for LinearSolverEigen::solve [EXT g2o] (the plug-in slot
 * filled at kitti_surf.cpp:553-558).  BLOCK_JACOBI: (H_ii + lambda I)^-1 per vertex.  MULTILEVEL:
 * block-Jacobi plus an aggregation coarse-space correction on the gauge near-null space
 * of the graph (Sim3: delta_i = Ad(S_i S_root^-1) xi; scale-trans: (s_i/s_root) diag(1, R_i R_root^T);
 * scale: s_i/s_root); pose-graph kinds only, also in the partitioned solve (Sim3).  AUTO (default):
 * MULTILEVEL for graphs with >= 20000 free vertices; smaller Sim3 / scale-trans graphs start with
 * BLOCK_JACOBI, switch to MULTILEVEL once a solve has needed more than 256 PCG iterations, and back
 * when a MULTILEVEL solve finishes within 8.  Naming BLOCK_JACOBI or MULTILEVEL also selects the PCG as the linear
 * solver (s3o_set_linear_solver) unless the caller has chosen one. */
enum s3o_preconditioner { S3O_PRECOND_AUTO = 0, S3O_PRECOND_BLOCK_JACOBI = 1, S3O_PRECOND_MULTILEVEL = 2 };
/* Linear solver behind BlockSolver::solve (the LinearSolverEigen slot, kitti_surf.cpp:553-557).  DIRECT: sparse
 * block Cholesky on the device -- symbolic analysis once per structure (multiple-minimum-degree order whose
 * elimination rounds are the parallel schedule), numeric factorisation + triangular solves per LM trial in one
 * kernel; exact like the reference's LDL^T.  PCG: preconditioned conjugate gradients (s3o_set_pcg,
 * s3o_set_preconditioner).  AUTO (default): DIRECT when the factor is small and shallow (<= 400 000 block
 * products, <= 128 elimination rounds: the KITTI-size chain-dominated graphs of the reference, banded BA Schur
 * systems), PCG otherwise and
 * always in the partitioned solve. */
enum s3o_linear_solver { S3O_LINSOLVER_AUTO = 0, S3O_LINSOLVER_PCG = 1, S3O_LINSOLVER_DIRECT = 2 };
/* g2o OptimizationAlgorithm::SolverResult */
enum s3o_solver_result { S3O_RESULT_TERMINATE = 2, S3O_RESULT_OK = 1, S3O_RESULT_FAIL = -1 };

const char *s3o_last_error(void);
int s3o_version(void);
int s3o_device_count(void);

/* ---- lifetime ------------------------------------------------------------------------- */
int s3o_create(int kind, int device, s3o_problem **out);
int s3o_destroy(s3o_problem *p);
/* run all work of this problem on an existing CUDA stream (cudaStream_t passed as void*);
 * NULL = a private non-blocking stream created by s3o_create */
int s3o_set_stream(s3o_problem *p, void *cuda_stream);

/* ---- partitioned solve across the GPUs of one box (SURVEY.md section 8e) -----------------
 * One process per GPU.  Rank 0 obtains a 128-byte NCCL unique id, the host program broadcasts it
 * (e.g. torch.distributed), and every rank calls s3o_set_comm BEFORE s3o_set_edges.  Every rank
 * passes the SAME full vertex and edge arrays; the library keeps the rows of the free-vertex range
 * it owns (rank r owns Hessian indices [r*seg, (r+1)*seg), seg = ceil(n_free/world)), evaluates the
 * edges that touch them, exchanges halo entries of the PCG direction over NVLink (NCCL send/recv),
 * all-reduces the PCG dot products / chi2 / scale, and all-gathers the step before retracting, so
 * all ranks hold the same estimates after s3o_optimize.  Lock-step getters (s3o_get_hessian,
 * s3o_solve's x, ...) then refer to the local rows. */
int s3o_comm_unique_id(char *id128);
int s3o_set_comm(s3o_problem *p, int rank, int world, const char *id128);
/* host-only twin: the partition plan of one rank (counts only + the ghost list) for tests */
int s3o_host_partition(int n_vertices, const uint8_t *fixed, int n_edges, const int32_t *v0, const int32_t *v1,
                       int rank, int world, int32_t *n_own, int32_t *n_ghost, int32_t *n_local_edges,
                       int32_t *n_primary, int32_t *ghosts /* n_vertices */, int32_t *send_count /* world */,
                       int32_t *recv_count /* world */, int32_t *send_idx_global /* n_vertices*(world-1) upper bound */);

/* ---- graph (replaces addVertex / addEdge) --------------------------------------------- */
/* est: n x est_dim (SIM3 8, SCALE_TRANS 4, SCALE 1); fixed: n bytes or NULL;
 * aux: n x 4 rotation quaternions (SCALE_TRANS only, vST->Rw2i at kitti_surf.cpp:792-793) */
int s3o_set_vertices(s3o_problem *p, int n, const double *est, const uint8_t *fixed, const double *aux);
/* v0/v1: vertex indices (EdgeSim3 setVertex(0,.) / setVertex(1,.)); meas: n x est_dim;
 * info: n x d x d row-major symmetric, or NULL for identity (matLambdasim at kitti_surf.cpp:592) */
int s3o_set_edges(s3o_problem *p, int n, const int32_t *v0, const int32_t *v1, const double *meas,
                  const double *info);
/* overwrite the current estimates only (same n as s3o_set_vertices); structure is kept */
int s3o_set_estimates(s3o_problem *p, const double *est);
int s3o_set_robust(s3o_problem *p, int kind, double param);
int s3o_set_jacobian_mode(s3o_problem *p, int mode, double h /* numeric step, g2o: 1e-9 */);
int s3o_set_math_mode(s3o_problem *p, int mode);
int s3o_set_scale_model(s3o_problem *p, int model /* s3o_scale_model; S3O_KIND_SCALE / S3O_KIND_SCALE_TRANS */);
/* tau (g2o 1e-5), user lambda init (<=0: tau*max diag), maxTrialsAfterFailure (g2o 10) */
int s3o_set_lm(s3o_problem *p, double tau, double user_lambda_init, int max_trials);
/* block-Jacobi PCG: relative residual tolerance |r|/|b| and iteration cap */
int s3o_set_pcg(s3o_problem *p, double rel_tol, int max_iter);
int s3o_set_preconditioner(s3o_problem *p, int kind /* s3o_preconditioner */);
int s3o_set_linear_solver(s3o_problem *p, int kind /* s3o_linear_solver */);

/* ---- structure (replaces initializeOptimization + BlockSolver::buildStructure) -------- */
int s3o_build_structure(s3o_problem *p, int *n_free, int *n_blocks);
/* g2o-order upper block-CCS of Hpp: colptr[n_free+1], rowidx[n_blocks] (rows <= col, ascending) */
int s3o_get_structure(s3o_problem *p, int32_t *colptr, int32_t *rowidx);
/* Hessian index of every vertex (fixed -> -1) */
int s3o_get_hessian_index(s3o_problem *p, int32_t *hidx);

/* Host-only twin of the structure build (no device needed): fills the g2o-order upper block-CCS
 * for a graph given as plain arrays.  colptr must hold n_vertices+1 ints, rowidx n_vertices+n_edges
 * ints (upper bounds); hidx (may be NULL) n_vertices ints. */
int s3o_host_structure(int n_vertices, const uint8_t *fixed, int n_edges, const int32_t *v0, const int32_t *v1,
                       int *n_free, int *n_blocks, int32_t *colptr, int32_t *rowidx, int32_t *hidx);

/* Host-only view of the aggregation hierarchy the MULTILEVEL preconditioner builds for a graph:
 * n_levels coarse levels, their vertex and (full-pattern) block counts (first `cap` entries), and
 * the aggregate of every free vertex on the finest level (aggregate0: n_free ints, may be NULL).
 * With world > 1 no aggregate crosses the vertex ranges of s3o_host_partition. */
int s3o_host_multilevel(int n_vertices, const uint8_t *fixed, int n_edges, const int32_t *v0, const int32_t *v1,
                        int world /* ranks of the partitioned solve, 1 = one GPU */, int cap, int *n_levels,
                        int32_t *level_vertices, int32_t *level_blocks, int32_t *aggregate0);

/* Host-only view of the factorisation plan the DIRECT linear solver builds for a graph (no device needed; for
 * tests and tools).  Blocks of L are listed column by column in elimination order, pivot block first.  Call once
 * with every array NULL to get counts = [n_free, rounds, blocks of L, update-list entries, block products], then
 * with buffers: perm[n_free] elimination position -> Hessian index; lev_ptr[rounds+1] columns of each round;
 * cptr[n_free+1]; brow[nL] row position of each block; src[nL] (BSR-upper block << 1) | transposed or -1 for
 * fill-in (BSR order: s3o_host_structure's blocks sorted by (row, col), diagonal first in each row);
 * upd_ptr[nL+1], upd_a/upd_b: block t -= L[upd_a] L[upd_b]^T in list order.  max_pairs <= 0: no limit. */
int s3o_host_direct_plan(int n_vertices, const uint8_t *fixed, int n_edges, const int32_t *v0, const int32_t *v1,
                         int64_t max_pairs, int64_t *counts /* 5 */, int32_t *perm, int32_t *lev_ptr, int32_t *cptr,
                         int32_t *brow, int32_t *src, int32_t *upd_ptr, int32_t *upd_a, int32_t *upd_b);

/* ---- lock-step pieces (each mirrors one g2o step; used by the parity tests) ------------ */
int s3o_chi2(s3o_problem *p, double *chi2);                 /* computeActiveErrors + activeRobustChi2 */
int s3o_edge_errors(s3o_problem *p, double *err /* n_edges x d, caller's edge order */);
int s3o_linearize(s3o_problem *p);                          /* BlockSolver::buildSystem */
/* blocks in the g2o CCS order of s3o_get_structure, each d x d row-major; b: n_free*d */
int s3o_get_hessian(s3o_problem *p, double *blocks, double *b);
int s3o_max_diag(s3o_problem *p, double *max_diag);
/* solve (H + lambda I) x = b with the configured linear solver; x: n_free*d (may be NULL).  S3O_ERR_SOLVE on a
 * breakdown (matrix not positive definite). */
int s3o_solve(s3o_problem *p, double lambda, double *x, int *pcg_iters, double *rel_residual);
/* y = (H + lambda I) x on the device (x, y: n_free*d host arrays) -- for backward-error checks */
int s3o_hessian_multiply(s3o_problem *p, double lambda, const double *x, double *y);
/* oplus on every free vertex.  Partitioned solve: x holds the rows this rank owns (n_own * d); the step is
 * all-gathered inside, so the call is collective and leaves identical estimates on every rank. */
int s3o_update(s3o_problem *p, const double *x);

/* Eigenvector of the smallest eigenvalue of H = J^T Omega J at the current estimates, by inverse
 * iteration with the PCG solver (replaces the dense Eigen::JacobiSVD null-vector solve of the
 * stepwise scale initialisation, kitti_surf.cpp:887-934: H of the 1-DoF scale graph with no fixed
 * vertex is the Gram matrix of the reference's constraint matrix).  x: n_free*d, unit 2-norm, in
 * Hessian-index order; lambda_min / lambda_max: smallest / largest eigenvalue estimates (squared
 * singular values of J); stops when the eigenvalue estimate changes by less than tol relative. */
int s3o_smallest_eigenvector(s3o_problem *p, int max_iter, double tol, double *x, double *lambda_min,
                             double *lambda_max, int *iterations);

/* Marginal covariances: blocks of H^-1, where H = J^T Omega' J is the Gauss-Newton Hessian (robust weights
 * included, no LM damping) linearised at the CURRENT estimates, in the tangent of the left update S <- exp(d) S
 * (Sim3 [omega upsilon sigma], scale-trans [s t], scale [s]).  g2o SparseOptimizer::computeMarginals.
 * rows/cols: n_pairs Hessian indices (s3o_get_hessian_index; fixed vertices have none); out: n_pairs x d x d,
 * row-major, block (rows[k], cols[k]).  rows == cols == NULL: every diagonal block in Hessian order
 * (n_pairs must equal n_free).  S3O_ERR_SOLVE when H is singular (a connected component without a fixed
 * vertex); S3O_ERR_UNSUPPORTED for BA (s3o_ba_compute_marginals), the partitioned solve, and the NULL form on a
 * graph whose factor exceeds the forced cap.
 * Every call linearises again at the current estimates, so the result does not depend on what ran before it
 * (g2o uses the H of its last buildSystem, which is one step behind the estimates optimize() returns).  H is
 * factorised by the sparse block Cholesky (a plan under the forced cap of s3o_set_linear_solver(DIRECT) when the
 * linear solver in use has none; the linear solver the LM picks does not change), and the selected inverse gives
 * every block on the pattern of the factor -- all diagonal blocks and every pair joined by an edge -- for about
 * twice the block products of the factorisation.  A pair off that pattern costs d triangular solves for each
 * distinct column vertex among such pairs.
 * Beyond the forced cap (the 100k- and 1M-pose graphs) explicit pairs take an iterative route instead: the pairs
 * are grouped by column vertex c, and for each distinct c the d right-hand sides H x = e_(c,m), m = 0..d-1, are
 * solved by PCG without damping (the multilevel preconditioner for the Sim3, scale-trans and scale kinds under the
 * difference scale model, block-Jacobi otherwise), each refined until its true residual |e - H x|_2 is at most
 * S3O_MARGINALS_PCG_TOL (|e| = 1); where fp64 cannot resolve that (the residual's rounding floor eps |H| |x| lies
 * above it when kappa(H) ~ 1e12), refinement stops once a round no longer halves the residual, provided the
 * normwise backward error |e - H x| / (|H|_F |x|) is at most 1e-13.  Cost: d PCG solves per distinct column vertex, whatever the number of rows
 * requested with it.  Block (r, c) is always column c's solve; diagonal blocks come back exactly symmetric,
 * (X + X^T) / 2.  A solve that misses the tolerance within 20 000 PCG iterations, or breaks down, returns
 * S3O_ERR_SOLVE naming the column vertex, the component and the residual reached.  The NULL form would take
 * n_free * d solves there and returns S3O_ERR_UNSUPPORTED: request explicit pairs.  The environment variable
 * S3O_MARGINALS_ROUTE=pcg takes the iterative route on any graph (to compare both routes on one H).  The LM's
 * state (lambda, its scalars, the preconditioner choice) and the solver statistics are the same after the call.
 * Like s3o_smallest_eigenvector, the call leaves the problem unlinearised (s3o_solve needs s3o_linearize again). */
#define S3O_MARGINALS_PCG_TOL 1e-10
int s3o_compute_marginals(s3o_problem *p, int n_pairs, const int32_t *rows, const int32_t *cols, double *out);

/* ---- the hot call (replaces optimizer.optimize(n)) ------------------------------------- */
/* hist (may be NULL): per LM iteration [chi2, lambda, trials, rho, pcg_iters]; returns via
 * out-params the number of iterations run (g2o's return value), final chi2 and lambda.
 * stop_rel_gain > 0 adds g2o's optional gain rule 0 <= (chi2_prev-chi2)/chi2 < gain. */
int s3o_optimize(s3o_problem *p, int max_iter, double stop_rel_gain, int *iterations,
                 double *final_chi2, double *final_lambda, double *hist, int hist_cap);
int s3o_get_vertices(s3o_problem *p, double *est);
/* Partitioned solve (s3o_set_comm): the host round trip of the estimates, sharded over the ranks.  Every rank keeps all
 * estimates on its device, but its host only moves the slice [first, first + count) of the vertex ids that
 * s3o_estimate_slice reports (the even split; the whole range without a communicator).  s3o_set_estimates_slice is
 * COLLECTIVE: the slices are all-gathered over NVLink.  s3o_get_vertices_slice is local.  Same LM-state semantics as
 * s3o_set_estimates. */
int s3o_estimate_slice(s3o_problem *p, int *first, int *count);
int s3o_set_estimates_slice(s3o_problem *p, const double *est_slice);
int s3o_get_vertices_slice(s3o_problem *p, double *est_slice);
/* Optional stop rules of s3o_optimize (g2o's optimize() has none; 0 switches a rule off):
 *  max_abs_step (pose-graph kinds): stop once the estimated distance to the stationary point is below it in every
 *    tangent component (rad, m, log-scale).  The estimate comes from the accepted steps' max-norms s_k, which contract
 *    near the solution (the LM damps a weakly constrained mode by lambda / (mu + lambda) per iteration):
 *    s_k r / (1 - r) with r = s_k / s_(k-1) once r < 1/2, s_k itself before that.  Unlike a relative chi2 gain it does
 *    not depend on the size of the graph.  With inexact solves (PCG tolerance above 1e-4) the rule has to hold in two
 *    consecutive iterations.
 *  min_rel_predicted_decrease: stop when a step's predicted decrease sum x_j (lambda x_j + b_j) falls below this
 *    fraction of chi2 -- from there on the fp64 chi2 sums cannot resolve the step, g2o's acceptance test
 *    rho = (chi2 - chi2_new) / predicted is decided by round-off and the LM only burns trials (1e-12 is about the
 *    resolution of a sum over millions of edges).
 * s3o_stats reports s_k (last_step_inf), the estimate (est_distance) and which rule ended the last call
 * (stop_reason: 0 iteration count, 1 chi2 gain, 2 step, 3 resolution, 4 g2o Terminate). */
int s3o_set_stop_rules(s3o_problem *p, double max_abs_step, double min_rel_predicted_decrease);
/* resume = 1: the next s3o_optimize continues the LM sequence (keeps lambda, nu and the current
 * chi2) instead of re-initialising lambda at its first iteration -- lets a caller drive the LM one
 * iteration at a time.  The LM state is dropped by s3o_set_vertices / s3o_set_estimates /
 * s3o_restore_estimates.  resume = 2: as 1, but s3o_set_estimates keeps the LM state (the caller
 * re-uploads the estimates the previous s3o_optimize produced, e.g. after a host round trip). */
int s3o_set_lm_resume(s3o_problem *p, int resume);
/* device-side copy of the current estimates (g2o SparseOptimizer::push) and its restore (pop
 * without discarding): no host traffic */
int s3o_snapshot_estimates(s3o_problem *p);
int s3o_restore_estimates(s3o_problem *p);

/* ---- bundle adjustment, kind S3O_KIND_BA (replaces the g2o calls of ba_demo, bal_example.cpp:44-243)
 *   new VertexSE3Expmap; setId(0..C-1); setEstimate(SE3Quat(q_w2c, t))     :110-117,:168-185  s3o_ba_set_cameras
 *   new VertexSBAPointXYZ; setMarginalized(true); setEstimate(p)           :119-129,:187-194  s3o_ba_set_points
 *   new EdgeProjectXYZ2UV; setVertex(0, point); setVertex(1, cam);
 *     setInformation(I/sigma^2); setMeasurement(uv); setParameterId(0,0)   :131-166           s3o_ba_set_observations
 *   RobustKernelHuber, setDelta(2.5)                                       :149-153           s3o_set_robust
 *   CameraParameters(f, pp, 0)                                             :87-96             s3o_ba_set_intrinsics
 *   initializeOptimization / optimize(n)                                   :198,:213          s3o_build_structure / s3o_optimize
 * Camera state: 7 doubles [qx qy qz qw tx ty tz] (g2o SE3Quat, world -> camera), tangent [omega, upsilon];
 * point: xyz.  Hessian order: free cameras (6 each, id order) then free points (3 each).  The points
 * are always marginalised (Schur complement, as BlockSolver_6_3 does): s3o_build_structure returns the
 * number of free cameras and of upper blocks of H_schur, s3o_get_structure its g2o-order block-CCS;
 * s3o_solve / s3o_update take x = [6 n_free_cameras | 3 n_free_points].  Call order: cameras and
 * points first, then observations. */
int s3o_ba_set_cameras(s3o_problem *p, int n, const double *est /* n x 7 */, const uint8_t *fixed /* or NULL */);
int s3o_ba_set_points(s3o_problem *p, int n, const double *xyz /* n x 3 */, const uint8_t *fixed /* or NULL */);
/* info: n x 3 packed symmetric [xx xy yy], or NULL for identity */
int s3o_ba_set_observations(s3o_problem *p, int n, const int32_t *cam_idx, const int32_t *point_idx,
                            const double *uv /* n x 2 */, const double *info);
int s3o_ba_set_intrinsics(s3o_problem *p, double focal, double cx, double cy);
int s3o_ba_set_estimates(s3o_problem *p, const double *cams /* or NULL */, const double *points /* or NULL */);
int s3o_ba_get_cameras(s3o_problem *p, double *est);
int s3o_ba_get_points(s3o_problem *p, double *xyz);
int s3o_ba_get_sizes(s3o_problem *p, int *n_free_cameras, int *n_free_points, int *n_schur_blocks,
                     int64_t *n_contributions);
/* lock-step read-outs: errors n_obs x 2 and Hpl n_obs x 6 x 3 (= Jc^T O' Jp) in the caller's
 * observation order; Hpp n_free_cameras x 6 x 6; Hll n_free_points x 3 x 3; b = [b_cameras | b_points] */
int s3o_ba_edge_errors(s3o_problem *p, double *err);
int s3o_ba_get_system(s3o_problem *p, double *Hpp, double *Hll, double *Hpl, double *b);
/* damped Schur complement S = (Hpp + lambda I) - sum Hpl (Hll + lambda I)^-1 Hpl^T (blocks in the CCS
 * order of s3o_get_structure) and bs = bp - sum Hpl (Hll + lambda I)^-1 bl */
int s3o_ba_get_schur(s3o_problem *p, double lambda, double *blocks, double *bs);
/* Marginal covariances of bundle adjustment (g2o SparseOptimizer::computeMarginals on the BA graph): blocks of
 * Sigma = H^-1, H = [[Hpp, Hpl], [Hpl^T, Hll]] the full Gauss-Newton Hessian (robust weights and information included,
 * no LM damping) linearised at the CURRENT estimates, with the same semantics as s3o_compute_marginals.  Tangents:
 * camera [omega, upsilon] of T <- exp(d) T, point xyz.  Hessian indices: free cameras 0 .. ncf-1 in camera-id order,
 * then free points ncf .. ncf+npf-1 in point-id order (ncf, npf: s3o_ba_get_sizes); fixed vertices have none.
 * out: the blocks back to back, block k dim(rows[k]) x dim(cols[k]) row-major (dim 6 for a camera, 3 for a point)
 * at the sum of the sizes of the blocks before it.  rows == cols == NULL: every diagonal block, cameras then points
 * (n_pairs must equal ncf + npf; out holds 36 ncf + 9 npf doubles).  Pairs served: any two cameras; the diagonal
 * block of a point; (camera, point) and (point, camera) when that camera observes that point.  Camera blocks come
 * from the selected inverse of the Schur complement S = Hpp - Hpl Hll^-1 Hpl^T (s3o_compute_marginals' machinery on
 * the 6x6 system), points from Sigma(c_a, l) = -Z_a and Sigma(l, l) = Hll^-1 + sum_a Y_a^T Z_a with
 * Y_a = Hpl_a Hll^-1, Z_a = sum_b S^-1(c_a, c_b) Y_b over the point's observations by free cameras.
 * Returns S3O_ERR_UNSUPPORTED for two distinct points, a camera-point pair whose camera does not observe the point,
 * or a Schur factor beyond the forced cap; S3O_ERR_INVALID for bad arguments, an index out of range, or a problem that
 * is not BA; S3O_ERR_SOLVE, naming a vertex, when H is singular: a connected component of the observation graph fixes
 * neither a camera and one more vertex nor three points (the 7-DoF gauge of monocular BA is free), or a free point is
 * seen by fewer than two distinct cameras; S3O_ERR_SOLVE also when a pivot of the factorisation of S fails or a free
 * point's det(Hll) is not positive.  The LM state (step, lambda, snapshots, direct_solves) is untouched, and the
 * problem is left unlinearised. */
int s3o_ba_compute_marginals(s3o_problem *p, int n_pairs, const int32_t *rows, const int32_t *cols, double *out);

/* ---- LinearSolver-level plug-in: g2o::LinearSolver<M>::{init(), solve(A, x, b)} (the innermost slot of
 * OptimizationAlgorithmLevenberg(BlockSolverX(LinearSolverEigen)), kitti_surf.cpp:553-557, bal_example.cpp:73-83) ----
 * For callers that keep g2o's own LM loop and block solver and only swap the linear solver: A is g2o's
 * SparseBlockMatrix, i.e. an upper block-CCS (colptr[n+1], rowidx[nb], rows ascending, row <= column, every column
 * with its diagonal block) of d x d blocks, each row-major or (Eigen's default) column-major; b and x are n*d.
 * Solves (A + lambda I) x = b on the device: sparse block Cholesky when the factor is small (see
 * s3o_linear_solver), block-Jacobi PCG (s3o_set_pcg on the handle) otherwise.  The handle caches the pattern, the
 * factorisation plan and all device buffers between calls (LinearSolver::init() once, solve() per LM trial).  The
 * whole-LM entry s3o_optimize avoids the per-trial PCIe round trip of A, x, b that this cut implies.
 * Returns S3O_OK, or S3O_ERR_SOLVE when the matrix is not positive definite / the PCG did not converge (g2o:
 * solve() == false -> the LM raises lambda). */
typedef struct s3o_problem s3o_linsolver;
int s3o_linsolver_create(int device, int block_dim /* 1, 4, 6 or 7 */, s3o_linsolver **out);
int s3o_linsolver_destroy(s3o_linsolver *s);
int s3o_linsolver_solve(s3o_linsolver *s, int n_block_cols, const int32_t *colptr, const int32_t *rowidx,
                        const double *blocks, int column_major, double lambda, const double *b, double *x,
                        int *method /* out, may be NULL: s3o_linear_solver used */, int *pcg_iterations /* may be NULL */);

/* ---- statistics ------------------------------------------------------------------------ */
typedef struct s3o_stats {
    double ms_linearize, ms_solve, ms_chi2, ms_update, ms_total; /* CUDA-event time, last optimize */
    int64_t kernel_launches;   /* kernels launched by this problem since create / reset */
    int64_t pcg_iterations;    /* PCG iterations since create / reset */
    int64_t lm_iterations, lm_trials;
    int64_t h2d_bytes, d2h_bytes;
    int32_t n_vertices, n_free, n_edges, n_blocks, dim;
    /* CUDA-event time of the SpMV kernel alone, sampled on 1 of every 16 PCG iterations */
    double ms_spmv_sampled;
    int64_t n_spmv_sampled;
    int32_t multilevel_levels; /* coarse levels of the multilevel preconditioner in use (0: block-Jacobi) */
    int32_t p2p_halo;          /* partitioned solve: 1 if the SpMV reads ghost columns from the peers' memory (CUDA IPC
                                  over NVLink), 0 if they are exchanged by NCCL send/recv */
    int64_t direct_solves;     /* exact solves (sparse block Cholesky) since create / reset */
    int32_t direct_levels;     /* elimination rounds of the factorisation plan (0: PCG in use) */
    int32_t direct_blocks;     /* blocks of the factor L */
    int64_t pcg_unconverged;   /* PCG solves that ended on the iteration cap or a breakdown (inexact LM steps) */
    double sum_ms_linearize, sum_ms_solve, sum_ms_update; /* the per-call phase times above, summed since create / reset */
    double last_step_inf;      /* max |x_j| of the last accepted LM step (pose-graph kinds) */
    double est_distance;       /* estimated max-norm distance to the stationary point after it (s3o_set_stop_rules) */
    int32_t stop_reason;       /* why the last s3o_optimize returned (s3o_set_stop_rules) */
    int32_t reserved0;
    int64_t multilevel_rebuilds; /* solves that rebuilt the coarse operators P^T H P of the multilevel preconditioner ... */
    int64_t multilevel_reuses;   /* ... and solves that kept them (LM retry: same linearisation point, new lambda) */
} s3o_stats;
int s3o_get_stats(s3o_problem *p, s3o_stats *out);
int s3o_reset_stats(s3o_problem *p);

/* ---- trajectory alignment and its RMSE (evaluation modes of the reference, kitti_surf.cpp:1091-1161,
 * :1432-1452) ---------------------------------------------------------------------------------
 * Similarity S221 (4x4 row-major, [cR t; 0 1]) that maps the query positions onto the train positions:
 * Eigen::umeyama(query, train, true), or with only_scale != 0 the reference's extent-ratio scale
 * (mean over the x and z axes, no rotation / translation).  rmse and max_dev are those of
 * train_i - S221 query_i.  n x 3 arrays, row-major.  Moments are reduced on `device`. */
int s3o_align_similarity(int device, int n, const double *query_xyz, const double *train_xyz, int only_scale,
                         double *S221 /* 16 */, double *rmse, double *max_dev);

/* ---- PTAM sigma estimate (MEstimator.h FindSigmaSquared) on the current edge chi2 values - */
int s3o_estimate_sigma_squared(s3o_problem *p, int robust_kind, double *sigma_squared);

#ifdef __cplusplus
}
#endif
#endif /* SIM3OPT_B200_H */
