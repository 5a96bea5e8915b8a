// kernels.cuh -- device data layout and launcher declarations.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace s3o {

// Device scalars of the PCG / LM bookkeeping.  Everything the inner loop needs stays on the
// device; the host reads this struct back once per LM trial (and per PCG batch).
struct DevScalars {
    double rz;        // r.z of the current iterate
    double rz_new;    // r.z after the update   } adjacent: all-reduced together
    double rr;        // |r|^2                  } in the partitioned solve
    double pq;        // p.(H+lambda I)p
    double alpha, beta;
    double rr0;       // |b|^2
    double tol2;      // (rel_tol)^2
    double chi2;      // last chi2 reduction
    double scale;     // sum x_j (lambda x_j + b_j)   (computeScale)
    double maxdiag;   // max |H_jj|                  (computeLambdaInit)
    double xmax;      // max |x_j| of the last step  (step-size stop rule)
    int done;         // 0 running, 1 converged, 2 iteration cap, 3 breakdown
    int iters, max_iter;
    int precond_fail;
    int halo_fail;    // partitioned solve: a neighbour's epoch flag did not arrive (peer died); see halo_wait_kernel
    unsigned counters[8];
};

struct GraphDev {
    int kind, d, est_dim, ninfo;
    int nv, nv_pad, ne, ne_pad, nf, nb;
    const double *est;       // [est_dim][nv_pad]
    const double *aux;       // [4][nv_pad] or null
    const int32_t *hidx;     // [nv]
    const int32_t *sv0, *sv1; // [ne]
    const double *meas;      // [est_dim][ne_pad]
    const double *info;      // [ninfo][ne_pad] packed upper triangles, [d][ne_pad] diagonals when info_diag, or null (identity)
    bool info_diag;          // every information matrix is diagonal (checked on the host in s3o_set_edges)
    int robust_kind;
    double robust_param;
    bool math_corrected;     // s3o_set_math_mode
    int model_flags;         // bit 0: math_corrected, bit 1: log-ratio scale model (s3o_set_scale_model)
    const uint8_t *primary;  // [ne] partitioned solve: 1 if this rank counts the edge's chi2 (null: all)
    const int32_t *ghidx;    // [nv] partitioned solve: global Hessian index addressing the gathered step
};

struct StructDev {
    const int32_t *rowptr, *colidx, *blk_row;
    const int32_t *blk_ebeg, *blk_eend;
    const int32_t *blk_src;   // [nb] single-edge off-diagonal blocks: (sorted edge << 1) | transposed, else -1
    const int32_t *multi_blk; // [n_multi] off-diagonal blocks fed by more than one edge
    int n_multi;
    const int32_t *colT_ptr, *colT_blk;
    const int32_t *inc_ptr, *inc_ent;
    const int32_t *e_blk;
    const int32_t *tile_row;  // [ntiles+1]
    int ntiles;
    int n_own;                // rows owned by this rank (= nf on one GPU); columns >= n_own are ghosts
    double *const *ghost_src; // partitioned solve with peer-to-peer halos: where ghost column g lives in its owner's p
                              // (CUDA IPC mapping of the peer's vector); null: ghosts are local copies filled by NCCL
};

constexpr int kMaxPartials = 4096;

// ---- packing ---------------------------------------------------------------------------
void launch_pack_vertices(const double *aos, int n, int n_pad, int dim, double *soa, cudaStream_t st);
void launch_unpack_vertices(const double *soa, int n, int n_pad, int dim, double *aos, cudaStream_t st);
void launch_pack_edges(const double *meas_aos, const double *info_aos, const int32_t *perm, int ne, int ne_pad,
                       int est_dim, int d, int info_diag, double *meas, double *info, cudaStream_t st);

// ---- per-edge --------------------------------------------------------------------------
void launch_chi2(const GraphDev &g, double *partials, DevScalars *sc, cudaStream_t st);
void launch_edge_errors(const GraphDev &g, double *err_sorted /* [ne][d] */, double *chi2_sorted /* [ne] or null */,
                        cudaStream_t st);
// e_blk / blk_src / Hdirect: single-edge off-diagonal blocks are written straight into the Hessian
void launch_linearize(const GraphDev &g, int jac_mode, double h, double *scratch /* [ne][scr] */, const int32_t *e_blk,
                      const int32_t *blk_src, double *Hdirect, cudaStream_t st);
int scratch_stride(int d);
void launch_assemble(const GraphDev &g, const StructDev &s, const double *scratch, double *H, double *b,
                     cudaStream_t st);
void launch_retract(const GraphDev &g, const double *x, double *est_out, cudaStream_t st);

// ---- linear algebra on the BSR-upper Hessian --------------------------------------------
// `dist` != 0: the kernel only leaves its local sums in DevScalars; the caller all-reduces them and
// launches the matching launch_pcg_fin_* kernel.
void launch_maxdiag(int d, const double *H, const int32_t *rowptr, int nf, double *partials, DevScalars *sc,
                    cudaStream_t st);
void launch_pcg_fin_init(DevScalars *sc, double tol, int max_iter, cudaStream_t st);
void launch_pcg_fin_spmv(DevScalars *sc, cudaStream_t st);
void launch_pcg_fin_update(DevScalars *sc, cudaStream_t st);
void launch_pack_rows(int d, const double *vec, const int32_t *idx, int n, double *out, const DevScalars *sc,
                      cudaStream_t st);
void launch_precond(int d, const double *H, const int32_t *rowptr, int nf, double lambda, double *Minv,
                    DevScalars *sc, cudaStream_t st);
void launch_spmv(int d, const double *H, const StructDev &s, int nf, double lambda, const double *p, double *q1,
                 double *T, double *partials, DevScalars *sc, int pcg_mode, cudaStream_t st);
void launch_finish_q(int d, const StructDev &s, int nf, const double *q1, const double *T, double *q, cudaStream_t st);
void launch_pcg_init(int d, int nf, const double *b, const double *Minv, double *x, double *r, double *z, double *p,
                     double *partials, DevScalars *sc, double tol, int max_iter, int dist, cudaStream_t st);
void launch_pcg_update(int d, const StructDev &s, int nf, const double *q1, const double *T, const double *Minv,
                       const double *p, double *x, double *r, double *z, double *partials, DevScalars *sc,
                       int dist, cudaStream_t st);
void launch_pcg_pupdate(int d, int nf, const double *z, double *p, const DevScalars *sc, cudaStream_t st);
void launch_scale(int n, const double *x, const double *b, double lambda, double *partials, DevScalars *sc,
                  cudaStream_t st);
int launches_per_pcg_iter();
// peer-to-peer halo: publish "my p is complete for this product" / wait until every neighbour has
void launch_halo_signal(long long *own_flag, long long epoch, cudaStream_t st);
void launch_halo_wait(long long *const *peer_flags, int n_peers, long long epoch, DevScalars *sc, cudaStream_t st);
void launch_scale_vec(int n, const double *in, double s, double *out, cudaStream_t st);
void launch_fill_const(int n, double v, double *out, cudaStream_t st);
void launch_fill_alternating(int n, double *out, cudaStream_t st);
// tiled thread-per-block SpMV (spmv.cu)
int spmv_tile_blocks(int d);
int spmv2_configure();
int spmv3_tile_blocks(int d);
void launch_spmv3(int d, const double *H, const StructDev &s, int nf, double lambda, const double *p, double *q1,
                  double *T, double *partials, DevScalars *sc, int pcg_mode, int grid_cap, int dist, cudaStream_t st);
// v4 (d = 7 only): v3 + descriptor staging, register-pipelined index / vector prefetch, NS-deep ring
int spmv4_tile_blocks(int cfg);
bool spmv4_fits(int ntiles, int grid_cap);
void launch_spmv4(const double *H, const StructDev &s, int nf, double lambda, const double *p, double *q1, double *T,
                  double *partials, DevScalars *sc, int pcg_mode, int cfg, int grid_cap, int dist, cudaStream_t st);
void launch_spmv2(int d, const double *H, const StructDev &s, int nf, double lambda, const double *p, double *q1,
                  double *T, double *partials, DevScalars *sc, int pcg_mode, int dist, cudaStream_t st);

}  // namespace s3o
