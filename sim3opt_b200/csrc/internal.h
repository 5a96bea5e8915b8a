// internal.h -- shared declarations of the sim3opt_b200 library (host side).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#include "../../include/sim3opt_b200.h"

namespace s3o {

void set_error(const char *fmt, ...);

#define S3O_CUDA(call)                                                                      \
    do {                                                                                    \
        cudaError_t _e = (call);                                                            \
        if (_e != cudaSuccess) {                                                            \
            s3o::set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #call,               \
                           cudaGetErrorString(_e));                                         \
            return S3O_ERR_CUDA;                                                            \
        }                                                                                   \
    } while (0)

inline int pad32(int n) { return (n + 31) & ~31; }

// S3O_SETUP_TRACE=1: wall-clock of the set-up stages on stderr (diagnostic)
inline void setup_mark(const char *what) {
    static const bool on = getenv("S3O_SETUP_TRACE") != nullptr;
    static std::chrono::steady_clock::time_point last = std::chrono::steady_clock::now();
    if (!on) return;
    const auto now = std::chrono::steady_clock::now();
    if (what) fprintf(stderr, "[s3o setup] %-28s %8.1f ms\n", what, std::chrono::duration<double, std::milli>(now - last).count());
    last = now;
}


// Host-side result of the structure build (SURVEY.md row a14).
struct HostStructure {
    int nv = 0, ne = 0;          // vertices, user edges
    int nf = 0, nb = 0;          // free vertices, upper blocks
    int ne_act = 0;              // active edges (at least one free end), in sorted order
    std::vector<int32_t> hidx;   // [nv] Hessian index or -1
    std::vector<int32_t> free2v; // [nf]
    std::vector<int32_t> perm;   // [ne_act] sorted position -> user edge index
    std::vector<int32_t> sv0, sv1;      // [ne_act] vertex ids in sorted order
    std::vector<int32_t> e_blk;         // [ne_act] off-diagonal block (BSR index) or -1
    std::vector<int32_t> rowptr, colidx;        // BSR upper, diagonal first in each row
    std::vector<int32_t> blk_ebeg, blk_eend;    // [nb] sorted-edge range feeding each off-diag block
                                                //      (diag blocks: empty range)
    std::vector<int32_t> blk_src;               // [nb] off-diag block fed by exactly one edge: (sorted edge << 1) | transposed; else -1
    std::vector<int32_t> multi_blk;             // off-diagonal blocks fed by more than one edge (duplicate edges)
    std::vector<int32_t> colT_ptr, colT_blk;    // [nf+1], [nb-nf]: off-diag blocks by column (rows ascending)
    std::vector<int32_t> inc_ptr, inc_ent;      // [nf+1], incidences: (sorted edge << 1) | side
    std::vector<int32_t> ccs_colptr, ccs_rowidx; // g2o-order upper block-CCS
    std::vector<int32_t> ccs2bsr;               // [nb] CCS position -> BSR block index
    std::vector<int32_t> tile_row;              // [ntiles+1] first block row of each SpMV tile
    int tile_blocks = 0;                        // tile capacity (blocks) the tiles were packed for
    int max_row_blocks = 0;
};

// Packs whole block rows into tiles of at most `cap` blocks; a row with more than `cap` blocks
// gets a tile of its own (processed in chunks by one CTA).
void build_tiles(const std::vector<int32_t> &rowptr, int nf, int cap, std::vector<int32_t> &tile_row);
int spmv_tile_blocks(int d);

void build_structure_host(int nv, const uint8_t *fixed, int ne, const int32_t *v0, const int32_t *v1,
                          HostStructure &S);
// same with an explicit Hessian-index map (hidx[v] in [0,nfree) or -1): used by the partitioned path,
// where "free" means owned or ghost on this rank
void build_structure_from_hidx(int nv, const int32_t *hidx, int nfree, int ne, const int32_t *v0, const int32_t *v1,
                               HostStructure &S);

// Device twin (structure_dev.cu): the same arrays from integer kernels (stable radix sort + scans); bit-identical.
// Device copies of the index arrays that build_structure_device leaves alive for the caller (ownership passes:
// cudaFree them).  The arrays no host code reads are not copied back at all.
struct DeviceStructure {
    int32_t *hidx = nullptr, *sv0 = nullptr, *sv1 = nullptr, *blk_ebeg = nullptr, *blk_eend = nullptr, *blk_src = nullptr,
            *multi_blk = nullptr, *inc_ptr = nullptr, *inc_ent = nullptr, *e_blk = nullptr, *rowptr = nullptr, *colidx = nullptr,
            *blk_row = nullptr, *colT_ptr = nullptr, *colT_blk = nullptr, *perm = nullptr;
    bool valid = false;
};
int build_structure_device(cudaStream_t st, int nv, const uint8_t *fixed, const int32_t *hidx_in, int nfree_in, int ne,
                           const int32_t *v0, const int32_t *v1, HostStructure &S, DeviceStructure *keep = nullptr);
// Device merge of appended vertices and edges into a built structure (s3o_add_vertices / s3o_add_edges, merged by
// s3o_build_structure).  S, keep and the edge records out equal what build_structure_device and the edge packing give
// for the concatenated arrays, bit for bit: appended free vertices are numbered n_free_old, n_free_old + 1, ..., and
// an appended edge sorts after the built edges with the same key.  The built arrays are read, not freed.
struct StructureMerge {
    // the built structure: vertices, free vertices, active edges, caller edges; device arrays in sorted order
    int nv_old = 0, nf_old = 0, na_old = 0, ne_old = 0;
    const int32_t *hidx = nullptr, *sv0 = nullptr, *sv1 = nullptr, *perm = nullptr;
    // appended: vertices nv_old..nv-1 (fixed flags, host) and caller edges ne_old..ne-1 (endpoints, host)
    int nv = 0, ne = 0;
    const uint8_t *fixed_new = nullptr;
    const int32_t *v0_new = nullptr, *v1_new = nullptr;
    // edge records.  Information representations: 0 none (identity), 1 diagonal, 2 full.  Built: SoA planes at pitch
    // ne_pad_old (d planes when diagonal, d(d+1)/2 packed upper triangles when full).  Appended: caller order, AoS
    // (est_dim measurement entries; d or d*d information entries), already in the merged representation info_rep.
    int est_dim = 0, d = 0, ne_pad_old = 0, info_rep_old = 0, info_rep = 0;
    const double *meas = nullptr, *info = nullptr, *meas_new = nullptr, *info_new = nullptr;
    // out: the merged records at pitch pad32(active edges) in info_rep (the caller frees them), and the bytes copied
    // from the host (fixed flags and endpoints of the appended elements)
    double *meas_out = nullptr, *info_out = nullptr;
    int64_t h2d_bytes = 0;
};
int merge_structure_device(cudaStream_t st, StructureMerge &M, HostStructure &S, DeviceStructure &keep);

// Vertex-range partition of the free vertices across `world` ranks (SURVEY.md section 8e).
// Rank r owns global Hessian indices [r*seg, min((r+1)*seg, nf)), seg = ceil(nf/world).
struct PartitionPlan {
    int rank = 0, world = 1;
    int nf_global = 0, seg = 0;
    int own_lo = 0, n_own = 0, n_ghost = 0;
    std::vector<int32_t> ghidx;        // [nv] global Hessian index, -1 fixed
    std::vector<int32_t> lhidx;        // [nv] local Hessian index: owned [0,n_own), ghosts after, else -1
    std::vector<int32_t> ghosts;       // global Hessian indices of the ghosts, ascending
    std::vector<int32_t> local_edges;  // user edge indices with at least one owned endpoint (user order)
    std::vector<uint8_t> primary;      // per local edge: 1 if this rank counts its chi2
    std::vector<int32_t> recv_count, recv_off;   // [world] ghost runs per owner (in ghost order)
    std::vector<int32_t> send_count, send_off;   // [world]
    std::vector<int32_t> send_idx;               // local owned indices to pack, grouped by peer
};
void build_partition_plan(int nv, const uint8_t *fixed, int ne, const int32_t *v0, const int32_t *v1, int rank,
                          int world, PartitionPlan &P);

}  // namespace s3o
