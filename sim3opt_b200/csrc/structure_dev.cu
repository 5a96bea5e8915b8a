// structure_dev.cu -- sparsity pattern and BSR index build on the device.
//
// Same outputs as build_structure_from_hidx (structure.cpp), which replaces SparseOptimizer::initializeOptimization +
// BlockSolver::buildStructure [EXT g2o] (SURVEY.md row a14; reference call site kitti_surf.cpp:674), computed by
// integer kernels: a stable LSD radix sort of the active edges by their (min,max) Hessian-index pair (ties keep the
// caller's edge order, which fixes every summation order downstream), run-boundary flags + exclusive scans for the
// BSR-upper rows / columns / per-block edge ranges, and two more stable sorts for the per-vertex incidence lists and
// the column view; the g2o-order block-CCS falls out of the column view.  Everything is integer work with one
// writer per output, so the result is bit-identical to the host build (tests/test_gpu_structure.py).
#include <algorithm>
#include <vector>

#include "internal.h"
#include "problem.h"

namespace s3o {

namespace {

constexpr int kScanThreads = 256, kScanItems = 8, kScanTile = kScanThreads * kScanItems;

// ---- exclusive scan (int32), two levels: tile sums -> scan of the sums -> tile-local scan + offset -----------
__global__ void scan_tile_sums_kernel(const int32_t *__restrict__ in, int n, int32_t *__restrict__ sums) {
    __shared__ int32_t sh[kScanThreads / 32];
    const int base = blockIdx.x * kScanTile;
    int32_t v = 0;
    for (int k = 0; k < kScanItems; ++k) {
        const int t = base + threadIdx.x * kScanItems + k;
        if (t < n) v += in[t];
    }
    for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        int32_t s = 0;
        for (int w = 0; w < kScanThreads / 32; ++w) s += sh[w];
        sums[blockIdx.x] = s;
    }
}
// exclusive scan of up to kScanThreads * cap entries by ONE block (the second level)
__global__ void scan_small_kernel(int32_t *data, int n, int32_t *total) {
    __shared__ int32_t sh[kScanThreads];
    const int per = (n + kScanThreads - 1) / kScanThreads;
    const int lo = threadIdx.x * per, hi = min(n, lo + per);
    int32_t s = 0;
    for (int t = lo; t < hi; ++t) s += data[t];
    sh[threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        int32_t run = 0;
        for (int w = 0; w < kScanThreads; ++w) { const int32_t c = sh[w]; sh[w] = run; run += c; }
        if (total) *total = run;
    }
    __syncthreads();
    int32_t run = sh[threadIdx.x];
    for (int t = lo; t < hi; ++t) { const int32_t c = data[t]; data[t] = run; run += c; }
}
__global__ void scan_apply_kernel(const int32_t *__restrict__ in, int n, const int32_t *__restrict__ offs,
                                  int32_t *__restrict__ out) {
    __shared__ int32_t sh[kScanThreads];
    const int base = blockIdx.x * kScanTile;
    int32_t loc[kScanItems];
    int32_t s = 0;
    for (int k = 0; k < kScanItems; ++k) {
        const int t = base + threadIdx.x * kScanItems + k;
        loc[k] = t < n ? in[t] : 0;
        s += loc[k];
    }
    sh[threadIdx.x] = s;
    __syncthreads();
    // exclusive prefix over the block's threads (Hillis-Steele on 256 entries)
    for (int off = 1; off < kScanThreads; off <<= 1) {
        const int32_t add = threadIdx.x >= off ? sh[threadIdx.x - off] : 0;
        __syncthreads();
        sh[threadIdx.x] += add;
        __syncthreads();
    }
    int32_t run = offs[blockIdx.x] + sh[threadIdx.x] - s;
    for (int k = 0; k < kScanItems; ++k) {
        const int t = base + threadIdx.x * kScanItems + k;
        if (t < n) out[t] = run;
        run += loc[k];
    }
}

struct Scratch {
    cudaStream_t st;
    int32_t *tile_sums = nullptr, *d_total = nullptr;
    size_t tile_cap = 0;
};

// out[t] = sum of in[0..t), out may alias in; returns the total through *total_host (synchronises)
int exclusive_scan(Scratch &S, const int32_t *in, int32_t *out, int n, int32_t *total_host) {
    if (n <= 0) { if (total_host) *total_host = 0; return S3O_OK; }
    const int tiles = (n + kScanTile - 1) / kScanTile;
    if ((size_t)tiles > S.tile_cap) {
        if (S.tile_sums) cudaFree(S.tile_sums);
        S.tile_cap = (size_t)tiles * 2;
        S3O_CUDA(cudaMalloc((void **)&S.tile_sums, S.tile_cap * sizeof(int32_t)));
    }
    if (!S.d_total) S3O_CUDA(cudaMalloc((void **)&S.d_total, sizeof(int32_t)));
    scan_tile_sums_kernel<<<tiles, kScanThreads, 0, S.st>>>(in, n, S.tile_sums);
    scan_small_kernel<<<1, kScanThreads, 0, S.st>>>(S.tile_sums, tiles, S.d_total);
    scan_apply_kernel<<<tiles, kScanThreads, 0, S.st>>>(in, n, S.tile_sums, out);
    if (total_host) {
        S3O_CUDA(cudaMemcpyAsync(total_host, S.d_total, sizeof(int32_t), cudaMemcpyDeviceToHost, S.st));
        S3O_CUDA(cudaStreamSynchronize(S.st));
    }
    return S3O_OK;
}

// ---- stable LSD radix sort, 8 bits per pass, 64-bit keys with a 32-bit payload --------------------------------
// One warp owns a contiguous chunk; inside a chunk the keys are ranked 32 at a time with match_any (order inside
// a tile = lane order = input order), so equal digits keep their input order: the sort is stable and, with integer
// counts only, reproducible.
constexpr int kSortChunk = 2048;

__global__ void radix_hist_kernel(const uint64_t *__restrict__ keys, int n, int shift, int nchunks, int32_t *__restrict__ hist) {
    __shared__ int32_t bins[256];
    const int chunk = blockIdx.x;
    for (int b = threadIdx.x; b < 256; b += blockDim.x) bins[b] = 0;
    __syncthreads();
    const int lo = chunk * kSortChunk, hi = min(n, lo + kSortChunk);
    for (int t = lo + threadIdx.x; t < hi; t += blockDim.x) atomicAdd(&bins[(int)((keys[t] >> shift) & 255u)], 1);
    __syncthreads();
    for (int b = threadIdx.x; b < 256; b += blockDim.x) hist[(size_t)b * nchunks + chunk] = bins[b];
}

__global__ void radix_scatter_kernel(const uint64_t *__restrict__ keys, const int32_t *__restrict__ vals, int n, int shift,
                                     int nchunks, const int32_t *__restrict__ base, uint64_t *__restrict__ keys_out,
                                     int32_t *__restrict__ vals_out) {
    __shared__ int32_t pos[256];
    const int chunk = blockIdx.x, lane = threadIdx.x;      // one warp per block
    for (int b = lane; b < 256; b += 32) pos[b] = base[(size_t)b * nchunks + chunk];
    __syncwarp();
    const int lo = chunk * kSortChunk, hi = min(n, lo + kSortChunk);
    for (int t0 = lo; t0 < hi; t0 += 32) {
        const int t = t0 + lane;
        const bool act = t < hi;
        const uint64_t k = act ? keys[t] : 0;
        const int d = act ? (int)((k >> shift) & 255u) : 256 + lane;       // inactive lanes match nobody
        const unsigned peers = __match_any_sync(0xffffffffu, d);
        const int rank = __popc(peers & ((1u << lane) - 1u));
        int dst = 0;
        if (act) dst = pos[d] + rank;
        __syncwarp();
        if (act && rank == 0) pos[d] += __popc(peers);
        __syncwarp();
        if (act) { keys_out[dst] = k; vals_out[dst] = vals[t]; }
    }
}

struct SortBuf {
    uint64_t *k0 = nullptr, *k1 = nullptr;
    int32_t *v0 = nullptr, *v1 = nullptr, *hist = nullptr;
    size_t cap = 0, hist_cap = 0;
};

// sorts (keys, vals) of length n on the low `bits` bits; result pointers through *keys_sorted / *vals_sorted
int radix_sort(Scratch &S, SortBuf &B, int n, int bits, uint64_t **keys_sorted, int32_t **vals_sorted) {
    *keys_sorted = B.k0;
    *vals_sorted = B.v0;
    if (n <= 0) return S3O_OK;
    const int nchunks = (n + kSortChunk - 1) / kSortChunk;
    if ((size_t)256 * nchunks > B.hist_cap) {
        if (B.hist) cudaFree(B.hist);
        B.hist_cap = (size_t)256 * nchunks;
        S3O_CUDA(cudaMalloc((void **)&B.hist, B.hist_cap * sizeof(int32_t)));
    }
    uint64_t *ki = B.k0, *ko = B.k1;
    int32_t *vi = B.v0, *vo = B.v1;
    for (int shift = 0; shift < bits; shift += 8) {
        radix_hist_kernel<<<nchunks, 128, 0, S.st>>>(ki, n, shift, nchunks, B.hist);
        int rc = exclusive_scan(S, B.hist, B.hist, 256 * nchunks, nullptr);
        if (rc) return rc;
        radix_scatter_kernel<<<nchunks, 32, 0, S.st>>>(ki, vi, n, shift, nchunks, B.hist, ko, vo);
        std::swap(ki, ko);
        std::swap(vi, vo);
    }
    *keys_sorted = ki;
    *vals_sorted = vi;
    S3O_CUDA(cudaGetLastError());
    return S3O_OK;
}

int sort_reserve(SortBuf &B, size_t n) {
    if (n <= B.cap) return S3O_OK;
    if (B.k0) { cudaFree(B.k0); cudaFree(B.k1); cudaFree(B.v0); cudaFree(B.v1); }
    B.cap = n;
    S3O_CUDA(cudaMalloc((void **)&B.k0, n * sizeof(uint64_t)));
    S3O_CUDA(cudaMalloc((void **)&B.k1, n * sizeof(uint64_t)));
    S3O_CUDA(cudaMalloc((void **)&B.v0, n * sizeof(int32_t)));
    S3O_CUDA(cudaMalloc((void **)&B.v1, n * sizeof(int32_t)));
    return S3O_OK;
}
void sort_free(SortBuf &B) {
    if (B.k0) { cudaFree(B.k0); cudaFree(B.k1); cudaFree(B.v0); cudaFree(B.v1); }
    if (B.hist) cudaFree(B.hist);
    B = SortBuf();
}

// ---- structure kernels --------------------------------------------------------------------------------------
__global__ void free_flag_kernel(const uint8_t *__restrict__ fixed, int nv, int32_t *__restrict__ flag) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v < nv) flag[v] = fixed[v] ? 0 : 1;
}
__global__ void hidx_kernel(const uint8_t *__restrict__ fixed, const int32_t *__restrict__ excl, int nv, int32_t *__restrict__ hidx,
                            int32_t *__restrict__ free2v) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= nv) return;
    if (fixed[v]) hidx[v] = -1;
    else { hidx[v] = excl[v]; free2v[excl[v]] = v; }
}
__global__ void free2v_kernel(const int32_t *__restrict__ hidx, int nv, int32_t *__restrict__ free2v) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v < nv && hidx[v] >= 0) free2v[hidx[v]] = v;
}
__global__ void edge_active_kernel(const int32_t *__restrict__ hidx, const int32_t *__restrict__ v0, const int32_t *__restrict__ v1,
                                   int ne, int32_t *__restrict__ act) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < ne) act[k] = (hidx[v0[k]] >= 0 || hidx[v1[k]] >= 0) ? 1 : 0;
}
// one edge's sort key: (row = min, column = max) Hessian pair; an edge with one free end sorts at (h,h)
__device__ __forceinline__ uint64_t edge_key(int hi, int hj, int bits) {
    int r, c;
    if (hi < 0) r = c = hj;
    else if (hj < 0) r = c = hi;
    else { r = min(hi, hj); c = max(hi, hj); }
    return ((uint64_t)(uint32_t)r << bits) | (uint32_t)c;
}

// active edges, in the caller's order, with their key
__global__ void edge_keys_kernel(const int32_t *__restrict__ hidx, const int32_t *__restrict__ v0, const int32_t *__restrict__ v1,
                                 int ne, const int32_t *__restrict__ excl, int bits, uint64_t *__restrict__ keys,
                                 int32_t *__restrict__ vals) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= ne) return;
    const int hi = hidx[v0[k]], hj = hidx[v1[k]];
    if (hi < 0 && hj < 0) return;
    const int pos = excl[k];
    keys[pos] = edge_key(hi, hj, bits);
    vals[pos] = k;
}
__global__ void sorted_edges_kernel(const int32_t *__restrict__ perm, const int32_t *__restrict__ v0, const int32_t *__restrict__ v1,
                                    int na, int32_t *__restrict__ sv0, int32_t *__restrict__ sv1) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= na) return;
    const int k = perm[t];
    sv0[t] = v0[k];
    sv1[t] = v1[k];
}
// first edge of each off-diagonal block
__global__ void newflag_kernel(const uint64_t *__restrict__ keys, int na, int bits, int32_t *__restrict__ newflag) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= na) return;
    const uint64_t key = keys[t];
    const int r = (int)(key >> bits), c = (int)(key & ((1ull << bits) - 1));
    newflag[t] = (c != r && (t == 0 || keys[t - 1] != key)) ? 1 : 0;
}
// first sorted position whose row is >= r (binary search), rowptr[r] = r + off-diagonal blocks before it
__global__ void rowptr_kernel(const uint64_t *__restrict__ keys, int na, int bits, const int32_t *__restrict__ excl_new,
                              int total_new, int nf, int32_t *__restrict__ rowptr, int32_t *__restrict__ colidx,
                              int32_t *__restrict__ blk_row, int32_t *__restrict__ blk_ebeg, int32_t *__restrict__ blk_eend) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r > nf) return;
    int lo = 0, hi = na;
    const uint64_t target = (uint64_t)(uint32_t)r << bits;
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (keys[mid] < target) lo = mid + 1; else hi = mid; }
    const int before = lo < na ? excl_new[lo] : total_new;
    const int b = r + before;
    rowptr[r] = b;
    if (r < nf) { colidx[b] = r; blk_row[b] = r; blk_ebeg[b] = 0; blk_eend[b] = 0; }
}
__global__ void blocks_kernel(const uint64_t *__restrict__ keys, int na, int bits, const int32_t *__restrict__ excl_new,
                              const int32_t *__restrict__ newflag, int32_t *__restrict__ e_blk, int32_t *__restrict__ colidx,
                              int32_t *__restrict__ blk_row, int32_t *__restrict__ blk_ebeg, int32_t *__restrict__ blk_eend) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= na) return;
    const uint64_t key = keys[t];
    const int r = (int)(key >> bits), c = (int)(key & ((1ull << bits) - 1));
    if (c == r) { e_blk[t] = -1; return; }
    const int b = r + excl_new[t] + newflag[t];       // r + 1 diagonal blocks up to row r, inclusive count - 1 before
    e_blk[t] = b;
    if (newflag[t]) { colidx[b] = c; blk_row[b] = r; blk_ebeg[b] = t; }
    if (t == na - 1 || keys[t + 1] != key) blk_eend[b] = t + 1;
}
__global__ void blk_src_kernel(int nb, const int32_t *__restrict__ blk_ebeg, const int32_t *__restrict__ blk_eend,
                               const int32_t *__restrict__ hidx, const int32_t *__restrict__ sv0, const int32_t *__restrict__ sv1,
                               int32_t *__restrict__ blk_src, int32_t *__restrict__ multi_flag) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nb) return;
    const int cnt = blk_eend[b] - blk_ebeg[b];
    int src = -1;
    if (cnt == 1) {
        const int t = blk_ebeg[b];
        src = (t << 1) | (hidx[sv0[t]] > hidx[sv1[t]] ? 1 : 0);
    }
    blk_src[b] = src;
    multi_flag[b] = cnt > 1 ? 1 : 0;
}
__global__ void compact_index_kernel(int n, const int32_t *__restrict__ flag, const int32_t *__restrict__ excl, int32_t *__restrict__ out) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n && flag[t]) out[excl[t]] = t;
}
// incidence candidates in (sorted edge, side) order: entry 2t = vertex(0) side, 2t+1 = vertex(1) side
__global__ void inc_flags_kernel(int na, const int32_t *__restrict__ hidx, const int32_t *__restrict__ sv0,
                                 const int32_t *__restrict__ sv1, int32_t *__restrict__ flag) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= na) return;
    flag[2 * t] = hidx[sv0[t]] >= 0 ? 1 : 0;
    flag[2 * t + 1] = hidx[sv1[t]] >= 0 ? 1 : 0;
}
__global__ void inc_keys_kernel(int na, const int32_t *__restrict__ hidx, const int32_t *__restrict__ sv0,
                                const int32_t *__restrict__ sv1, const int32_t *__restrict__ excl, uint64_t *__restrict__ keys,
                                int32_t *__restrict__ vals) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= na) return;
    const int hi = hidx[sv0[t]], hj = hidx[sv1[t]];
    if (hi >= 0) { keys[excl[2 * t]] = (uint64_t)hi; vals[excl[2 * t]] = t << 1; }
    if (hj >= 0) { keys[excl[2 * t + 1]] = (uint64_t)hj; vals[excl[2 * t + 1]] = (t << 1) | 1; }
}
// ptr[h] = first position of key >= h in the sorted key array (h = 0..n)
__global__ void segment_ptr_kernel(const uint64_t *__restrict__ keys, int m, int n, int32_t *__restrict__ ptr) {
    const int h = blockIdx.x * blockDim.x + threadIdx.x;
    if (h > n) return;
    int lo = 0, hi = m;
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (keys[mid] < (uint64_t)h) lo = mid + 1; else hi = mid; }
    ptr[h] = lo;
}
__global__ void offdiag_flag_kernel(int nb, const int32_t *__restrict__ colidx, const int32_t *__restrict__ blk_row, int32_t *__restrict__ flag) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < nb) flag[b] = colidx[b] != blk_row[b] ? 1 : 0;
}
__global__ void colT_keys_kernel(int nb, const int32_t *__restrict__ colidx, const int32_t *__restrict__ flag,
                                 const int32_t *__restrict__ excl, uint64_t *__restrict__ keys, int32_t *__restrict__ vals) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < nb && flag[b]) { keys[excl[b]] = (uint64_t)colidx[b]; vals[excl[b]] = b; }
}
// g2o-order upper block-CCS: column c = the rows of its column-view blocks (ascending), then the diagonal
__global__ void ccs_kernel(int nf, const int32_t *__restrict__ colT_ptr, const int32_t *__restrict__ colT_blk,
                           const int32_t *__restrict__ blk_row, const int32_t *__restrict__ rowptr, int32_t *__restrict__ ccs_colptr,
                           int32_t *__restrict__ ccs_rowidx, int32_t *__restrict__ ccs2bsr) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c > nf) return;
    const int p0 = colT_ptr[c] + c;
    ccs_colptr[c] = p0;
    if (c == nf) return;
    const int cnt = colT_ptr[c + 1] - colT_ptr[c];
    for (int i = 0; i < cnt; ++i) {
        const int k = colT_blk[colT_ptr[c] + i];
        ccs_rowidx[p0 + i] = blk_row[k];
        ccs2bsr[p0 + i] = k;
    }
    ccs_rowidx[p0 + cnt] = c;
    ccs2bsr[p0 + cnt] = rowptr[c];
}

// ---- merge of appended vertices / edges into a built structure ----------------------------------------------
__global__ void append_hidx_kernel(const uint8_t *__restrict__ fixed, const int32_t *__restrict__ excl, int n, int nv_old,
                                   int nf_old, int32_t *__restrict__ hidx) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v < n) hidx[nv_old + v] = fixed[v] ? -1 : nf_old + excl[v];
}
// keys of the built (sorted) edges at the new key width: the Hessian indices of old vertices do not move, so the
// order is kept
__global__ void rekey_kernel(const int32_t *__restrict__ hidx, const int32_t *__restrict__ sv0, const int32_t *__restrict__ sv1,
                             int na, int bits, uint64_t *__restrict__ keys) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < na) keys[t] = edge_key(hidx[sv0[t]], hidx[sv1[t]], bits);
}
// merged position of built edge t: t + #(new keys < key); of new edge j: j + #(built keys <= key).  Ties put the
// built edges first, which is the stable order of the concatenated caller arrays.
__device__ __forceinline__ int count_below(const uint64_t *__restrict__ keys, int n, uint64_t key, bool inclusive) {
    int lo = 0, hi = n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (keys[mid] < key || (inclusive && keys[mid] == key)) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}
__global__ void merge_old_kernel(int na_old, const uint64_t *__restrict__ okeys, const int32_t *__restrict__ operm,
                                 const int32_t *__restrict__ osv0, const int32_t *__restrict__ osv1, int na_new,
                                 const uint64_t *__restrict__ nkeys, uint64_t *__restrict__ keys, int32_t *__restrict__ perm,
                                 int32_t *__restrict__ sv0, int32_t *__restrict__ sv1, int32_t *__restrict__ pos) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= na_old) return;
    const uint64_t key = okeys[t];
    const int q = t + count_below(nkeys, na_new, key, false);
    keys[q] = key; perm[q] = operm[t]; sv0[q] = osv0[t]; sv1[q] = osv1[t];
    pos[t] = q;
}
__global__ void merge_new_kernel(int na_new, const uint64_t *__restrict__ nkeys, const int32_t *__restrict__ nperm,
                                 const int32_t *__restrict__ v0, const int32_t *__restrict__ v1, int ne_old, int na_old,
                                 const uint64_t *__restrict__ okeys, uint64_t *__restrict__ keys, int32_t *__restrict__ perm,
                                 int32_t *__restrict__ sv0, int32_t *__restrict__ sv1, int32_t *__restrict__ pos) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= na_new) return;
    const uint64_t key = nkeys[j];
    const int q = j + count_below(okeys, na_old, key, true), k = nperm[j];
    keys[q] = key; perm[q] = ne_old + k; sv0[q] = v0[k]; sv1[q] = v1[k];
    pos[j] = q;
}
// built edge records to their merged positions; information from representation rep_old to rep (0 none = identity,
// 1 diagonal planes, 2 packed upper triangles)
__global__ void move_edges_kernel(int na, const int32_t *__restrict__ pos, int est_dim, int d, int pitch_old,
                                  const double *__restrict__ meas_old, const double *__restrict__ info_old, int rep_old,
                                  int pitch, double *__restrict__ meas, double *__restrict__ info, int rep) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= na) return;
    const size_t q = (size_t)pos[t];
    for (int k = 0; k < est_dim; ++k) meas[(size_t)k * pitch + q] = meas_old[(size_t)k * pitch_old + t];
    if (rep == 1) {
        for (int r = 0; r < d; ++r) info[(size_t)r * pitch + q] = rep_old == 1 ? info_old[(size_t)r * pitch_old + t] : 1.0;
    } else if (rep == 2) {
        int f = 0;
        for (int r = 0; r < d; ++r)
            for (int c = r; c < d; ++c, ++f) {
                double v;
                if (rep_old == 2) v = info_old[(size_t)f * pitch_old + t];
                else if (r != c) v = 0.0;
                else v = rep_old == 1 ? info_old[(size_t)r * pitch_old + t] : 1.0;
                info[(size_t)f * pitch + q] = v;
            }
    }
}

template <class T>
int to_host(cudaStream_t st, std::vector<T> &dst, const T *src, size_t n) {
    dst.resize(n);
    if (n) S3O_CUDA(cudaMemcpyAsync(dst.data(), src, n * sizeof(T), cudaMemcpyDeviceToHost, st));
    return S3O_OK;
}

inline int grid_for(long long n) { return (int)std::max<long long>(1, (n + 255) / 256); }

// Device temporaries of one build (freed on exit unless taken for the caller), with the scan and sort buffers.
struct Builder {
    Scratch sc;
    SortBuf sb;
    std::vector<void *> tmp;
    explicit Builder(cudaStream_t st) { sc.st = st; }
    ~Builder() {
        for (void *ptr : tmp) cudaFree(ptr);
        if (sc.tile_sums) cudaFree(sc.tile_sums);
        if (sc.d_total) cudaFree(sc.d_total);
        sort_free(sb);
    }
    template <class T>
    T *alloc(size_t count) {
        void *ptr = nullptr;
        if (cudaMalloc(&ptr, count ? count * sizeof(T) : 16) != cudaSuccess) return nullptr;
        tmp.push_back(ptr);
        return (T *)ptr;
    }
    template <class T>
    T *take(T *ptr) {           // out of the scratch list: the caller frees it
        tmp.erase(std::find(tmp.begin(), tmp.end(), (void *)ptr));
        return ptr;
    }
};

#define SD_CHECK(call)                  \
    do {                                \
        int _rc = (call);               \
        if (_rc) return _rc;            \
    } while (0)
#define SD_ALLOC(T, name, count)                                                                   \
    T *name = B.alloc<T>((size_t)(count));                                                         \
    if (!name) { set_error("%s: out of device memory", who); return S3O_ERR_CUDA; }

// Derive half, shared by the full build and the merge.  In: the Hessian indices (nv) and free2v (nf), and the nf
// active edges sorted by key at key width `bits` with their caller ids and endpoints (all in B's list).  Out: the
// BSR-upper rows / columns / per-block edge ranges, blk_src and the multi-edge blocks, the incidences, the column view
// and the g2o block-CCS, then the host copies (all of them when keep is null; else only those the hierarchy builder,
// the factorisation plan and the getters read, and the device arrays pass to *keep).
int derive_structure(Builder &B, const char *who, int nv, int nf, int bits, int na, int32_t *d_hidx, int32_t *d_free2v,
                     const uint64_t *d_keys, int32_t *d_perm, int32_t *d_sv0, int32_t *d_sv1, HostStructure &S,
                     DeviceStructure *keep) {
    cudaStream_t st = B.sc.st;
    S.nf = nf;
    S.ne_act = na;
    SD_CHECK(sort_reserve(B.sb, (size_t)std::max(2 * (long long)na, (long long)nf + na) + 1));
    SD_ALLOC(int32_t, d_flag, 2 * (size_t)na + 2);
    SD_ALLOC(int32_t, d_excl, 2 * (size_t)na + 2);
    SD_ALLOC(int32_t, d_newflag, (size_t)na + 1);
    SD_ALLOC(int32_t, d_exnew, (size_t)na + 1);
    if (na) newflag_kernel<<<grid_for(na), 256, 0, st>>>(d_keys, na, bits, d_newflag);
    int32_t n_off = 0;
    SD_CHECK(exclusive_scan(B.sc, d_newflag, d_exnew, na, &n_off));
    const int nb = S.nb = nf + n_off;

    // ---- BSR-upper rows / columns / per-block edge ranges
    SD_ALLOC(int32_t, d_rowptr, (size_t)nf + 1);
    SD_ALLOC(int32_t, d_colidx, std::max(nb, 1));
    SD_ALLOC(int32_t, d_blk_row, std::max(nb, 1));
    SD_ALLOC(int32_t, d_ebeg, std::max(nb, 1));
    SD_ALLOC(int32_t, d_eend, std::max(nb, 1));
    SD_ALLOC(int32_t, d_e_blk, std::max(na, 1));
    rowptr_kernel<<<grid_for(nf + 1), 256, 0, st>>>(d_keys, na, bits, d_exnew, n_off, nf, d_rowptr, d_colidx, d_blk_row, d_ebeg, d_eend);
    if (na) blocks_kernel<<<grid_for(na), 256, 0, st>>>(d_keys, na, bits, d_exnew, d_newflag, d_e_blk, d_colidx, d_blk_row, d_ebeg, d_eend);
    SD_ALLOC(int32_t, d_blk_src, std::max(nb, 1));
    SD_ALLOC(int32_t, d_bflag, (size_t)nb + 1);
    SD_ALLOC(int32_t, d_bexcl, (size_t)nb + 1);
    if (nb) blk_src_kernel<<<grid_for(nb), 256, 0, st>>>(nb, d_ebeg, d_eend, d_hidx, d_sv0, d_sv1, d_blk_src, d_bflag);
    int32_t n_multi = 0;
    SD_CHECK(exclusive_scan(B.sc, d_bflag, d_bexcl, nb, &n_multi));
    SD_ALLOC(int32_t, d_multi, std::max(n_multi, 1));
    if (nb) compact_index_kernel<<<grid_for(nb), 256, 0, st>>>(nb, d_bflag, d_bexcl, d_multi);

    // ---- incidences per free vertex, ordered by sorted edge position
    int32_t n_inc = 0;
    if (na) inc_flags_kernel<<<grid_for(na), 256, 0, st>>>(na, d_hidx, d_sv0, d_sv1, d_flag);
    SD_CHECK(exclusive_scan(B.sc, d_flag, d_excl, 2 * na, &n_inc));
    if (na) inc_keys_kernel<<<grid_for(na), 256, 0, st>>>(na, d_hidx, d_sv0, d_sv1, d_excl, B.sb.k0, B.sb.v0);
    uint64_t *ikeys = nullptr;
    int32_t *ivals = nullptr;
    SD_CHECK(radix_sort(B.sc, B.sb, n_inc, bits, &ikeys, &ivals));
    SD_ALLOC(int32_t, d_inc_ptr, (size_t)nf + 1);
    SD_ALLOC(int32_t, d_inc_ent, std::max(n_inc, 1));
    segment_ptr_kernel<<<grid_for(nf + 1), 256, 0, st>>>(ikeys, n_inc, nf, d_inc_ptr);
    if (n_inc) cudaMemcpyAsync(d_inc_ent, ivals, sizeof(int32_t) * n_inc, cudaMemcpyDeviceToDevice, st);

    // ---- column view of the off-diagonal blocks (rows ascending inside a column), then the g2o block-CCS
    if (nb) offdiag_flag_kernel<<<grid_for(nb), 256, 0, st>>>(nb, d_colidx, d_blk_row, d_bflag);
    int32_t n_off2 = 0;
    SD_CHECK(exclusive_scan(B.sc, d_bflag, d_bexcl, nb, &n_off2));
    if (nb) colT_keys_kernel<<<grid_for(nb), 256, 0, st>>>(nb, d_colidx, d_bflag, d_bexcl, B.sb.k0, B.sb.v0);
    uint64_t *ckeys = nullptr;
    int32_t *cvals = nullptr;
    SD_CHECK(radix_sort(B.sc, B.sb, n_off2, bits, &ckeys, &cvals));
    SD_ALLOC(int32_t, d_colT_ptr, (size_t)nf + 1);
    SD_ALLOC(int32_t, d_colT_blk, std::max(n_off2, 1));
    segment_ptr_kernel<<<grid_for(nf + 1), 256, 0, st>>>(ckeys, n_off2, nf, d_colT_ptr);
    if (n_off2) cudaMemcpyAsync(d_colT_blk, cvals, sizeof(int32_t) * n_off2, cudaMemcpyDeviceToDevice, st);
    SD_ALLOC(int32_t, d_ccs_colptr, (size_t)nf + 1);
    SD_ALLOC(int32_t, d_ccs_rowidx, std::max(nb, 1));
    SD_ALLOC(int32_t, d_ccs2bsr, std::max(nb, 1));
    ccs_kernel<<<grid_for(nf + 1), 256, 0, st>>>(nf, d_colT_ptr, d_colT_blk, d_blk_row, d_rowptr, d_ccs_colptr, d_ccs_rowidx, d_ccs2bsr);

    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("%s: %s", who, cudaGetErrorString(e)); return S3O_ERR_CUDA; }

    // ---- back to the host structure: everything when the caller keeps no device copies, else only what host code
    // reads (hierarchy builder, factorisation plan, getters); the edge-side arrays stay on the device
    SD_CHECK(to_host(st, S.hidx, d_hidx, (size_t)nv));
    SD_CHECK(to_host(st, S.free2v, d_free2v, (size_t)nf));
    SD_CHECK(to_host(st, S.perm, d_perm, (size_t)na));
    SD_CHECK(to_host(st, S.rowptr, d_rowptr, (size_t)nf + 1));
    SD_CHECK(to_host(st, S.colidx, d_colidx, (size_t)nb));
    SD_CHECK(to_host(st, S.multi_blk, d_multi, (size_t)n_multi));
    SD_CHECK(to_host(st, S.ccs_colptr, d_ccs_colptr, (size_t)nf + 1));
    SD_CHECK(to_host(st, S.ccs_rowidx, d_ccs_rowidx, (size_t)nb));
    SD_CHECK(to_host(st, S.ccs2bsr, d_ccs2bsr, (size_t)nb));
    if (!keep) {
        SD_CHECK(to_host(st, S.sv0, d_sv0, (size_t)na));
        SD_CHECK(to_host(st, S.sv1, d_sv1, (size_t)na));
        SD_CHECK(to_host(st, S.e_blk, d_e_blk, (size_t)na));
        SD_CHECK(to_host(st, S.blk_ebeg, d_ebeg, (size_t)nb));
        SD_CHECK(to_host(st, S.blk_eend, d_eend, (size_t)nb));
        SD_CHECK(to_host(st, S.blk_src, d_blk_src, (size_t)nb));
        SD_CHECK(to_host(st, S.inc_ptr, d_inc_ptr, (size_t)nf + 1));
        SD_CHECK(to_host(st, S.inc_ent, d_inc_ent, (size_t)n_inc));
        SD_CHECK(to_host(st, S.colT_ptr, d_colT_ptr, (size_t)nf + 1));
        SD_CHECK(to_host(st, S.colT_blk, d_colT_blk, (size_t)n_off2));
    }
    e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { set_error("%s: %s", who, cudaGetErrorString(e)); return S3O_ERR_CUDA; }
    if (keep) {
        keep->hidx = B.take(d_hidx); keep->sv0 = B.take(d_sv0); keep->sv1 = B.take(d_sv1);
        keep->blk_ebeg = B.take(d_ebeg); keep->blk_eend = B.take(d_eend); keep->blk_src = B.take(d_blk_src);
        keep->multi_blk = B.take(d_multi); keep->inc_ptr = B.take(d_inc_ptr); keep->inc_ent = B.take(d_inc_ent);
        keep->e_blk = B.take(d_e_blk); keep->rowptr = B.take(d_rowptr); keep->colidx = B.take(d_colidx);
        keep->blk_row = B.take(d_blk_row); keep->colT_ptr = B.take(d_colT_ptr); keep->colT_blk = B.take(d_colT_blk);
        keep->perm = B.take(d_perm);
        keep->valid = true;
    }
    return S3O_OK;
}

inline int key_bits(int nf) {
    int bits = 1;
    while ((1ll << bits) <= nf) ++bits;
    return bits;
}

}  // namespace

// Device twin of build_structure_host / build_structure_from_hidx.  fixed (nv bytes) or hidx_in (nv ints, local
// Hessian numbering of the partitioned solve) describe the free vertices; v0 / v1 are the caller's edges.  Sort half
// here (Hessian indices, active edges sorted by key); the rest is derive_structure.
int build_structure_device(cudaStream_t st, int nv, const uint8_t *fixed, const int32_t *hidx_in, int nfree_in, int ne,
                           const int32_t *v0, const int32_t *v1, HostStructure &S, DeviceStructure *keep) {
    static const char *who = "build_structure_device";
    S = HostStructure();
    S.nv = nv;
    S.ne = ne;
    Builder B(st);
    const int nmax = std::max(std::max(nv, ne), 1);
    SD_ALLOC(int32_t, d_v0, std::max(ne, 1));
    SD_ALLOC(int32_t, d_v1, std::max(ne, 1));
    SD_ALLOC(int32_t, d_hidx, std::max(nv, 1));
    SD_ALLOC(int32_t, d_free2v, std::max(nv, 1));
    SD_ALLOC(int32_t, d_flag, (size_t)nmax + 1);
    SD_ALLOC(int32_t, d_excl, (size_t)nmax + 1);
    if (ne) {
        cudaMemcpyAsync(d_v0, v0, sizeof(int32_t) * ne, cudaMemcpyHostToDevice, st);
        cudaMemcpyAsync(d_v1, v1, sizeof(int32_t) * ne, cudaMemcpyHostToDevice, st);
    }
    // ---- Hessian indices: free vertices numbered in id order
    int nf = 0;
    if (hidx_in) {
        cudaMemcpyAsync(d_hidx, hidx_in, sizeof(int32_t) * nv, cudaMemcpyHostToDevice, st);
        nf = nfree_in;
        if (nv) free2v_kernel<<<grid_for(nv), 256, 0, st>>>(d_hidx, nv, d_free2v);
    } else {
        SD_ALLOC(uint8_t, d_fixed, std::max(nv, 1));
        if (nv) {
            if (fixed) cudaMemcpyAsync(d_fixed, fixed, nv, cudaMemcpyHostToDevice, st);
            else cudaMemsetAsync(d_fixed, 0, nv, st);
            free_flag_kernel<<<grid_for(nv), 256, 0, st>>>(d_fixed, nv, d_flag);
        }
        int32_t total = 0;
        SD_CHECK(exclusive_scan(B.sc, d_flag, d_excl, nv, &total));
        nf = total;
        if (nv) hidx_kernel<<<grid_for(nv), 256, 0, st>>>(d_fixed, d_excl, nv, d_hidx, d_free2v);
    }
    const int bits = key_bits(nf);

    // ---- active edges sorted by (min,max) Hessian pair, ties in the caller's order
    int32_t na = 0;
    if (ne) edge_active_kernel<<<grid_for(ne), 256, 0, st>>>(d_hidx, d_v0, d_v1, ne, d_flag);
    SD_CHECK(exclusive_scan(B.sc, d_flag, d_excl, ne, &na));
    SD_CHECK(sort_reserve(B.sb, (size_t)std::max(2 * (long long)na, (long long)nf + na) + 1));
    if (ne) edge_keys_kernel<<<grid_for(ne), 256, 0, st>>>(d_hidx, d_v0, d_v1, ne, d_excl, bits, B.sb.k0, B.sb.v0);
    uint64_t *skeys = nullptr;
    int32_t *sperm = nullptr;
    SD_CHECK(radix_sort(B.sc, B.sb, na, 2 * bits, &skeys, &sperm));
    // the sort buffers are reused by the derive half: keep the sorted keys / permutation in their own arrays
    SD_ALLOC(uint64_t, d_keys, std::max(na, 1));
    SD_ALLOC(int32_t, d_perm, std::max(na, 1));
    if (na) {
        cudaMemcpyAsync(d_keys, skeys, sizeof(uint64_t) * na, cudaMemcpyDeviceToDevice, st);
        cudaMemcpyAsync(d_perm, sperm, sizeof(int32_t) * na, cudaMemcpyDeviceToDevice, st);
    }
    SD_ALLOC(int32_t, d_sv0, std::max(na, 1));
    SD_ALLOC(int32_t, d_sv1, std::max(na, 1));
    if (na) sorted_edges_kernel<<<grid_for(na), 256, 0, st>>>(d_perm, d_v0, d_v1, na, d_sv0, d_sv1);
    return derive_structure(B, who, nv, nf, bits, na, d_hidx, d_free2v, d_keys, d_perm, d_sv0, d_sv1, S, keep);
}

// Merge half of s3o_build_structure on a built problem with appended vertices / edges (see StructureMerge).
int merge_structure_device(cudaStream_t st, StructureMerge &M, HostStructure &S, DeviceStructure &keep) {
    static const char *who = "s3o_build_structure (merge)";
    Builder B(st);
    const int nvn = M.nv - M.nv_old, nen = M.ne - M.ne_old;
    S = HostStructure();
    S.nv = M.nv;
    S.ne = M.ne;
    const int nmax = std::max(std::max(nvn, nen), 1);
    SD_ALLOC(int32_t, d_flag, (size_t)nmax + 1);
    SD_ALLOC(int32_t, d_excl, (size_t)nmax + 1);

    // ---- Hessian indices: the built ones, then n_free_old + the scan of the new vertices' free flags
    SD_ALLOC(int32_t, d_hidx, std::max(M.nv, 1));
    if (M.nv_old) cudaMemcpyAsync(d_hidx, M.hidx, sizeof(int32_t) * M.nv_old, cudaMemcpyDeviceToDevice, st);
    int nf = M.nf_old;
    if (nvn) {
        SD_ALLOC(uint8_t, d_fixed, nvn);
        cudaMemcpyAsync(d_fixed, M.fixed_new, nvn, cudaMemcpyHostToDevice, st);
        M.h2d_bytes += nvn;
        free_flag_kernel<<<grid_for(nvn), 256, 0, st>>>(d_fixed, nvn, d_flag);
        int32_t total = 0;
        SD_CHECK(exclusive_scan(B.sc, d_flag, d_excl, nvn, &total));
        nf += total;
        append_hidx_kernel<<<grid_for(nvn), 256, 0, st>>>(d_fixed, d_excl, nvn, M.nv_old, M.nf_old, d_hidx);
    }
    SD_ALLOC(int32_t, d_free2v, std::max(nf, 1));
    if (M.nv) free2v_kernel<<<grid_for(M.nv), 256, 0, st>>>(d_hidx, M.nv, d_free2v);
    const int bits = key_bits(nf);
    setup_mark("merge: hessian indices");

    // ---- the built edges' keys at the (possibly wider) key width; the new active edges' keys, sorted
    SD_ALLOC(uint64_t, d_okeys, std::max(M.na_old, 1));
    if (M.na_old) rekey_kernel<<<grid_for(M.na_old), 256, 0, st>>>(d_hidx, M.sv0, M.sv1, M.na_old, bits, d_okeys);
    SD_ALLOC(int32_t, d_v0, std::max(nen, 1));
    SD_ALLOC(int32_t, d_v1, std::max(nen, 1));
    int32_t na_new = 0;
    uint64_t *nkeys = nullptr;
    int32_t *nperm = nullptr;
    if (nen) {
        cudaMemcpyAsync(d_v0, M.v0_new, sizeof(int32_t) * nen, cudaMemcpyHostToDevice, st);
        cudaMemcpyAsync(d_v1, M.v1_new, sizeof(int32_t) * nen, cudaMemcpyHostToDevice, st);
        M.h2d_bytes += 8ll * nen;
        edge_active_kernel<<<grid_for(nen), 256, 0, st>>>(d_hidx, d_v0, d_v1, nen, d_flag);
        SD_CHECK(exclusive_scan(B.sc, d_flag, d_excl, nen, &na_new));
        SD_CHECK(sort_reserve(B.sb, (size_t)na_new + 1));
        edge_keys_kernel<<<grid_for(nen), 256, 0, st>>>(d_hidx, d_v0, d_v1, nen, d_excl, bits, B.sb.k0, B.sb.v0);
        SD_CHECK(radix_sort(B.sc, B.sb, na_new, 2 * bits, &nkeys, &nperm));
    }
    setup_mark("merge: keys + sort of new edges");

    // ---- merged order, edge arrays and edge records at the fresh build's pitch
    const int na = M.na_old + na_new, pitch = pad32(na);
    SD_ALLOC(uint64_t, d_keys, std::max(na, 1));
    SD_ALLOC(int32_t, d_perm, std::max(na, 1));
    SD_ALLOC(int32_t, d_sv0, std::max(na, 1));
    SD_ALLOC(int32_t, d_sv1, std::max(na, 1));
    SD_ALLOC(int32_t, d_opos, std::max(M.na_old, 1));
    SD_ALLOC(int32_t, d_npos, std::max((int)na_new, 1));
    if (M.na_old)
        merge_old_kernel<<<grid_for(M.na_old), 256, 0, st>>>(M.na_old, d_okeys, M.perm, M.sv0, M.sv1, na_new, nkeys, d_keys,
                                                              d_perm, d_sv0, d_sv1, d_opos);
    if (na_new)
        merge_new_kernel<<<grid_for(na_new), 256, 0, st>>>(na_new, nkeys, nperm, d_v0, d_v1, M.ne_old, M.na_old, d_okeys,
                                                            d_keys, d_perm, d_sv0, d_sv1, d_npos);
    const int iw = M.info_rep == 1 ? M.d : M.d * (M.d + 1) / 2;
    double *meas = B.alloc<double>((size_t)pitch * M.est_dim), *info = nullptr;
    if (!meas) { set_error("%s: out of device memory", who); return S3O_ERR_CUDA; }
    if (M.info_rep && !(info = B.alloc<double>((size_t)pitch * iw))) { set_error("%s: out of device memory", who); return S3O_ERR_CUDA; }
    if (na) {
        cudaMemsetAsync(meas, 0, (size_t)pitch * M.est_dim * sizeof(double), st);
        if (info) cudaMemsetAsync(info, 0, (size_t)pitch * iw * sizeof(double), st);
    }
    if (M.na_old)
        move_edges_kernel<<<grid_for(M.na_old), 256, 0, st>>>(M.na_old, d_opos, M.est_dim, M.d, M.ne_pad_old, M.meas, M.info,
                                                               M.info_rep_old, pitch, meas, info, M.info_rep);
    launch_pack_edges(M.meas_new, M.info_rep ? M.info_new : nullptr, nperm, na_new, pitch, M.est_dim, M.d,
                      M.info_rep == 1 ? 1 : 0, meas, info, st, d_npos);
    setup_mark("merge: merge + scatter");
    SD_CHECK(derive_structure(B, who, M.nv, nf, bits, na, d_hidx, d_free2v, d_keys, d_perm, d_sv0, d_sv1, S, &keep));
    M.meas_out = B.take(meas);
    M.info_out = info ? B.take(info) : nullptr;
    setup_mark("merge: derive");
    return S3O_OK;
}

#undef SD_CHECK
#undef SD_ALLOC

}  // namespace s3o
