// spmv.cu -- tiled symmetric BSR-upper SpMV  q = (H + lambda I) p,  one thread per block.
//
// Replaces the per-trial  LinearSolverEigen::solve  numeric work [EXT g2o] (SURVEY.md row a16) as
// the inner product of the PCG.  Layout facts it relies on: blocks are BSR-upper with the diagonal
// block first in every row; a tile is a run of whole block rows whose blocks are contiguous in
// memory (host packs at most TB blocks per tile; a row with more blocks has a tile of its own and
// is walked in chunks).
//
// Per tile:   stage   the tile's blocks (contiguous, <= TB*D*D doubles) into shared memory with
//                     fully coalesced streaming loads
//             phase A thread t owns block kbeg+t: reads it from shared memory once (stride D*D
//                     doubles between lanes: conflict-free) and forms both  H p_j  (row part)
//                     and  H^T p_i  (column part) in registers
//             phase B the column parts leave as one coalesced copy into T[k]; the row parts are
//                     summed per (row, component) in block order -- fixed order, no atomics --
//                     and p.q is accumulated as  sum_i p_i . (diag_i + 2 off_i)
#include "../../include/sim3opt_b200.h"
#include "kernels.cuh"
#include "reduce.cuh"

namespace s3o {

int spmv_tile_blocks(int d) { return d >= 6 ? 128 : 256; }

template <int D> struct Spmv2Cfg;
template <> struct Spmv2Cfg<7> { static constexpr int NT = 128, TB = 128; };
template <> struct Spmv2Cfg<6> { static constexpr int NT = 128, TB = 128; };
template <> struct Spmv2Cfg<4> { static constexpr int NT = 256, TB = 256; };
template <> struct Spmv2Cfg<1> { static constexpr int NT = 256, TB = 256; };

template <int D, int TB>
constexpr size_t spmv2_smem_bytes() { return sizeof(double) * (size_t)(TB * D * D + 2 * TB * D + TB); }

template <int D, int NT, int TB>
__global__ void __launch_bounds__(NT) spmv2_kernel(const double *__restrict__ H, StructDev s, int nf, double lambda,
                                                   const double *__restrict__ p, double *__restrict__ q1,
                                                   double *__restrict__ T, double *__restrict__ partials,
                                                   DevScalars *sc, int pcg_mode, int dist) {
    constexpr int DD = D * D;
    extern __shared__ double smem[];
    double *tile = smem;              // [TB*DD]
    double *ys = tile + TB * DD;      // [TB*D] row parts
    double *ts = ys + TB * D;         // [TB*D] column parts
    double *wt = ts + TB * D;         // [TB] weight of a block's row part in p.q (1: diagonal or ghost column, 2: owned off-diagonal)
    __shared__ double sh[32];
    if (pcg_mode && sc->done) return;
    const int t = threadIdx.x;
    double local = 0;
    for (int tl = blockIdx.x; tl < s.ntiles; tl += gridDim.x) {
        const int row0 = s.tile_row[tl], row1 = s.tile_row[tl + 1];
        const int kbeg = s.rowptr[row0], kend = s.rowptr[row1];
        const int nrows = row1 - row0;
        double hub1 = 0, hub2 = 0;    // running sums of a hub row walked in chunks (thread c < D)
        for (int sub = kbeg; sub < kend; sub += TB) {
            const int cnt = min(TB, kend - sub);
            // ---- stage ------------------------------------------------------------------
            const double *src = H + (size_t)sub * DD;
            for (int idx = t; idx < cnt * DD; idx += NT) tile[idx] = __ldcs(src + idx);
            // ---- phase A ----------------------------------------------------------------
            double acc[D], tt[D];
            int i = 0, j = 0;
            double pi[D], pj[D];
            for (int kl = t; kl < cnt; kl += NT) {       // NT >= TB in every configuration: one pass
                i = s.blk_row[sub + kl];
                j = s.colidx[sub + kl];
#pragma unroll
                for (int c = 0; c < D; ++c) pi[c] = p[(size_t)i * D + c];
                if (j != i) {
#pragma unroll
                    for (int c = 0; c < D; ++c) pj[c] = p[(size_t)j * D + c];
                }
            }
            __syncthreads();
            for (int kl = t; kl < cnt; kl += NT) {
                const double *Hs = tile + kl * DD;
                const bool ghost = j >= s.n_own;     // partitioned solve: the column belongs to another rank
                wt[kl] = (j == i || ghost) ? 1.0 : 2.0;
                if (j == i) {
#pragma unroll
                    for (int r = 0; r < D; ++r) {
                        double a = lambda * pi[r];
#pragma unroll
                        for (int c = 0; c < D; ++c) a += Hs[r * D + c] * pi[c];
                        acc[r] = a;
                        tt[r] = 0;
                    }
                } else {
#pragma unroll
                    for (int c = 0; c < D; ++c) tt[c] = 0;
#pragma unroll
                    for (int r = 0; r < D; ++r) {
                        double a = 0;
#pragma unroll
                        for (int c = 0; c < D; ++c) {
                            const double h = Hs[r * D + c];
                            a += h * pj[c];
                            tt[c] += h * pi[r];
                        }
                        acc[r] = a;
                    }
                }
#pragma unroll
                for (int c = 0; c < D; ++c) {
                    ys[kl * D + c] = acc[c];
                    ts[kl * D + c] = ghost ? 0.0 : tt[c];
                }
            }
            __syncthreads();
            // ---- phase B ----------------------------------------------------------------
            double *Tdst = T + (size_t)sub * D;
            for (int idx = t; idx < cnt * D; idx += NT) Tdst[idx] = ts[idx];
            if (kend - kbeg <= TB) {
                for (int w = t; w < nrows * D; w += NT) {
                    const int rl = w / D, c = w - rl * D;
                    const int row = row0 + rl;
                    const int a = s.rowptr[row] - sub, e = s.rowptr[row + 1] - sub;
                    double y = 0, yw = 0;
                    for (int kl = a; kl < e; ++kl) {
                        const double v = ys[kl * D + c];
                        y += v;
                        yw += wt[kl] * v;
                    }
                    q1[(size_t)row * D + c] = y;
                    local += p[(size_t)row * D + c] * yw;
                }
            } else if (t < D) {                         // hub row: exactly one row in this tile
                for (int kl = 0; kl < cnt; ++kl) {
                    const double v = ys[kl * D + t];
                    hub1 += v;
                    hub2 += wt[kl] * v;
                }
                if (sub + cnt >= kend) {
                    q1[(size_t)row0 * D + t] = hub1;
                    local += p[(size_t)row0 * D + t] * hub2;
                }
            }
            __syncthreads();
        }
    }
    if (!pcg_mode) return;
    const double bs = block_sum<NT>(local, sh);
    if (threadIdx.x == 0) partials[blockIdx.x] = bs;
    if (last_block(&sc->counters[3])) {
        const double pq = sum_partials<NT>(partials, gridDim.x, sh);
        if (threadIdx.x == 0) {
            // partitioned solve: a rank whose halo wait timed out poisons its p.q, the all-reduce carries the NaN to
            // every rank and they all leave the PCG through the same breakdown exit
            sc->pq = (dist && sc->halo_fail) ? nan("") : pq;
            if (!dist) fin_spmv(sc);
        }
    }
}


// ======================================================================================
// v3: the same tile algorithm with the staging done by the TMA engine.
// ======================================================================================
// Persistent CTAs walk their tiles with a two-deep shared-memory ring: one elected thread issues a
// single cp.async.bulk (global -> shared, completion on an mbarrier) for tile n+1 while the CTA
// computes tile n, so the block stream never waits on registers or on the LSU.  The bulk copy needs
// 16-byte aligned addresses and sizes; a d x d block is d*d*8 bytes (392 for d=7), so a tile that
// starts on an odd block index is fetched from 8 bytes earlier and the tile data begins at
// element 1 of the buffer (the H array carries 16 bytes of tail padding).
// Precondition (checked on the host): no block row exceeds the tile capacity.
__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(unsigned long long *bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra WAIT_LOOP;\n"
        "DONE:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void *dst, const void *src, unsigned bytes, unsigned long long *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

template <int D> struct Spmv3Cfg;
template <> struct Spmv3Cfg<7> { static constexpr int NT = 128, TB = 112; };
template <> struct Spmv3Cfg<6> { static constexpr int NT = 128, TB = 128; };
template <> struct Spmv3Cfg<4> { static constexpr int NT = 256, TB = 256; };
template <> struct Spmv3Cfg<1> { static constexpr int NT = 256, TB = 256; };

template <int D, int TB>
constexpr size_t spmv3_smem_bytes() { return sizeof(double) * (size_t)(2 * (TB * D * D + 2) + 2 * TB * D + TB) + 16; }

template <int D, int NT, int TB>
__global__ void __launch_bounds__(NT) spmv3_kernel(const double *__restrict__ H, StructDev s, int nf, double lambda,
                                                   const double *__restrict__ p, double *__restrict__ q1,
                                                   double *__restrict__ T, double *__restrict__ partials,
                                                   DevScalars *sc, int pcg_mode, int dist) {
    constexpr int DD = D * D;
    constexpr int BUF = TB * DD + 2;          // doubles per ring slot (tile + alignment slack), even
    extern __shared__ __align__(16) double smem[];
    double *ring = smem;                      // [2][BUF]
    double *ys = ring + 2 * BUF;              // [TB*D]
    double *ts = ys + TB * D;                 // [TB*D]
    double *wt = ts + TB * D;                 // [TB] p.q weight of each block's row part
    unsigned long long *bar = reinterpret_cast<unsigned long long *>(wt + TB);       // [2]
    __shared__ double sh[32];
    if (pcg_mode && sc->done) return;
    const int t = threadIdx.x;
    if (t == 0) {
        mbar_init(&bar[0], 1);
        mbar_init(&bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    auto issue = [&](int tl, int slot) {      // called by thread 0 only
        const int kb = s.rowptr[s.tile_row[tl]], ke = s.rowptr[s.tile_row[tl + 1]];
        const int shift = (int)(((size_t)kb * DD) & 1);
        const unsigned bytes = (unsigned)((((size_t)(ke - kb) * DD + shift) * 8 + 15) & ~(size_t)15);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_expect_tx(&bar[slot], bytes);
        tma_bulk_g2s(ring + slot * BUF, H + (size_t)kb * DD - shift, bytes, &bar[slot]);
    };
    double local = 0;
    int n = 0;
    if (t == 0 && (int)blockIdx.x < s.ntiles) issue(blockIdx.x, 0);
    for (int tl = blockIdx.x; tl < s.ntiles; tl += gridDim.x, ++n) {
        const int slot = n & 1;
        const int nxt = tl + gridDim.x;
        if (t == 0 && nxt < s.ntiles) issue(nxt, slot ^ 1);
        const int row0 = s.tile_row[tl], row1 = s.tile_row[tl + 1];
        const int kbeg = s.rowptr[row0], kend = s.rowptr[row1];
        const int nrows = row1 - row0, cnt = kend - kbeg;
        const int shift = (int)(((size_t)kbeg * DD) & 1);
        // gather this thread's block indices and vectors while the tile is in flight
        int i = 0, j = 0;
        double pi[D], pj[D];
        if (t < cnt) {
            i = s.blk_row[kbeg + t];
            j = s.colidx[kbeg + t];
#pragma unroll
            for (int c = 0; c < D; ++c) pi[c] = p[(size_t)i * D + c];
            if (j != i) {
#pragma unroll
                for (int c = 0; c < D; ++c) pj[c] = p[(size_t)j * D + c];
            }
        }
        mbar_wait(&bar[slot], (unsigned)((n >> 1) & 1));
        if (t < cnt) {
            const double *Hs = ring + slot * BUF + shift + t * DD;
            double acc[D], tt[D];
            const bool ghost = j >= s.n_own;          // partitioned solve: column owned by another rank
            wt[t] = (j == i || ghost) ? 1.0 : 2.0;
            if (j == i) {
#pragma unroll
                for (int r = 0; r < D; ++r) {
                    double a = lambda * pi[r];
#pragma unroll
                    for (int c = 0; c < D; ++c) a += Hs[r * D + c] * pi[c];
                    acc[r] = a;
                    tt[r] = 0;
                }
            } else {
#pragma unroll
                for (int c = 0; c < D; ++c) tt[c] = 0;
#pragma unroll
                for (int r = 0; r < D; ++r) {
                    double a = 0;
#pragma unroll
                    for (int c = 0; c < D; ++c) {
                        const double h = Hs[r * D + c];
                        a += h * pj[c];
                        tt[c] += h * pi[r];
                    }
                    acc[r] = a;
                }
            }
#pragma unroll
            for (int c = 0; c < D; ++c) {
                ys[t * D + c] = acc[c];
                ts[t * D + c] = ghost ? 0.0 : tt[c];
            }
        }
        __syncthreads();
        double *Tdst = T + (size_t)kbeg * D;
        for (int idx = t; idx < cnt * D; idx += NT) Tdst[idx] = ts[idx];
        for (int w = t; w < nrows * D; w += NT) {
            const int rl = w / D, c = w - rl * D;
            const int row = row0 + rl;
            const int a = s.rowptr[row] - kbeg, e = s.rowptr[row + 1] - kbeg;
            double y = 0, yw = 0;
            for (int kl = a; kl < e; ++kl) {
                const double v = ys[kl * D + c];
                y += v;
                yw += wt[kl] * v;
            }
            q1[(size_t)row * D + c] = y;
            local += p[(size_t)row * D + c] * yw;
        }
        __syncthreads();
    }
    if (!pcg_mode) return;
    const double bs = block_sum<NT>(local, sh);
    if (threadIdx.x == 0) partials[blockIdx.x] = bs;
    if (last_block(&sc->counters[3])) {
        const double pq = sum_partials<NT>(partials, gridDim.x, sh);
        if (threadIdx.x == 0) {
            // partitioned solve: a rank whose halo wait timed out poisons its p.q, the all-reduce carries the NaN to
            // every rank and they all leave the PCG through the same breakdown exit
            sc->pq = (dist && sc->halo_fail) ? nan("") : pq;
            if (!dist) fin_spmv(sc);
        }
    }
}


// ======================================================================================
// v4: v3 with every global-load latency taken off the per-tile critical path.
// ======================================================================================
// ncu on v3 (profiles/r1_spmv3_s1m.summary.txt): DRAM 55 % busy, 12 % of the warp slots active --
// per tile a CTA pays three dependent global round trips in sequence (tile descriptor -> block
// indices -> p gathers; then rowptr again in phase B) while only one bulk copy is in flight.
// Here the CTA's tile descriptors are staged in shared memory once, block indices are fetched two
// tiles ahead and the p vectors / row segments one tile ahead (register double buffering), and the
// ring is NS deep, so an iteration only waits on the mbarrier of a tile issued NS-1 tiles ago.
template <int D, int NT, int TB, int NS, int KMAX>
__global__ void __launch_bounds__(NT) spmv4_kernel(const double *__restrict__ H, StructDev s, int nf, double lambda,
                                                   const double *__restrict__ p, double *__restrict__ q1,
                                                   double *__restrict__ T, double *__restrict__ partials,
                                                   DevScalars *sc, int pcg_mode, int dist) {
    constexpr int DD = D * D;
    constexpr int BUF = TB * DD + 2;          // doubles per ring slot (tile + alignment slack), even
    extern __shared__ __align__(16) double smem[];
    double *ring = smem;                      // [NS][BUF]
    double *ys = ring + NS * BUF;             // [TB*D]
    double *ts = ys + TB * D;                 // [TB*D]
    double *wt = ts + TB * D;                 // [TB]
    unsigned long long *bar = reinterpret_cast<unsigned long long *>(wt + TB);       // [NS]
    int *drow = reinterpret_cast<int *>(bar + NS);     // [KMAX+1] first row of my k-th tile (and one past)
    int *dblk = drow + KMAX + 1;                       // [KMAX+1] first block of my k-th tile
    __shared__ double sh[32];
    if (pcg_mode && sc->done) return;
    const int t = threadIdx.x, G = gridDim.x;
    const int ntl = ((int)blockIdx.x < s.ntiles) ? (s.ntiles - 1 - (int)blockIdx.x) / G + 1 : 0;   // my tiles
    if (t == 0) {
#pragma unroll
        for (int k = 0; k < NS; ++k) mbar_init(&bar[k], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // descriptors: row range [drow[2k], drow[2k+1]) would need two arrays; tiles of one CTA are not
    // adjacent, so keep begin and end separately: drow[k] = tile_row[tl], and the end is re-read as
    // tile_row[tl+1] into the second half of the arrays
    int *drow_e = dblk + KMAX + 1, *dblk_e = drow_e + KMAX + 1;
    for (int k = t; k < ntl; k += NT) {
        const int tl = blockIdx.x + k * G;
        const int r0 = s.tile_row[tl], r1 = s.tile_row[tl + 1];
        drow[k] = r0; drow_e[k] = r1;
        dblk[k] = s.rowptr[r0]; dblk_e[k] = s.rowptr[r1];
    }
    __syncthreads();
    auto issue = [&](int k, int slot) {       // thread 0 only: bulk copy of my k-th tile
        const int kb = dblk[k], ke = dblk_e[k];
        const int shift = (int)(((size_t)kb * DD) & 1);
        const unsigned bytes = (unsigned)((((size_t)(ke - kb) * DD + shift) * 8 + 15) & ~(size_t)15);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_expect_tx(&bar[slot], bytes);
        tma_bulk_g2s(ring + slot * BUF, H + (size_t)kb * DD - shift, bytes, &bar[slot]);
    };
    if (t == 0)
        for (int k = 0; k < NS - 1 && k < ntl; ++k) issue(k, k);
    // register pipeline: (i, j, pi, pj, ra, re) belong to the tile computed now, (ib, jb) to the next
    int i = 0, j = 0, ib = 0, jb = 0, ra = 0, re = 0;
    double pi[D], pj[D];
#pragma unroll
    for (int c = 0; c < D; ++c) { pi[c] = 0; pj[c] = 0; }
    if (ntl > 0) {
        const int kb = dblk[0], cnt = dblk_e[0] - kb;
        if (t < cnt) {
            i = s.blk_row[kb + t]; j = s.colidx[kb + t];
#pragma unroll
            for (int c = 0; c < D; ++c) pi[c] = p[(size_t)i * D + c];
            if (j != i) {
                if (s.ghost_src && j >= s.n_own) {       // ghost column: read the owner's p over NVLink
                    const double *src = s.ghost_src[j - s.n_own];
#pragma unroll
                    for (int c = 0; c < D; ++c) pj[c] = __ldcg(src + c);
                } else {
#pragma unroll
                    for (int c = 0; c < D; ++c) pj[c] = p[(size_t)j * D + c];
                }
            }
        }
        const int nrows = drow_e[0] - drow[0];
        if (t < nrows * D) { const int row = drow[0] + t / D; ra = s.rowptr[row]; re = s.rowptr[row + 1]; }
    }
    if (ntl > 1) {
        const int kb = dblk[1], cnt = dblk_e[1] - kb;
        if (t < cnt) { ib = s.blk_row[kb + t]; jb = s.colidx[kb + t]; }
    }
    double local = 0;
    for (int n = 0; n < ntl; ++n) {
        const int slot = n % NS;
        if (t == 0 && n + NS - 1 < ntl) issue(n + NS - 1, (n + NS - 1) % NS);
        // ---- prefetch: indices of tile n+2, vectors and row segment of tile n+1 -------------
        int i2 = 0, j2 = 0, ran = 0, ren = 0;
        double pin[D], pjn[D];
        if (n + 2 < ntl) {
            const int kb = dblk[n + 2], cnt = dblk_e[n + 2] - kb;
            if (t < cnt) { i2 = __ldg(s.blk_row + kb + t); j2 = __ldg(s.colidx + kb + t); }
        }
        if (n + 1 < ntl) {
            const int cnt = dblk_e[n + 1] - dblk[n + 1];
            if (t < cnt) {
#pragma unroll
                for (int c = 0; c < D; ++c) pin[c] = p[(size_t)ib * D + c];
                if (jb != ib) {
                    if (s.ghost_src && jb >= s.n_own) {
                        const double *src = s.ghost_src[jb - s.n_own];
#pragma unroll
                        for (int c = 0; c < D; ++c) pjn[c] = __ldcg(src + c);
                    } else {
#pragma unroll
                        for (int c = 0; c < D; ++c) pjn[c] = p[(size_t)jb * D + c];
                    }
                }
            }
            const int nrows = drow_e[n + 1] - drow[n + 1];
            if (t < nrows * D) { const int row = drow[n + 1] + t / D; ran = __ldg(s.rowptr + row); ren = __ldg(s.rowptr + row + 1); }
        }
        // ---- tile n --------------------------------------------------------------------------
        const int row0 = drow[n], row1 = drow_e[n];
        const int kbeg = dblk[n], kend = dblk_e[n];
        const int nrows = row1 - row0, cnt = kend - kbeg;
        const int shift = (int)(((size_t)kbeg * DD) & 1);
        mbar_wait(&bar[slot], (unsigned)((n / NS) & 1));
        if (t < cnt) {
            const double *Hs = ring + slot * BUF + shift + t * DD;
            double acc[D], tt[D];
            const bool ghost = j >= s.n_own;          // partitioned solve: column owned by another rank
            wt[t] = (j == i || ghost) ? 1.0 : 2.0;
            if (j == i) {
#pragma unroll
                for (int r = 0; r < D; ++r) {
                    double a = lambda * pi[r];
#pragma unroll
                    for (int c = 0; c < D; ++c) a += Hs[r * D + c] * pi[c];
                    acc[r] = a;
                    tt[r] = 0;
                }
            } else {
#pragma unroll
                for (int c = 0; c < D; ++c) tt[c] = 0;
#pragma unroll
                for (int r = 0; r < D; ++r) {
                    double a = 0;
#pragma unroll
                    for (int c = 0; c < D; ++c) {
                        const double h = Hs[r * D + c];
                        a += h * pj[c];
                        tt[c] += h * pi[r];
                    }
                    acc[r] = a;
                }
            }
#pragma unroll
            for (int c = 0; c < D; ++c) {
                ys[t * D + c] = acc[c];
                ts[t * D + c] = ghost ? 0.0 : tt[c];
            }
        }
        __syncthreads();
        double *Tdst = T + (size_t)kbeg * D;
        for (int idx = t; idx < cnt * D; idx += NT) Tdst[idx] = ts[idx];
        for (int w = t; w < nrows * D; w += NT) {
            const int rl = w / D, c = w - rl * D;
            const int row = row0 + rl;
            const int a = (w == t ? ra : s.rowptr[row]) - kbeg, e = (w == t ? re : s.rowptr[row + 1]) - kbeg;
            double y = 0, yw = 0;
            for (int kl = a; kl < e; ++kl) {
                const double v = ys[kl * D + c];
                y += v;
                yw += wt[kl] * v;
            }
            q1[(size_t)row * D + c] = y;
            local += p[(size_t)row * D + c] * yw;
        }
        __syncthreads();
        // ---- rotate the register pipeline ---------------------------------------------------
        i = ib; j = jb; ib = i2; jb = j2; ra = ran; re = ren;
#pragma unroll
        for (int c = 0; c < D; ++c) { pi[c] = pin[c]; pj[c] = pjn[c]; }
    }
    if (!pcg_mode) return;
    const double bs = block_sum<NT>(local, sh);
    if (threadIdx.x == 0) partials[blockIdx.x] = bs;
    if (last_block(&sc->counters[3])) {
        const double pq = sum_partials<NT>(partials, gridDim.x, sh);
        if (threadIdx.x == 0) {
            // partitioned solve: a rank whose halo wait timed out poisons its p.q, the all-reduce carries the NaN to
            // every rank and they all leave the PCG through the same breakdown exit
            sc->pq = (dist && sc->halo_fail) ? nan("") : pq;
            if (!dist) fin_spmv(sc);
        }
    }
}

// d = 7 configurations of v4: (tile blocks, ring depth)
struct Spmv4Cfg { static constexpr int NT = 128, KMAX = 384; };
template <int TB, int NS>
constexpr size_t spmv4_smem_bytes() {
    return sizeof(double) * (size_t)(NS * (TB * 49 + 2) + 2 * TB * 7 + TB) + 8 * NS + 4 * 4 * (Spmv4Cfg::KMAX + 1) + 16;
}
// cfg 0: TB=112 NS=2, 1: TB=80 NS=3, 2: TB=56 NS=4 (S3O_SPMV4_CFG, per problem).  The tiles are cut for the TB of
// the problem's cfg, so launch_spmv4 must get that same cfg: a smaller TB overruns the ring slot and ys / ts / wt.
int spmv4_tile_blocks(int cfg) { return cfg == 0 ? 112 : (cfg == 1 ? 80 : 56); }
// persistent grid: grid_cap CTAs (2 per SM); a graph with more than grid_cap * KMAX tiles gets the next
// multiple of grid_cap that keeps every CTA's descriptor list within KMAX
static int spmv4_grid(int ntiles, int grid_cap) {
    if (ntiles <= grid_cap) return ntiles;
    const int waves = (int)(((long long)ntiles + (long long)grid_cap * Spmv4Cfg::KMAX - 1) / ((long long)grid_cap * Spmv4Cfg::KMAX));
    return grid_cap * waves;
}
bool spmv4_fits(int ntiles, int grid_cap) {
    const int grid = spmv4_grid(ntiles, grid_cap);
    return grid > 0 && grid <= kMaxPartials && (ntiles + grid - 1) / grid <= Spmv4Cfg::KMAX;
}

void launch_spmv4(const double *H, const StructDev &s, int nf, double lambda, const double *p, double *q1, double *T,
                  double *partials, DevScalars *sc, int pcg_mode, int cfg, int grid_cap, int dist, cudaStream_t st) {
    if (nf == 0 || s.ntiles == 0) return;
    const int grid = spmv4_grid(s.ntiles, grid_cap);
    constexpr int NT = Spmv4Cfg::NT, KM = Spmv4Cfg::KMAX;
    switch (cfg) {
    case 0: spmv4_kernel<7, NT, 112, 2, KM><<<grid, NT, spmv4_smem_bytes<112, 2>(), st>>>(H, s, nf, lambda, p, q1, T, partials, sc, pcg_mode, dist); break;
    case 1: spmv4_kernel<7, NT, 80, 3, KM><<<grid, NT, spmv4_smem_bytes<80, 3>(), st>>>(H, s, nf, lambda, p, q1, T, partials, sc, pcg_mode, dist); break;
    case 2: spmv4_kernel<7, NT, 56, 4, KM><<<grid, NT, spmv4_smem_bytes<56, 4>(), st>>>(H, s, nf, lambda, p, q1, T, partials, sc, pcg_mode, dist); break;
    }
}

int spmv3_tile_blocks(int d) { return d == 7 ? Spmv3Cfg<7>::TB : (d == 6 ? Spmv3Cfg<6>::TB : 256); }

void launch_spmv3(int d, const double *H, const StructDev &s, int nf, double lambda, const double *p, double *q1,
                  double *T, double *partials, DevScalars *sc, int pcg_mode, int grid_cap, int dist, cudaStream_t st) {
    if (nf == 0 || s.ntiles == 0) return;
    const int grid = s.ntiles < grid_cap ? s.ntiles : grid_cap;
#define S3O_SPMV3(D)                                                                                              \
    spmv3_kernel<D, Spmv3Cfg<D>::NT, Spmv3Cfg<D>::TB><<<grid, Spmv3Cfg<D>::NT, spmv3_smem_bytes<D, Spmv3Cfg<D>::TB>(), st>>>( \
        H, s, nf, lambda, p, q1, T, partials, sc, pcg_mode, dist);
    switch (d) {
    case 7: S3O_SPMV3(7) break;
    case 4: S3O_SPMV3(4) break;
    case 6: S3O_SPMV3(6) break;
    case 1: S3O_SPMV3(1) break;
    }
#undef S3O_SPMV3
}

static int g_spmv2_ready = 0;

int spmv2_configure() {
    if (g_spmv2_ready) return 0;
    cudaError_t e;
    e = cudaFuncSetAttribute(spmv2_kernel<7, Spmv2Cfg<7>::NT, Spmv2Cfg<7>::TB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)spmv2_smem_bytes<7, Spmv2Cfg<7>::TB>());
    if (e != cudaSuccess) return -1;
    e = cudaFuncSetAttribute(spmv2_kernel<6, Spmv2Cfg<6>::NT, Spmv2Cfg<6>::TB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)spmv2_smem_bytes<6, Spmv2Cfg<6>::TB>());
    if (e != cudaSuccess) return -1;
    e = cudaFuncSetAttribute(spmv3_kernel<6, Spmv3Cfg<6>::NT, Spmv3Cfg<6>::TB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)spmv3_smem_bytes<6, Spmv3Cfg<6>::TB>());
    if (e != cudaSuccess) return -1;
    e = cudaFuncSetAttribute(spmv2_kernel<4, Spmv2Cfg<4>::NT, Spmv2Cfg<4>::TB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)spmv2_smem_bytes<4, Spmv2Cfg<4>::TB>());
    if (e != cudaSuccess) return -1;
    e = cudaFuncSetAttribute(spmv2_kernel<1, Spmv2Cfg<1>::NT, Spmv2Cfg<1>::TB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)spmv2_smem_bytes<1, Spmv2Cfg<1>::TB>());
    if (e != cudaSuccess) return -1;
    e = cudaFuncSetAttribute(spmv3_kernel<7, Spmv3Cfg<7>::NT, Spmv3Cfg<7>::TB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)spmv3_smem_bytes<7, Spmv3Cfg<7>::TB>());
    if (e != cudaSuccess) return -1;
    e = cudaFuncSetAttribute(spmv3_kernel<4, Spmv3Cfg<4>::NT, Spmv3Cfg<4>::TB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)spmv3_smem_bytes<4, Spmv3Cfg<4>::TB>());
    if (e != cudaSuccess) return -1;
    e = cudaFuncSetAttribute(spmv3_kernel<1, Spmv3Cfg<1>::NT, Spmv3Cfg<1>::TB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)spmv3_smem_bytes<1, Spmv3Cfg<1>::TB>());
    if (e != cudaSuccess) return -1;
    if (cudaFuncSetAttribute(spmv4_kernel<7, Spmv4Cfg::NT, 112, 2, Spmv4Cfg::KMAX>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)spmv4_smem_bytes<112, 2>()) != cudaSuccess) return -1;
    if (cudaFuncSetAttribute(spmv4_kernel<7, Spmv4Cfg::NT, 80, 3, Spmv4Cfg::KMAX>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)spmv4_smem_bytes<80, 3>()) != cudaSuccess) return -1;
    if (cudaFuncSetAttribute(spmv4_kernel<7, Spmv4Cfg::NT, 56, 4, Spmv4Cfg::KMAX>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)spmv4_smem_bytes<56, 4>()) != cudaSuccess) return -1;
    g_spmv2_ready = 1;
    return 0;
}

void launch_spmv2(int d, const double *H, const StructDev &s, int nf, double lambda, const double *p, double *q1,
                  double *T, double *partials, DevScalars *sc, int pcg_mode, int dist, cudaStream_t st) {
    if (nf == 0 || s.ntiles == 0) return;
    const int cap = 148 * 24;   // persistent-style grid: a multiple of the SM count, <= kMaxPartials
    const int grid = s.ntiles < cap ? s.ntiles : cap;
#define S3O_SPMV2(D)                                                                                              \
    spmv2_kernel<D, Spmv2Cfg<D>::NT, Spmv2Cfg<D>::TB><<<grid, Spmv2Cfg<D>::NT, spmv2_smem_bytes<D, Spmv2Cfg<D>::TB>(), st>>>( \
        H, s, nf, lambda, p, q1, T, partials, sc, pcg_mode, dist);
    switch (d) {
    case 7: S3O_SPMV2(7) break;
    case 4: S3O_SPMV2(4) break;
    case 6: S3O_SPMV2(6) break;
    case 1: S3O_SPMV2(1) break;
    }
#undef S3O_SPMV2
}

}  // namespace s3o
