// direct.h -- sparse block Cholesky of the damped Hessian on the device (the exact-solve path).
//
// Replaces g2o::LinearSolverEigen (Eigen::SimplicialLDLT: symbolic analysis once, numeric factorisation per
// LM trial; reference plug-in sites kitti_surf.cpp:553-557, :728-732, bal_example.cpp:73-83) for graphs whose
// factor stays small -- the KITTI-size, chain-dominated graphs of the reference's own pipelines, where a
// Krylov solve needs O(10^3) iterations (SURVEY.md 0.A take-away 4) and every kernel launch is pure latency.
//
//   host, once per structure (direct_host.cpp):
//     multiple-minimum-degree ordering: each round eliminates an independent set of (near-)minimum-degree
//     vertices, so the rounds are at once the fill-reducing order AND the parallel schedule (on a chain this
//     is odd-even / cyclic reduction: log2(N) rounds); the column structures fall out of the same
//     elimination-graph simulation.  Emits, in elimination order, the block pattern of L, the scatter map
//     from the BSR-upper Hessian, and for every block of L the ordered list of (L_ij, L_kj) products it
//     receives (left-looking gather: one writer per block, fixed summation order, no atomics).
//   device, per LM trial (direct.cu): ONE kernel factorises level by level (gather -> 7x7 Cholesky of the
//     pivots -> scale the columns) and runs both triangular solves; CTA barriers between phases for small
//     factors, a cooperative grid for larger ones.
#pragma once
#include <stdint.h>
#include <vector>

#include "internal.h"

namespace s3o {

struct DirectPlan {
    int n = 0;                             // block rows (free vertices)
    int nlev = 0;
    long long n_pairs = 0;                 // block products of one factorisation
    std::vector<int32_t> perm;             // [n] elimination position -> Hessian index
    std::vector<int32_t> lev_ptr;          // [nlev+1] columns (elimination positions) of each level
    // L in elimination order, column by column: blocks [cptr[j], cptr[j+1]), the pivot block first,
    // then the sub-diagonal blocks with ascending row position
    std::vector<int32_t> cptr;             // [n+1]
    std::vector<int32_t> brow;             // [nL] row position of each block
    std::vector<int32_t> src;              // [nL] (BSR block << 1) | transposed, or -1 (fill-in)
    std::vector<int32_t> upd_ptr;          // [nL+1]
    std::vector<int32_t> upd_a, upd_b;     // block pairs: target -= L[a] * L[b]^T
    std::vector<int32_t> row_ptr;          // [n+1] sub-diagonal blocks by row (forward solve)
    std::vector<int32_t> row_blk, row_col; // block index / column position, columns ascending
};

// Symbolic analysis of the BSR-upper pattern (rowptr/colidx over n block rows, diagonal first in each row).
// Returns false (plan left empty) when the factor would need more than `max_pairs` block products.
bool direct_analyze(int n, const std::vector<int32_t> &rowptr, const std::vector<int32_t> &colidx, long long max_pairs,
                    DirectPlan &plan);

// Block index of L(row, col), row >= col (elimination positions), or -1 when the block is not in the pattern.
int32_t direct_find_block(const DirectPlan &plan, int col, int row);

// Gather lists of the selected inverse Sigma = H^-1 on the pattern of L (Takahashi recurrences, direct.cu), stored
// like L ([nL][d*d], block t = Sigma(brow[t], col(t))).  For every sub-diagonal block t = (i, j), the operands of
//   Sigma_ij = -(sum_{k in S(j)} Sigma_ik L_kj) L_jj^-1
// in the order of column j's sub-diagonal blocks (L_kj is block cptr[j] + 1 + m for the m-th operand):
// sel_sig[sel_ptr[t] + m] = (Sigma block holding (i, k) << 1) | transposed (i < k: the block holds Sigma_ki).
// Diagonal blocks have empty lists (their recurrence reads column j's own sub-diagonal blocks).
void selinv_lists(const DirectPlan &plan, std::vector<int32_t> &sel_ptr, std::vector<int32_t> &sel_sig);

}  // namespace s3o
