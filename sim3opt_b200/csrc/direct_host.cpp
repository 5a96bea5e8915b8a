// direct_host.cpp -- symbolic analysis for the device sparse block Cholesky (see direct.h).
//
// Plays the role of SimplicialLDLT::analyzePattern behind g2o::LinearSolverEigen (reference plug-in site
// kitti_surf.cpp:553-557): fill-reducing ordering + pattern of the factor, once per block structure.
#include <algorithm>
#include <numeric>

#include "direct.h"

namespace s3o {

namespace {

// sorted-unique union of a and b without the two excluded ids
void merge_into(std::vector<int32_t> &a, const std::vector<int32_t> &b, int32_t skip0, int32_t skip1,
                std::vector<int32_t> &tmp) {
    tmp.clear();
    tmp.reserve(a.size() + b.size());
    size_t i = 0, j = 0;
    while (i < a.size() || j < b.size()) {
        int32_t v;
        if (j >= b.size() || (i < a.size() && a[i] < b[j])) v = a[i++];
        else if (i >= a.size() || b[j] < a[i]) v = b[j++];
        else { v = a[i]; ++i; ++j; }
        if (v != skip0 && v != skip1) tmp.push_back(v);
    }
    a.swap(tmp);
}

}  // namespace

int32_t direct_find_block(const DirectPlan &P, int col, int row) {
    if (row == col) return P.cptr[col];
    const int32_t *b = P.brow.data() + P.cptr[col] + 1, *e = P.brow.data() + P.cptr[col + 1];
    const int32_t *it = std::lower_bound(b, e, row);
    return (it != e && *it == row) ? (int32_t)(it - P.brow.data()) : -1;
}

bool direct_analyze(int n, const std::vector<int32_t> &rowptr, const std::vector<int32_t> &colidx, long long max_pairs,
                    DirectPlan &P) {
    P = DirectPlan();
    P.n = n;
    if (n == 0) return true;
    // ---- elimination graph of the block pattern (both directions)
    std::vector<std::vector<int32_t>> adj(n);
    for (int r = 0; r < n; ++r)
        for (int k = rowptr[r]; k < rowptr[r + 1]; ++k) {
            const int c = colidx[k];
            if (c != r) { adj[r].push_back(c); adj[c].push_back(r); }
        }
    for (auto &a : adj) { std::sort(a.begin(), a.end()); a.erase(std::unique(a.begin(), a.end()), a.end()); }

    // ---- multiple minimum degree: one independent set of near-minimum-degree vertices per round
    std::vector<int32_t> alive(n), pos(n, -1), stamp(n, -1), tmp;
    std::iota(alive.begin(), alive.end(), 0);
    std::vector<std::vector<int32_t>> cstruct(n);       // column structure (Hessian indices) at elimination
    P.perm.reserve(n);
    P.lev_ptr.push_back(0);
    long long pairs = 0;
    int round = 0;
    while (!alive.empty()) {
        size_t md = (size_t)n;
        for (int v : alive) md = std::min(md, adj[v].size());
        const size_t thr = std::max(md + 1, (size_t)(1.2 * (double)md));
        for (int v : alive) {
            if (adj[v].size() > thr || stamp[v] == round) continue;      // too dense, or a neighbour was picked
            // v joins this round's independent set
            for (int u : adj[v]) stamp[u] = round;
            pos[v] = (int32_t)P.perm.size();
            P.perm.push_back(v);
        }
        // eliminate the set: neighbours of each pivot become a clique
        for (int q = P.lev_ptr.back(); q < (int)P.perm.size(); ++q) {
            const int v = P.perm[q];
            cstruct[v].swap(adj[v]);
            const std::vector<int32_t> &N = cstruct[v];
            const long long c = (long long)N.size();
            pairs += c * (c + 1) / 2;
            if (pairs > max_pairs) { P = DirectPlan(); return false; }
            for (int u : N) merge_into(adj[u], N, u, v, tmp);
        }
        P.lev_ptr.push_back((int32_t)P.perm.size());
        size_t w = 0;
        for (int v : alive)
            if (pos[v] < 0) alive[w++] = v;
        alive.resize(w);
        ++round;
    }
    P.nlev = round;
    P.n_pairs = pairs;

    // ---- pattern of L, column by column in elimination order (pivot block first, rows ascending)
    P.cptr.assign(n + 1, 0);
    for (int j = 0; j < n; ++j) P.cptr[j + 1] = P.cptr[j] + 1 + (int32_t)cstruct[P.perm[j]].size();
    const int nL = P.cptr[n];
    P.brow.resize(nL);
    for (int j = 0; j < n; ++j) {
        int32_t *dst = P.brow.data() + P.cptr[j];
        dst[0] = j;
        const std::vector<int32_t> &N = cstruct[P.perm[j]];
        for (size_t t = 0; t < N.size(); ++t) dst[1 + t] = pos[N[t]];
        std::sort(dst + 1, dst + 1 + N.size());
    }
    auto find_block = [&](int col, int row) { return direct_find_block(P, col, row); };

    // ---- scatter map from the BSR-upper Hessian
    P.src.assign(nL, -1);
    for (int r = 0; r < n; ++r)
        for (int k = rowptr[r]; k < rowptr[r + 1]; ++k) {
            const int c = colidx[k];
            const int pr = pos[r], pc = pos[c];
            if (r == c) { P.src[P.cptr[pr]] = k << 1; continue; }
            const int col = std::min(pr, pc), row = std::max(pr, pc);
            const int32_t t = find_block(col, row);
            // the BSR block has the rows of vertex r; L(row, col) has the rows of the later-eliminated vertex
            if (t >= 0) P.src[t] = (k << 1) | (pr == row ? 0 : 1);
        }

    // ---- left-looking update lists: target(i,k) -= L(i,j) L(k,j)^T for every column j holding rows i >= k
    std::vector<int32_t> cnt(nL + 1, 0);
    for (int j = 0; j < n; ++j)
        for (int a = P.cptr[j] + 1; a < P.cptr[j + 1]; ++a)
            for (int b = P.cptr[j] + 1; b <= a; ++b) cnt[find_block(P.brow[b], P.brow[a]) + 1]++;
    P.upd_ptr.assign(nL + 1, 0);
    for (int t = 0; t < nL; ++t) P.upd_ptr[t + 1] = P.upd_ptr[t] + cnt[t + 1];
    P.upd_a.resize((size_t)P.upd_ptr[nL]);
    P.upd_b.resize((size_t)P.upd_ptr[nL]);
    std::vector<int32_t> fill(P.upd_ptr.begin(), P.upd_ptr.end() - 1);
    for (int j = 0; j < n; ++j)           // j ascending: every list is in column order (fixed summation order)
        for (int a = P.cptr[j] + 1; a < P.cptr[j + 1]; ++a)
            for (int b = P.cptr[j] + 1; b <= a; ++b) {
                const int32_t t = find_block(P.brow[b], P.brow[a]);
                P.upd_a[fill[t]] = a;
                P.upd_b[fill[t]] = b;
                ++fill[t];
            }

    // ---- sub-diagonal blocks by row (forward substitution gathers along rows)
    P.row_ptr.assign(n + 1, 0);
    for (int j = 0; j < n; ++j)
        for (int t = P.cptr[j] + 1; t < P.cptr[j + 1]; ++t) P.row_ptr[P.brow[t] + 1]++;
    for (int i = 0; i < n; ++i) P.row_ptr[i + 1] += P.row_ptr[i];
    P.row_blk.resize((size_t)P.row_ptr[n]);
    P.row_col.resize((size_t)P.row_ptr[n]);
    std::vector<int32_t> rfill(P.row_ptr.begin(), P.row_ptr.end() - 1);
    for (int j = 0; j < n; ++j)
        for (int t = P.cptr[j] + 1; t < P.cptr[j + 1]; ++t) {
            const int i = P.brow[t];
            P.row_blk[rfill[i]] = t;
            P.row_col[rfill[i]] = j;
            ++rfill[i];
        }
    return true;
}

void selinv_lists(const DirectPlan &P, std::vector<int32_t> &sel_ptr, std::vector<int32_t> &sel_sig) {
    const int n = P.n, nL = (int)P.brow.size();
    sel_ptr.assign(nL + 1, 0);
    for (int j = 0; j < n; ++j) {
        const int ns = P.cptr[j + 1] - P.cptr[j] - 1;
        for (int t = P.cptr[j]; t < P.cptr[j + 1]; ++t) sel_ptr[t + 1] = sel_ptr[t] + (t == P.cptr[j] ? 0 : ns);
    }
    sel_sig.resize((size_t)sel_ptr[nL]);
    for (int j = 0; j < n; ++j)
        for (int a = P.cptr[j] + 1; a < P.cptr[j + 1]; ++a) {
            const int i = P.brow[a];
            int32_t *dst = sel_sig.data() + sel_ptr[a];
            for (int b = P.cptr[j] + 1; b < P.cptr[j + 1]; ++b) {
                const int k = P.brow[b];
                // S(j) is a clique of the filled graph: (max(i, k), min(i, k)) is always a block of L
                const int32_t s = direct_find_block(P, std::min(i, k), std::max(i, k));
                *dst++ = (s << 1) | (i < k ? 1 : 0);
            }
        }
}

}  // namespace s3o
