"""CPU tests of the gates the GPU tests of the sparse block Cholesky (csrc/direct.cu) are judged by.

A Python twin of direct.cu's schedule rule (which rounds run on the cooperative grid, how many CTAs it has, and which
pivot/scale branch each round takes), and three long-double gates on what the device returns:
  factor     A - L L^T on the pattern of L (fill-in included), entrywise against an envelope derived from the operations
             direct.cu performs: fixed-order gather sums, the per-pivot Cholesky, and the sub-diagonal rows multiplied
             by the explicit inverse L_kk^-T; pivots and their inverses exactly lower triangular, and
             |L_kk Linv_k - I| <= gamma_D |L_kk| |Linv_k| (column-by-column forward substitution bounds this product);
  solve      the componentwise backward error of x against A, bounded by the forward and backward substitutions'
             envelopes plus the factor's;
  selinv     the residual of both Takahashi recurrences (direct.cu, above SelinvDev) on every block of the pattern of L,
             from the device's Sigma, L and Linv.
Each gate is shown to accept an honest fp64 evaluation done in another summation order (numpy / LAPACK) and to reject
planted faults -- the ways a kernel branch goes subtly wrong -- by at least 100x.
"""
import numpy as np
import pytest
import scipy.linalg as sla

import sim3opt_b200 as s3

NT = 512                    # kDirectNT, threads per CTA of direct_kernel / selinv_kernel
U = 2.0 ** -53
ETA = 2.0 ** -1074          # a product that underflows into the subnormals is off by up to this much, absolutely
LD = np.longdouble


def gamma(n):
    n = np.asarray(n, dtype=float)
    return n * U / (1 - n * U)


# ---- patterns (n vertices, edges v0 - v1, no fixed vertex) ----------------------------------------------------------
def chain(n, loop=True):
    v0, v1 = np.arange(n - 1), np.arange(1, n)
    if loop:
        v0, v1 = np.r_[v0, 0], np.r_[v1, n - 1]
    return n, v0.astype(np.int32), v1.astype(np.int32)


def pairs(m):
    return 2 * m, np.arange(0, 2 * m, 2, dtype=np.int32), np.arange(1, 2 * m, 2, dtype=np.int32)


def diagonal(n):
    return n, np.zeros(0, np.int32), np.zeros(0, np.int32)


def plan_of(n, v0, v1, fixed=None):
    plan = s3.host_direct_plan(n, fixed, v0, v1, max_pairs=60000000)
    plan["bcol"] = np.repeat(np.arange(plan["n"]), np.diff(plan["cptr"]))
    return plan


# ---- the schedule rule of plan_and_upload and dk_pivot_scale --------------------------------------------------------
def schedule_twin(plan, d, sms, nt=NT):
    """Grid, wide rounds, and per round whether dk_pivot_scale takes its many-column branch (one thread per pivot,
    barrier, one thread per block row: more than 2 * warps columns) or one warp per column."""
    lp, cptr = plan["lev_ptr"], plan["cptr"]
    cols = np.diff(lp)
    blocks = cptr[lp[1:]] - cptr[lp[:-1]]
    items = blocks.astype(np.int64) * d * d
    wide = int(np.flatnonzero(items > 8 * nt).max()) + 1 if (items > 8 * nt).any() else 0
    grid = 0
    if wide:
        grid = max(1, min(sms, -(-int(items.max()) // (4 * nt))))
        if grid <= 1:
            wide = 0
    warps = [(grid * nt if lev < wide else nt) // 32 for lev in range(plan["rounds"])]
    many = [bool(c > 2 * w) for c, w in zip(cols, warps)]
    return dict(n=plan["n"], rounds=plan["rounds"], blocks=len(plan["brow"]), grid=grid, wide=wide,
                cols=[int(c) for c in cols], level_blocks=[int(b) for b in blocks], many=many)


REGIMES = {
    "single": lambda s: s["grid"] <= 1 and not any(s["many"]),
    "single_many": lambda s: s["grid"] <= 1 and any(s["many"]),
    "grid_tail_warp": lambda s: s["grid"] > 1 and 0 < s["wide"] < s["rounds"] and not any(s["many"]),
    "grid_many": lambda s: s["grid"] > 1 and any(s["many"][:s["wide"]]),
    "all_wide": lambda s: s["grid"] > 1 and s["wide"] == s["rounds"] and s["many"][0],
    "diagonal": lambda s: s["grid"] > 1 and s["rounds"] == 1 and s["wide"] == 1,
}


# ---- values ------------------------------------------------------------------------------------------------------------
def bsr_blocks(n, v0, v1, hidx=None):
    """BSR-upper block list in the library's order (rows ascending, diagonal first, then columns ascending)."""
    hidx = np.arange(n) if hidx is None else hidx
    rows = [set() for _ in range(int(hidx.max()) + 1)]
    for a, b in zip(v0, v1):
        ha, hb = hidx[a], hidx[b]
        if ha >= 0 and hb >= 0 and ha != hb:
            rows[min(ha, hb)].add(max(ha, hb))
    out = []
    for r in range(len(rows)):
        out.append((r, r))
        out += [(r, c) for c in sorted(rows[r])]
    return out


def spd_values(blocks, nf, d, seed, dominance=1.0):
    """Random blocks in BSR order of an SPD matrix (block diagonally dominant by `dominance` >= 1 times the spectral norms
    of each row's off-diagonal blocks); the off-diagonal blocks are dense and not symmetric, so a transposed operand
    shows."""
    rng = np.random.default_rng(seed)
    Hb = rng.standard_normal((len(blocks), d, d))
    shift = np.ones(nf)
    for k, (r, c) in enumerate(blocks):
        if r != c:
            nrm = np.linalg.norm(Hb[k], 2)
            shift[r] += nrm
            shift[c] += nrm
    for k, (r, c) in enumerate(blocks):
        if r == c:
            Hb[k] = Hb[k] @ Hb[k].T / d + dominance * shift[r] * np.eye(d)
    return Hb


def ccs_of(blocks, Hb):
    """The upper block-CCS of s3o_linsolver_solve (columns, rows ascending) for a BSR-ordered block list."""
    order = sorted(range(len(blocks)), key=lambda k: (blocks[k][1], blocks[k][0]))
    nf = max(c for _, c in blocks) + 1
    colptr = np.zeros(nf + 1, np.int32)
    for _, c in blocks:
        colptr[c + 1] += 1
    return np.cumsum(colptr).astype(np.int32), np.array([blocks[k][0] for k in order], np.int32), Hb[order]


def scatter(plan, Hb, lam):
    """A = P (H + lam I) P^T on the pattern of L, exactly (long double), block t = A(brow[t], col t), zero on fill-in."""
    src, d = plan["src"], Hb.shape[1]
    A = np.zeros((len(src), d, d), LD)
    on = src >= 0
    M = Hb[src[on] >> 1].astype(LD)
    tr = (src[on] & 1) == 1
    M[tr] = M[tr].swapaxes(1, 2)
    A[on] = M
    A[plan["cptr"][:-1]] += LD(lam) * np.eye(d, dtype=LD)
    return A


def dense_of(plan, A):
    """Dense P (H + lam I) P^T (elimination order) from the scattered blocks."""
    n, d = plan["n"], A.shape[1]
    M = np.zeros((n * d, n * d))
    for t, (i, j) in enumerate(zip(plan["brow"], plan["bcol"])):
        M[i * d:i * d + d, j * d:j * d + d] = A[t]
        M[j * d:j * d + d, i * d:i * d + d] = A[t].T
    return M


def _ratio(R, env):
    R, env = np.abs(R), np.asarray(env)
    out = np.zeros(R.shape)
    pos = env > 0
    out[pos] = (R[pos] / env[pos]).astype(float)
    out[~pos & (R > 0)] = np.inf
    return float(out.max()) if out.size else 0.0


def _t(M):
    return M.swapaxes(-1, -2)


def _segsum(P, ptr):
    """Sums of the contiguous segments [ptr[t], ptr[t+1]) of P (zero for empty segments)."""
    out = np.zeros((len(ptr) - 1,) + P.shape[1:], P.dtype)
    cnt = np.diff(ptr)
    if len(P):
        out[cnt > 0] = np.add.reduceat(P, ptr[:-1][cnt > 0], axis=0)
    return out


# ---- gates -------------------------------------------------------------------------------------------------------------
def factor_gate(plan, A, L, Linv):
    """(ratio, inverse ratio, envelope): worst |A - L L^T| / envelope over every entry of the pattern of L, worst
    |L_kk Linv_k - I| / (gamma_D |L_kk| |Linv_k|); a ratio <= 1 passes.  Asserts the exact zeros first."""
    d = A.shape[1]
    cptr, brow, bcol = plan["cptr"], plan["brow"], plan["bcol"]
    piv = cptr[:-1]
    iu = np.triu_indices(d, 1)
    assert (L[piv][:, iu[0], iu[1]] == 0).all(), "a pivot block is not lower triangular"
    assert (Linv[:, iu[0], iu[1]] == 0).all(), "an inverse pivot block is not lower triangular"
    Lq = L.astype(LD)
    La = np.abs(Lq)
    ptr, ua, ub = plan["upd_ptr"], plan["upd_a"], plan["upd_b"]
    G = A - _segsum(Lq[ua] @ _t(Lq[ub]), ptr)                  # the exact gather of the device's operands
    S = np.abs(A) + _segsum(La[ua] @ _t(La[ub]), ptr)
    # nq products of D terms, then the subtraction; fill-in far from the diagonal decays into the subnormals
    genv = gamma(np.diff(ptr) + d + 1)[:, None, None] * S + ((np.diff(ptr) + 2) * d * ETA)[:, None, None]
    Lk = Lq[cptr[bcol]]
    R = G - Lq @ _t(Lk)
    env = genv.copy()
    dg = brow == bcol
    env[dg] += gamma(d + 1) * (La[dg] @ _t(La[dg]))           # Cholesky of the pivot
    off = ~dg
    Lia = np.abs(Linv.astype(LD))
    # L_ik = fl(G Linv^T): |E| <= gamma_D |G| |Linv^T|, and G (L Linv - I)^T: gamma_D |G| |Linv^T| |L^T| once more
    env[off] += 2 * gamma(d) * ((np.abs(G[off]) + genv[off]) @ _t(Lia[bcol[off]]) @ _t(La[cptr[bcol[off]]]))
    env += 2 * d * ETA
    F = Lq[piv] @ Linv.astype(LD) - np.eye(d, dtype=LD)
    return _ratio(R, env), _ratio(F, gamma(d) * (La[piv] @ Lia) + d * ETA), env


def _bmul(plan, M, v, transpose=False, strict=False):
    """y = sum over blocks t = (i, j) of M_t v_j into row i (or M_t^T v_i into row j); one triangle of the pattern."""
    brow, bcol = plan["brow"], plan["bcol"]
    sel = brow != bcol if strict else np.ones(len(brow), bool)
    i, j, Mt = brow[sel], bcol[sel], M[sel]
    y = np.zeros(v.shape, v.dtype)
    if transpose:
        np.add.at(y, j, np.einsum("tab,ta->tb", Mt, v[i]))
    else:
        np.add.at(y, i, np.einsum("tab,tb->ta", Mt, v[j]))
    return y


def solve_gate(plan, A, L, Linv, fenv, x, b):
    """Worst |b - A x| / envelope, componentwise (elimination order inside; x, b in Hessian order, n x d)."""
    d = A.shape[1]
    perm, cptr = plan["perm"], plan["cptr"]
    xe = np.asarray(x, float).reshape(-1, d)[perm].astype(LD)
    be = np.asarray(b, float).reshape(-1, d)[perm].astype(LD)
    r = be - _bmul(plan, A, xe) - _bmul(plan, A, xe, transpose=True, strict=True)
    Lq, La = L.astype(LD), np.abs(L.astype(LD))
    Lia = np.abs(Linv.astype(LD))
    Pa = La[cptr[:-1]]
    xa = np.abs(xe)
    ya = np.abs(_bmul(plan, Lq, xe, transpose=True))             # y = L^T x, what the forward substitution produced
    per_row = np.bincount(plan["brow"], minlength=plan["n"]).max()
    per_col = np.diff(cptr).max()
    s = d * int(max(per_row, per_col)) + d + 1
    f_env = gamma(s) * (np.abs(be) + _bmul(plan, La, ya, strict=True)) + \
        2 * gamma(d) * np.einsum("kab,kbc,kcd,kd->ka", Pa, Lia, Pa, ya)
    g_env = gamma(s) * (ya + _bmul(plan, La, xa, transpose=True, strict=True)) + \
        2 * gamma(d) * np.einsum("kba,kcb,kdc,kd->ka", Pa, Lia, Pa, xa)
    env = f_env + _bmul(plan, La, g_env) + _bmul(plan, fenv, xa) + _bmul(plan, fenv, xa, transpose=True, strict=True)
    env += 4 * s * ETA
    return _ratio(r, 2 * env)             # 2: y above is L^T x, not the device's y (equal to first order)


def selinv_lists_py(plan):
    """For every sub-diagonal block t = (i, j) the operands of its recurrence: (t, Sigma block of (i, k), transposed,
    L block of (k, j)) for k in S(j), in column order -- the lists of direct_host.cpp selinv_lists."""
    cptr, brow = plan["cptr"], plan["brow"]
    tgt, sblk, tr, lblk = [], [], [], []
    for j in range(plan["n"]):
        a0, a1 = cptr[j] + 1, cptr[j + 1]
        for a in range(a0, a1):
            i = brow[a]
            for b in range(a0, a1):
                k = brow[b]
                lo, hi = min(i, k), max(i, k)
                s = cptr[lo] if lo == hi else cptr[lo] + 1 + int(np.searchsorted(brow[cptr[lo] + 1:cptr[lo + 1]], hi))
                assert brow[s] == hi
                tgt.append(a), sblk.append(s), tr.append(i < k), lblk.append(b)
    return [np.asarray(v, dtype=np.int64 if k != 2 else bool) for k, v in enumerate((tgt, sblk, tr, lblk))]


def selinv_gate(plan, L, Linv, Sig, lists=None):
    """Worst residual / envelope of the Takahashi recurrences on every block of the pattern of L:
         Sigma_ij + (sum_k Sigma_ik L_kj) Linv_j                     (i in S(j))
         Sigma_jj - Linv_j^T (Linv_j - sum_k L_kj^T Sigma_kj)
    with the device's L, Linv and Sigma (Sigma laid out like L)."""
    d = L.shape[1]
    cptr, brow, bcol = plan["cptr"], plan["brow"], plan["bcol"]
    tgt, sblk, tr, lblk = selinv_lists_py(plan) if lists is None else lists
    Lq, Sq, Iq = L.astype(LD), Sig.astype(LD), Linv.astype(LD)
    So = Sq[sblk]
    So[tr] = _t(So[tr])
    nL = len(brow)
    ptr = np.zeros(nL + 1, np.int64)
    np.add.at(ptr, tgt + 1, 1)
    ptr = np.cumsum(ptr)
    acc = _segsum(So @ Lq[lblk], ptr)
    acc_a = _segsum(np.abs(So) @ np.abs(Lq[lblk]), ptr)
    ns = np.diff(cptr) - 1
    g = gamma(ns[bcol] * d + d + 1)[:, None, None]
    off = brow != bcol
    R_off = Sq[off] + acc[off] @ Iq[bcol[off]]
    e_off = g[off] * (acc_a[off] @ np.abs(Iq[bcol[off]])) + ((ns[bcol[off]] + 2) * d * ETA)[:, None, None]
    piv = cptr[:-1]
    W = Iq.copy()
    Wa = np.abs(Iq)
    sub = np.flatnonzero(off)
    np.add.at(W, bcol[sub], -(_t(Lq[sub]) @ Sq[sub]))
    np.add.at(Wa, bcol[sub], np.abs(_t(Lq[sub])) @ np.abs(Sq[sub]))
    R_d = Sq[piv] - _t(Iq) @ W
    e_d = g[piv] * (_t(np.abs(Iq)) @ Wa) + ((ns + 2) * d * ETA)[:, None, None]
    e_d = np.maximum(e_d, _t(e_d))      # one triangle computed, mirrored
    return max(_ratio(R_off, e_off), _ratio(R_d, e_d))


def dense_inverse_check(plan, A, Sig):
    """|Sigma - A^-1| on the pattern against kappa(A) u |A^-1| (small cases): the worst ratio (<= 1 passes)."""
    d = A.shape[1]
    M = dense_of(plan, A.astype(float))
    Ainv = np.linalg.inv(M)
    kappa = np.linalg.cond(M)
    worst = 0.0
    scale = np.abs(Ainv).max()
    for t, (i, j) in enumerate(zip(plan["brow"], plan["bcol"])):
        err = np.abs(Sig[t] - Ainv[i * d:i * d + d, j * d:j * d + d]).max()
        worst = max(worst, err / (64 * len(M) * kappa * U * scale))
    return worst


# ---- an honest fp64 evaluation in another order, with plantable faults --------------------------------------------
def _chol_inplace(G, upper_reads=False):
    """dk_pivot_one's Cholesky; upper_reads: the running sums read the (stale) upper half instead of the factor."""
    d = G.shape[0]
    A = G.copy()
    for j in range(d):
        djj = A[j, j] - sum((A[m, j] * A[m, j] if upper_reads else A[j, m] * A[j, m]) for m in range(j))
        ljj = np.sqrt(djj)
        A[j, j] = ljj
        for r in range(j + 1, d):
            v = A[r, j] - sum((A[m, r] * A[m, j] if upper_reads else A[r, m] * A[j, m]) for m in range(j))
            A[r, j] = v / ljj
    return np.tril(A)


def host_factor(plan, A, fault=None, at=None):
    """Factor of the scattered blocks A in fp64: gathers summed before the subtraction, LAPACK Cholesky, triangular
    inverse by scipy, sub-diagonal blocks times Linv^T -- another order than direct.cu's.  Faults: "drop" skips update
    entry `at`; "pivot_upper" factors column `at` with the running sums read from the upper half; "scale_untransposed"
    scales row 0 of block `at` by Linv instead of Linv^T."""
    d = A.shape[1]
    cptr, brow, bcol, lp = plan["cptr"], plan["brow"], plan["bcol"], plan["lev_ptr"]
    ptr, ua, ub = plan["upd_ptr"], plan["upd_a"], plan["upd_b"]
    L = A.astype(float)
    Linv = np.zeros((plan["n"], d, d))
    for lev in range(plan["rounds"]):
        t0, t1 = cptr[lp[lev]], cptr[lp[lev + 1]]
        for t in range(t0, t1):
            qs = [q for q in range(ptr[t], ptr[t + 1]) if not (fault == "drop" and q == at)]
            if qs:
                L[t] = L[t] - np.sum(L[ua[qs]] @ _t(L[ub[qs]]), axis=0)
        for k in range(lp[lev], lp[lev + 1]):
            p = cptr[k]
            L[p] = _chol_inplace(L[p], True) if (fault == "pivot_upper" and k == at) else np.linalg.cholesky(L[p])
            Linv[k] = sla.solve_triangular(L[p], np.eye(d), lower=True)
        for t in range(t0, t1):
            if brow[t] != bcol[t]:
                G = L[t].copy()
                L[t] = G @ Linv[bcol[t]].T
                if fault == "scale_untransposed" and t == at:
                    L[t][0] = G[0] @ Linv[bcol[t]]
    return L, Linv


def host_solve(plan, L, b):
    """x from the block factor by two dense triangular solves (scipy), Hessian order."""
    d = L.shape[1]
    n, perm = plan["n"], plan["perm"]
    M = np.zeros((n * d, n * d))
    for t, (i, j) in enumerate(zip(plan["brow"], plan["bcol"])):
        M[i * d:i * d + d, j * d:j * d + d] = L[t]
    be = b.reshape(n, d)[perm].reshape(-1)
    y = sla.solve_triangular(M, be, lower=True)
    xe = sla.solve_triangular(M.T, y, lower=False).reshape(n, d)
    x = np.zeros((n, d))
    x[perm] = xe
    return x


def host_selinv(plan, L, Linv, fault_at=None):
    """Sigma on the pattern of L in fp64 by the recurrences, operands summed in reverse; fault_at: the index in the
    operand lists of one transposed operand read untransposed."""
    d = L.shape[1]
    cptr, brow, lp = plan["cptr"], plan["brow"], plan["lev_ptr"]
    tgt, sblk, tr, lblk = selinv_lists_py(plan)
    first = np.searchsorted(tgt, np.arange(len(brow)))
    last = np.searchsorted(tgt, np.arange(len(brow)), side="right")
    Sig = np.zeros(L.shape)
    for lev in range(plan["rounds"] - 1, -1, -1):
        cols = range(lp[lev], lp[lev + 1])
        for j in cols:
            for t in range(cptr[j] + 1, cptr[j + 1]):
                acc = np.zeros((d, d))
                for q in range(last[t] - 1, first[t] - 1, -1):
                    S = Sig[sblk[q]]
                    acc += (S.T if (tr[q] and q != fault_at) else S) @ L[lblk[q]]
                Sig[t] = -acc @ Linv[j]
        for j in cols:
            W = Linv[j] - sum((L[t].T @ Sig[t] for t in range(cptr[j] + 1, cptr[j + 1])), np.zeros((d, d)))
            D = Linv[j].T @ W
            Sig[cptr[j]] = np.tril(D) + np.tril(D, -1).T
    return Sig


# ---- tests -------------------------------------------------------------------------------------------------------------
def test_schedule_twin_on_the_suite_fixtures(kitti_k118):
    """The twin on KITTI K118 at 148 SMs: the Sim3 factor runs its 11 wide rounds on 21 CTAs and 15 on CTA 0, all one
    warp per column; its scale-trans twin (d = 4) takes the many-column branch on the grid and on CTA 0; d = 1 stays in
    one CTA.  The hand-built patterns of the GPU tests reach the regimes they are built for, for every d they run."""
    g = kitti_k118
    plan = plan_of(len(g["est"]), g["v0"], g["v1"], np.asarray(g["fixed"], np.uint8))
    s7 = schedule_twin(plan, 7, 148)
    assert (s7["grid"], s7["wide"], s7["rounds"]) == (21, 11, 26) and REGIMES["grid_tail_warp"](s7)
    s4 = schedule_twin(plan, 4, 148)
    assert s4["grid"] == 7 and any(s4["many"][:s4["wide"]]) and any(s4["many"][s4["wide"]:])
    s1 = schedule_twin(plan, 1, 148)
    assert s1["grid"] == 0 and sum(s1["many"]) == 4
    for d in (7, 6, 4, 1):
        assert REGIMES["single"](schedule_twin(plan_of(*chain(24)), d, 148))
        assert REGIMES["single_many"](schedule_twin(plan_of(*pairs(40)), d, 148))
        assert REGIMES["grid_many"](schedule_twin(plan_of(*chain(20000)), d, 148))
        assert REGIMES["all_wide"](schedule_twin(plan_of(*pairs(6000)), d, 148))
        assert REGIMES["diagonal"](schedule_twin(plan_of(*diagonal(6000)), d, 148))
    # the many-column branch of a level flips exactly at 2 * warps columns
    s = schedule_twin(plan_of(*pairs(32)), 7, 148)
    assert s["cols"][0] == 32 and not s["many"][0]
    s = schedule_twin(plan_of(*pairs(33)), 7, 148)
    assert s["cols"][0] == 33 and s["many"][0]


CASES = [("chain24", chain(24), 7), ("chain24", chain(24), 6), ("chain24", chain(24), 4), ("chain24", chain(24), 1),
         ("pairs40", pairs(40), 7), ("pairs40", pairs(40), 4)]


@pytest.mark.parametrize("name,graph,d", CASES, ids=[f"{c[0]}-d{c[2]}" for c in CASES])
def test_gates_accept_an_honest_evaluation(name, graph, d):
    plan = plan_of(*graph)
    Hb = spd_values(bsr_blocks(*graph), plan["n"], d, seed=d)
    lam = 0.37
    A = scatter(plan, Hb, lam)
    L, Linv = host_factor(plan, A)
    rf, ri, fenv = factor_gate(plan, A, L, Linv)
    b = np.random.default_rng(1).standard_normal((plan["n"], d))
    x = host_solve(plan, L, b)
    rs = solve_gate(plan, A, L, Linv, fenv, x, b)
    A0 = scatter(plan, Hb, 0.0)
    L0, Linv0 = host_factor(plan, A0)
    Sig = host_selinv(plan, L0, Linv0)
    rz = selinv_gate(plan, L0, Linv0, Sig)
    rd = dense_inverse_check(plan, A0, Sig)
    print(f"{name} d={d}: factor {rf:.2e} inverse {ri:.2e} solve {rs:.2e} selinv {rz:.2e} dense {rd:.2e}")
    assert max(rf, ri, rs, rz, rd) <= 1.0


def test_gates_accept_kitti_k1(kitti_k1):
    g = kitti_k1
    fixed = np.asarray(g["fixed"], np.uint8)
    nv = len(g["est"])
    hidx = -np.ones(nv, int)
    hidx[fixed == 0] = np.arange(int((fixed == 0).sum()))
    plan = plan_of(nv, g["v0"], g["v1"], fixed)
    Hb = spd_values(bsr_blocks(nv, g["v0"], g["v1"], hidx), plan["n"], 7, seed=3)
    A = scatter(plan, Hb, 0.0)
    L, Linv = host_factor(plan, A)
    rf, ri, fenv = factor_gate(plan, A, L, Linv)
    b = np.random.default_rng(2).standard_normal((plan["n"], 7))
    rs = solve_gate(plan, A, L, Linv, fenv, host_solve(plan, L, b), b)
    rz = selinv_gate(plan, L, Linv, host_selinv(plan, L, Linv))
    print(f"kitti_k1 d=7 (fill-in {len(plan['brow']) - len(Hb)} blocks): factor {rf:.2e} inverse {ri:.2e} "
          f"solve {rs:.2e} selinv {rz:.2e}")
    assert max(rf, ri, rs, rz) <= 1.0


def _planted(plan, Hb, lam, fault):
    """(factor gate margin, solve gate margin) of one planted fault on a pattern with fill-in."""
    A = scatter(plan, Hb, lam)
    cptr, brow, bcol = plan["cptr"], plan["brow"], plan["bcol"]
    src = plan["src"]
    sub = np.flatnonzero((brow != bcol) & (src >= 0))
    d = Hb.shape[1]
    Aused = A.copy()
    kw = {}
    if fault == "transposed_block":
        Aused[sub[0]] = _t(A[sub[0]])
    elif fault == "lambda_offdiag":
        Aused[sub[0]] += LD(lam) * np.eye(d, dtype=LD)
    elif fault == "drop":
        q = plan["upd_ptr"][cptr[plan["lev_ptr"][1]]]      # the first update of round 1: an operand of round 0
        assert q < plan["upd_ptr"][cptr[plan["lev_ptr"][2]]]
        kw = dict(fault="drop", at=int(q))
    elif fault == "pivot_upper":
        kw = dict(fault="pivot_upper", at=int(plan["lev_ptr"][1]))           # first column of round 1
    elif fault == "scale_untransposed":
        kw = dict(fault="scale_untransposed", at=int(sub[len(sub) // 2]))
    L, Linv = host_factor(plan, Aused, **kw)
    rf, ri, fenv = factor_gate(plan, A, L, Linv)
    b = np.random.default_rng(5).standard_normal((plan["n"], d))
    rs = solve_gate(plan, A, L, Linv, fenv, host_solve(plan, L, b), b)
    return max(rf, ri), rs


FAULTS = ["transposed_block", "drop", "lambda_offdiag", "pivot_upper", "scale_untransposed"]


@pytest.mark.parametrize("d", [7, 4])
def test_factor_and_solve_gates_reject_planted_faults(kitti_k1, d):
    g = kitti_k1
    fixed = np.asarray(g["fixed"], np.uint8)
    nv = len(g["est"])
    hidx = -np.ones(nv, int)
    hidx[fixed == 0] = np.arange(int((fixed == 0).sum()))
    plan = plan_of(nv, g["v0"], g["v1"], fixed)
    Hb = spd_values(bsr_blocks(nv, g["v0"], g["v1"], hidx), plan["n"], d, seed=4)
    for fault in FAULTS:
        mf, ms = _planted(plan, Hb, 0.37, fault)
        print(f"d={d} {fault}: factor gate margin {mf:.2e}, solve gate margin {ms:.2e}")
        assert mf >= 100 and ms >= 100, fault


@pytest.mark.parametrize("d", [7, 4])
def test_selinv_gate_rejects_an_untransposed_operand(kitti_k1, d):
    g = kitti_k1
    fixed = np.asarray(g["fixed"], np.uint8)
    nv = len(g["est"])
    hidx = -np.ones(nv, int)
    hidx[fixed == 0] = np.arange(int((fixed == 0).sum()))
    plan = plan_of(nv, g["v0"], g["v1"], fixed)
    Hb = spd_values(bsr_blocks(nv, g["v0"], g["v1"], hidx), plan["n"], d, seed=6)
    L, Linv = host_factor(plan, scatter(plan, Hb, 0.0))
    lists = selinv_lists_py(plan)
    q = int(np.flatnonzero(lists[2])[0])              # the first operand stored transposed
    Sig = host_selinv(plan, L, Linv, fault_at=q)
    m = selinv_gate(plan, L, Linv, Sig, lists)
    print(f"d={d} untransposed Takahashi operand: selinv gate margin {m:.2e}")
    assert m >= 100


def test_gamma_and_ratio():
    assert gamma(1) == pytest.approx(U) and gamma(0) == 0
    assert _ratio(np.array([0.0, 1.0]), np.array([0.0, 2.0])) == 0.5
    assert _ratio(np.array([1e-300]), np.array([0.0])) == np.inf
