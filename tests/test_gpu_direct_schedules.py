"""GPU tests of the sparse block Cholesky (csrc/direct.cu) in every schedule it runs, against the long-double gates of
test_direct_reference.py.

direct_kernel and selinv_kernel put the leading wide rounds on a cooperative grid and the narrow tail on CTA 0, and
dk_pivot_scale switches between one thread per pivot (many columns) and one warp per column.  Each case below is a
pattern built for one of those regimes; it asserts that the device's schedule (s3o_direct_schedule) equals the host
twin's at the SM count the device reports, and that the twin puts it in that regime.  Then the factor, the solve and
the selected inverse are checked by the gates, with bitwise reproducibility, and solves on a held factor
(do_factor = 0: the off-pattern marginal columns) against factorising and solving again.
"""
import numpy as np
import pytest

import sim3opt_b200 as s3
from test_direct_reference import (REGIMES, bsr_blocks, ccs_of, chain, dense_inverse_check, diagonal, factor_gate,
                                   pairs, plan_of, scatter, schedule_twin, selinv_gate, solve_gate, spd_values)

pytestmark = pytest.mark.gpu

KEYS = ("n", "rounds", "blocks", "grid", "wide", "cols", "level_blocks")


def _confirm(name, d, plan, dev, regime):
    twin = schedule_twin(plan, d, dev["sms"])
    for k in KEYS:
        assert dev[k] == twin[k], (name, d, k, dev[k], twin[k])
    many = [lev for lev, m in enumerate(twin["many"]) if m]
    print(f"{name} d={d}: {dev['sms']} SMs, grid {dev['grid']}, wide {dev['wide']} / {dev['rounds']} rounds, "
          f"{dev['blocks']} blocks of L, many-column rounds {many}")
    if regime:
        assert REGIMES[regime](twin), (name, d, regime)
    return twin


# ---- the linear-solver plug-in on chosen patterns with random SPD values -------------------------------------------
LS_CASES = [
    ("chain24", lambda: chain(24), "single", (7, 6, 4, 1)),
    ("pairs40", lambda: pairs(40), "single_many", (7, 6, 4, 1)),
    ("chain20000", lambda: chain(20000), "grid_many", (7, 6, 4, 1)),
    ("pairs6000", lambda: pairs(6000), "all_wide", (7, 6, 4, 1)),
    ("diagonal6000", lambda: diagonal(6000), "diagonal", (7, 6, 4, 1)),
]
LS_PARAMS = [(name, make, regime, d) for name, make, regime, ds in LS_CASES for d in ds]


def _ls_case(name, graph, regime, d, seed=0):
    n, v0, v1 = graph
    plan = plan_of(n, v0, v1)
    blocks = bsr_blocks(n, v0, v1)
    Hb = spd_values(blocks, n, d, seed=seed + d)
    colptr, rowidx, Hc = ccs_of(blocks, Hb)
    lam = 0.37
    b = np.random.default_rng(seed).standard_normal(n * d)
    ls = s3.LinearSolver(d)
    ls.set_linear_solver(s3.LINSOLVER_DIRECT)
    rc, x, method, _ = ls.solve(colptr, rowidx, Hc, b, lam)
    assert rc == 0 and method == s3.LINSOLVER_DIRECT
    _confirm(name, d, plan, ls.direct_schedule(), regime)
    L, Linv = ls.direct_factor()
    A = scatter(plan, Hb, lam)
    rf, ri, fenv = factor_gate(plan, A, L, Linv)
    rs = solve_gate(plan, A, L, Linv, fenv, x, b)
    print(f"    gates: factor {rf:.2e} inverse {ri:.2e} solve {rs:.2e}")
    assert rf <= 1 and ri <= 1 and rs <= 1
    rc, x2, _, _ = ls.solve(colptr, rowidx, Hc, b, lam)
    L2, Linv2 = ls.direct_factor()
    assert rc == 0 and np.array_equal(x, x2) and np.array_equal(L, L2) and np.array_equal(Linv, Linv2)
    return ls, plan, blocks, Hb, (colptr, rowidx, Hc), b, x


@pytest.mark.parametrize("name,make,regime,d", LS_PARAMS, ids=[f"{p[0]}-d{p[3]}" for p in LS_PARAMS])
def test_linsolver_schedules(name, make, regime, d):
    _ls_case(name, make(), regime, d)


@pytest.mark.parametrize("d", [7, 6, 4, 1])
def test_linsolver_kitti_k118_pattern(kitti_k118, d):
    """K118's Hessian pattern: for d = 7 a grid with a tail and one warp per column in every round."""
    g = kitti_k118
    fixed = np.asarray(g["fixed"], np.uint8)
    nv = len(g["est"])
    free = np.flatnonzero(fixed == 0)
    hidx = -np.ones(nv, np.int64)
    hidx[free] = np.arange(len(free))
    keep = (hidx[g["v0"]] >= 0) & (hidx[g["v1"]] >= 0)
    graph = (len(free), hidx[g["v0"][keep]].astype(np.int32), hidx[g["v1"][keep]].astype(np.int32))
    _ls_case("kitti_k118", graph, "grid_tail_warp" if d == 7 else None, d)


@pytest.mark.parametrize("name,make,d", [("chain24", lambda: chain(24), 7), ("pairs40", lambda: pairs(40), 4),
                                          ("chain20000", lambda: chain(20000), 7), ("chain20000", lambda: chain(20000), 1),
                                          ("pairs6000", lambda: pairs(6000), 6)],
                         ids=["chain24-d7", "pairs40-d4", "chain20000-d7", "chain20000-d1", "pairs6000-d6"])
def test_pivot_failure_is_reported_and_reset(name, make, d):
    """An indefinite diagonal block in a chosen round -- a wide one and a tail one on a grid, the first and the last in
    one CTA -- makes the solve return S3O_ERR_SOLVE; the next SPD solve on the same pattern is clean and bitwise equal to
    the one before the failure."""
    ls, plan, blocks, Hb, (colptr, rowidx, Hc), b, x = _ls_case(name, make(), None, d)
    sched = ls.direct_schedule()
    lp, perm = plan["lev_ptr"], plan["perm"]
    if sched["grid"] > 1:
        rounds = [0, sched["wide"] - 1] + ([sched["wide"], sched["rounds"] - 1] if sched["wide"] < sched["rounds"] else [])
    else:
        rounds = [0, sched["rounds"] - 1]
    diag_of = {r: k for k, (r, c) in enumerate(blocks) if r == c}
    for lev in rounds:
        col = int(lp[lev] + (lp[lev + 1] - lp[lev]) // 2)              # a column in the middle of the round
        Hbad = Hb.copy()
        Hbad[diag_of[int(perm[col])]] *= -1.0
        rc, _, _, _ = ls.solve(colptr, rowidx, ccs_of(blocks, Hbad)[2], b, 0.37)
        where = "grid" if lev < sched["wide"] else "CTA 0"
        print(f"{name} d={d}: indefinite pivot in round {lev} ({where}): rc {rc}")
        assert rc == -6
        rc, x2, _, _ = ls.solve(colptr, rowidx, Hc, b, 0.37)
        assert rc == 0 and np.all(np.isfinite(x2)) and np.array_equal(x, x2)


# ---- pose-graph problems: the selected inverse and solves on the held factor ----------------------------------------
def _pose_graph(kind, n_free, edges, seed):
    """Vertex 0 fixed, vertices 1..n_free free; edges among the free vertices (0-based free ids) plus one edge from the
    fixed vertex into every connected component; measurements from random poses with noise."""
    from oracle import kitti_io
    from sim3opt_b200 import synth
    rng = np.random.default_rng(seed)
    nv = n_free + 1
    v0, v1 = (np.asarray(e, np.int64) + 1 for e in edges)
    parent = np.arange(n_free)

    def root(a):
        while parent[a] != a:
            parent[a] = parent[parent[a]]
            a = parent[a]
        return a
    for a, c in zip(v0 - 1, v1 - 1):
        ra, rc = root(a), root(c)
        if ra != rc:
            parent[max(ra, rc)] = min(ra, rc)
    anchors = np.unique([root(a) for a in range(n_free)]) + 1
    v0 = np.r_[np.zeros(len(anchors), np.int64), v0].astype(np.int32)
    v1 = np.r_[anchors, v1].astype(np.int32)
    R, t, s = synth.sim3_exp(rng.standard_normal((nv, 7)) * np.array([0.3] * 3 + [2.0] * 3 + [0.2]))
    Ri, ti, si = R[v0], t[v0], s[v0]
    Rn, tn, sn = synth.sim3_exp(rng.standard_normal((len(v0), 7)) * 0.01)
    Rm, tm, sm = synth._mul(Rn, tn, sn, *synth._mul(R[v1], t[v1], s[v1], *synth._inv(Ri, ti, si)))
    g = dict(est=synth._pack(R, t, s), fixed=np.r_[1, np.zeros(n_free)].astype(np.uint8), v0=v0, v1=v1,
             meas=synth._pack(Rm, tm, sm))
    if kind == s3.KIND_SCALE_TRANS:
        g = kitti_io.to_scale_trans_graph(g)
    elif kind == s3.KIND_SCALE:
        g = dict(est=g["est"][:, 7:8], fixed=g["fixed"], v0=v0, v1=v1, meas=g["meas"][:, 7:8])
    p = s3.Problem(kind)
    p.set_vertices(g["est"], g["fixed"], g.get("aux"))
    p.set_edges(g["v0"], g["v1"], g["meas"])
    p.set_jacobian_mode(s3.JAC_ANALYTIC)
    return p, g


PG_CASES = [("chain24", lambda: chain(24)[1:], 24, "single"), ("pairs40", lambda: pairs(40)[1:], 80, "single_many"),
            ("chain20000", lambda: chain(20000)[1:], 20000, "grid_many"),
            ("pairs6000", lambda: pairs(6000)[1:], 12000, "all_wide")]
KINDS = [(s3.KIND_SIM3, 7), (s3.KIND_SCALE_TRANS, 4), (s3.KIND_SCALE, 1)]
PG_PARAMS = [(c[0], c[1], c[2], c[3], k, d) for c in PG_CASES for k, d in KINDS]


@pytest.mark.parametrize("name,edges,n_free,regime,kind,d", PG_PARAMS, ids=[f"{p[0]}-d{p[5]}" for p in PG_PARAMS])
def test_selected_inverse_and_held_factor(name, edges, n_free, regime, kind, d):
    p, g = _pose_graph(kind, n_free, edges(), seed=n_free + d)
    colptr, rowidx = p.build_structure()
    plan = plan_of(len(g["est"]), g["v0"], g["v1"], g["fixed"])
    perm, brow, bcol = plan["perm"], plan["brow"], plan["bcol"]
    on = np.stack([perm[brow], perm[bcol]], 1)
    pattern = {(int(a), int(c)) for a, c in on} | {(int(c), int(a)) for a, c in on}
    rng = np.random.default_rng(d)
    off = []
    while len(off) < 3:
        a, c = (int(v) for v in rng.integers(0, plan["n"], 2))
        if (a, c) not in pattern:
            off.append((a, c))
    req = np.r_[on, np.array(off)]
    out = p.marginals(req)
    _confirm(f"{name} ({['Sim3', 'scale-trans', 'scale'][kind]})", d, plan, p.direct_schedule(), regime)
    L, Linv = p.direct_factor()
    Sig = out[:len(on)]
    out2 = p.marginals(req)
    assert np.array_equal(out, out2)
    H, _ = p.linearize()
    order = np.lexsort((np.repeat(np.arange(len(colptr) - 1), np.diff(colptr)), rowidx))      # CCS -> BSR order
    Hb = H[order]
    A = scatter(plan, Hb, 0.0)
    rf, ri, _ = factor_gate(plan, A, L, Linv)
    rz = selinv_gate(plan, L, Linv, Sig)
    msg = f"    gates: factor {rf:.2e} inverse {ri:.2e} selinv {rz:.2e}"
    if plan["n"] <= 100:
        rd = dense_inverse_check(plan, A, Sig)
        msg += f" dense inverse {rd:.2e}"
        assert rd <= 1
    print(msg)
    assert rf <= 1 and ri <= 1 and rz <= 1
    # off-pattern blocks: d solves on the held factor; the same right-hand sides factorised and solved again
    ls = s3.LinearSolver(d)
    ls.set_linear_solver(s3.LINSOLVER_DIRECT)
    for q, (r, c) in enumerate(off):
        for m in range(d):
            e = np.zeros(plan["n"] * d)
            e[c * d + m] = 1.0
            rc, x, method, _ = ls.solve(colptr, rowidx, H, e, 0.0)
            assert rc == 0 and method == s3.LINSOLVER_DIRECT
            assert np.array_equal(out[len(on) + q][:, m], x[r * d:r * d + d]), (r, c, m)
    dev = ls.direct_schedule()
    assert all(dev[k] == p.direct_schedule()[k] for k in KEYS)
