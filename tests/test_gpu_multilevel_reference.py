"""The multilevel preconditioner (csrc/amg.cu) piece by piece against the long double host reference of
tests/test_multilevel_reference.py, in every cycle regime the code can take.

Each case builds a graph, sets the regime switches before the problem exists, and at two dampings checks, one level at
a time against the device's own previous level: the transfer frames, the Galerkin operators (pattern, values, exact
mirror blocks), the reuse path of an LM retry, the smoother inverses, the coarsest inverse, and one application
z = M^-1 r.  The regime the device reports must equal the one the host twin (ml_plan) predicts, so a case that stops
reaching its regime fails instead of passing on another path.
"""
import numpy as np
import pytest

from conftest import make_gpu
from test_multilevel_reference import (FRAME_TOL, KCYCLE_TOL, LD, U, Hierarchy, bound_ratio, bsr_blocks, chains,
                                       dense_of, frame_error, frames_ref, full_pattern_from_upper, galerkin_error,
                                       galerkin_ref, inverse_error, inverse_residual, kcycle_error, make_level,
                                       mass_ref, ml_plan, prolongation, regime, vcycle_error)

pytestmark = pytest.mark.gpu

PLAN_KEYS = ("n_levels", "kdepth", "kmask", "coop_first", "lt", "dense", "dense_coop", "coop_grid", "grid", "n", "G")


@pytest.fixture(scope="module")
def sphere_big():
    """sphere(30, 1000) at a late linearisation point (as tests/test_gpu_multilevel.py warms it)."""
    import sim3opt_b200 as s3
    from sim3opt_b200 import synth
    g = dict(synth.sphere(n_laps=30, poses_per_lap=1000, seed=7))
    warm = make_gpu(g, jac=1, math_mode=s3.MATH_CORRECTED)
    warm.set_pcg(0.1, 20000)
    warm.optimize(4)
    g["est"] = warm.vertices()
    return g


@pytest.fixture(scope="module")
def chains_large():
    return chains(300, 80)


def case_graph(name, request):
    import sim3opt_b200 as s3
    from oracle import kitti_io
    from sim3opt_b200 import synth
    if name == "kitti_k1_sim3":
        return request.getfixturevalue("kitti_k1"), s3.KIND_SIM3
    if name == "kitti_k1_scale_trans":
        return kitti_io.to_scale_trans_graph(request.getfixturevalue("kitti_k1")), s3.KIND_SCALE_TRANS
    if name == "kitti_k118_scale":
        g = request.getfixturevalue("kitti_k118")
        return dict(est=g["est"][:, 7:8], fixed=g["fixed"], v0=g["v0"], v1=g["v1"], meas=g["meas"][:, 7:8]), s3.KIND_SCALE
    if name == "sphere_10x300":
        return synth.sphere(10, 300, seed=11), s3.KIND_SIM3
    if name == "sphere_2x6":
        return synth.sphere(2, 6, seed=1), s3.KIND_SIM3
    if name.startswith("sphere_30x1000"):
        return request.getfixturevalue("sphere_big"), s3.KIND_SIM3
    if name == "chains_300x80":
        return request.getfixturevalue("chains_large"), s3.KIND_SIM3
    a, b = name.split("_")[1].split("x")
    return chains(int(a), int(b)), s3.KIND_SIM3


# name, switches, what the regime must be (beyond agreeing with the twin), whether the operators are checked
# (the switches change the cycle, not the operators: the variants of one graph check the application only)
CASES = [
    ("kitti_k1_sim3", {}, dict(kdepth=0, dense=1, dense_coop=0), True),
    ("kitti_k1_scale_trans", {}, dict(kdepth=0, dense=1, dense_coop=0), True),
    ("kitti_k118_scale", {}, dict(kdepth=0, dense=1, dense_coop=0), True),
    ("sphere_10x300", {"S3O_KCYCLE": "2"}, dict(kdepth=2, kmask=3, coop_first=0, dense=1, dense_coop=0), True),
    ("chains_40x50", {}, dict(kdepth=0, lt=0, dense=1, dense_coop=1), True),
    ("chains_200x50", {}, dict(kdepth=0, lt=2, dense=0), True),
    ("sphere_30x1000", {}, dict(kdepth=2, kmask=2, coop_first=0, dense=1, dense_coop=1), True),
    ("sphere_30x1000_v", {"S3O_KCYCLE": "0"}, dict(kdepth=0, lt=1, dense=1, dense_coop=1), False),
    ("sphere_30x1000_khost", {"S3O_KMASK": "3", "S3O_COOP_ROWS": "1000"}, dict(kdepth=2, kmask=3, coop_first=1), False),
    ("chains_300x80", {}, dict(kdepth=3, kmask=6, coop_first=0, dense=0), True),
    ("sphere_2x6", {}, dict(n_levels=0), True),
]


def fine_minv(gpu, lam, nf, d):
    """The fine level's block-Jacobi inverses, read through s3o_apply_preconditioner with block-Jacobi configured:
    probe c puts 1 in component c of every vertex, so z holds column c of every block (each an exact product)."""
    import sim3opt_b200 as s3
    gpu.set_preconditioner(s3.PRECOND_BLOCK_JACOBI)
    try:
        Minv = np.zeros((nf, d, d))
        for c in range(d):
            r = np.zeros((nf, d))
            r[:, c] = 1.0
            Minv[:, :, c] = gpu.apply_preconditioner(lam, r).reshape(nf, d)
    finally:
        gpu.set_preconditioner(s3.PRECOND_MULTILEVEL)
    return Minv


def diag_positions(rowptr, colidx):
    rows = np.repeat(np.arange(len(rowptr) - 1), np.diff(rowptr))
    pos = np.flatnonzero(rows == np.asarray(colidx))
    assert np.array_equal(rows[pos], np.arange(len(rowptr) - 1)), "a coarse row without its diagonal block"
    return pos


def check_operators(gpu, d, plan, levels, inv, Minv, lam, H, colptr, rowidx, est, aux, free2v, agg0):
    """Frames, Galerkin operators, smoother inverses and the coarsest inverse of one prepared set-up."""
    nl = plan["n_levels"]
    worst = {}
    for k in range(nl):
        L = levels[k]
        n = len(L["root_vid"])
        vid = free2v if k == 0 else levels[k - 1]["root_vid"]
        rvid = L["root_vid"][L["agg"]]
        # the root of every aggregate is one of its members, and it moves with itself
        assert np.array_equal(np.bincount(L["agg"][vid == rvid], minlength=n), np.ones(n, int)), k
        if k == 0:
            assert np.array_equal(L["agg"], agg0)
        fe = frame_error(L["rel"], frames_ref(d, est, aux, vid, rvid), est, vid, rvid, d)
        assert fe <= FRAME_TOL, (k, fe)
        # Galerkin: pattern = aggregate pairs with a fine block, ascending columns, diagonal present; values in the
        # rounding envelope of P^T A_k P with P from the (checked) device frames and A_k the device's previous level
        if k == 0:
            rows, cols, B = full_pattern_from_upper(colptr, rowidx, H, lam)
        else:
            F = levels[k - 1]
            rows, cols, B = bsr_blocks(F["rowptr"], F["colidx"], F["A"])
        ref = galerkin_ref(rows, cols, B, L["agg"], prolongation(L["rel"], d), n)
        keys = np.repeat(np.arange(n), np.diff(L["rowptr"])) * n + L["colidx"]
        assert np.array_equal(keys, ref[0]), f"level {k}: coarse pattern differs"
        ge = galerkin_error(L["A"], ref)
        assert ge <= 1.0, (k, ge)
        # an off-diagonal block is computed once and stored twice, so its mirror is its exact transpose; a diagonal
        # block sums non-symmetric rounded products and is symmetric to rounding only (within the gate above)
        odiag = keys // n != keys % n
        pos = np.searchsorted(keys, (keys % n) * n + keys // n)
        assert np.array_equal(L["A"][pos[odiag]], np.transpose(L["A"][odiag], (0, 2, 1))), \
            f"level {k}: mirror block not the transpose"
        # smoother inverses of the diagonal blocks
        dp = diag_positions(L["rowptr"], L["colidx"])
        ie = inverse_error(L["A"][dp], L["Dinv"])
        assert ie <= 1.0, (k, ie)
        worst[k] = (fe, ge, ie)
    # fine block-Jacobi inverses of H + lam I
    nf = len(colptr) - 1
    dcol = np.flatnonzero(np.asarray(rowidx) == np.repeat(np.arange(nf), np.diff(colptr)))
    fe0 = inverse_error(H[dcol] + lam * np.eye(d), Minv)
    assert fe0 <= 1.0, fe0
    if inv is not None:
        C = levels[-1]
        Ac = dense_of(C["rowptr"], C["colidx"], C["A"])
        N = Ac.shape[0]
        res, kap = inverse_residual(Ac, inv)
        assert res <= 10 * N * U * kap, (res, kap)
        asym = np.linalg.norm(inv - inv.T, 2)
        assert asym <= 10 * N * U * kap * np.linalg.norm(inv, 2), (asym, kap)
        worst["inv"] = (float(res / (N * U * kap)), float(kap))
    print(f"  lam {lam:.3e}: frame / Galerkin / smoother gate ratios per level {worst}, fine smoother {fe0:.2e}")


def check_reuse(d, lev1, lev2, lam1, lam2):
    """A second lambda at the same linearisation point: the off-diagonal blocks stay bit for bit, the diagonal blocks
    move by (lam2 - lam1) M with M = P^T M_prev P (M_0 = I)."""
    M = None
    dl = LD(lam2) - LD(lam1)
    for k, (a, b) in enumerate(zip(lev1, lev2)):
        n = len(a["root_vid"])
        P = prolongation(a["rel"], d)
        Menv = mass_ref(a["agg"], np.abs(P), None if M is None else np.abs(M), n)
        M = mass_ref(a["agg"], P, M, n)
        dp = diag_positions(a["rowptr"], a["colidx"])
        off = np.ones(len(a["A"]), bool)
        off[dp] = False
        assert np.array_equal(a["A"][off], b["A"][off]), f"level {k}: an off-diagonal block changed with lambda"
        diff = np.asarray(b["A"][dp], LD) - np.asarray(a["A"][dp], LD)
        nmax = int(np.bincount(a["agg"]).max()) * d * d * (k + 1)
        bound = 4 * U * (np.abs(a["A"][dp]) + np.abs(b["A"][dp])) + abs(dl) * 4 * nmax * U * Menv
        r = bound_ratio(np.abs(diff - dl * M), bound)
        assert r <= 1.0, (k, r)


def check_application(gpu, plan, levels, inv, Minv, lam, d, rng):
    # the V-cycle's tail kernel reads the coarsest inverse by columns (x_t = sum_c inv[c, t] r_c), the cooperative
    # kernel by rows: the two differ by the inverse's rounding asymmetry, which is far above the cycle's own rounding
    applied = None if inv is None else (inv.T if plan["kdepth"] == 0 else inv)
    h = Hierarchy(Minv, [make_level(L["agg"], prolongation(L["rel"], d), L["rowptr"], L["colidx"], L["A"], L["Dinv"])
                         for L in levels], applied, plan)
    n = Minv.shape[0] * d
    r1, r2 = rng.standard_normal(n), rng.standard_normal(n)
    z1, z2 = gpu.apply_preconditioner(lam, r1), gpu.apply_preconditioner(lam, r2)
    assert np.array_equal(z1, gpu.apply_preconditioner(lam, r1)), "an application is not reproducible"
    assert r1 @ z1 > 0 and r2 @ z2 > 0
    v_cycle = plan["kdepth"] == 0 or plan["kmask"] == 0
    if not v_cycle:                 # K-cycle: nonlinear in r, so neither symmetric nor linear
        e1, e2 = kcycle_error(z1, h.apply(r1)), kcycle_error(z2, h.apply(r2))
        assert max(e1, e2) <= KCYCLE_TOL, (e1, e2)
        print(f"  lam {lam:.3e}: K-cycle application, relative 2-norm error {max(e1, e2):.2e}")
        return
    terms = h.terms()
    env1, env2 = h.apply(r1, envelope=True), h.apply(r2, envelope=True)
    zr1, zr2 = h.apply(r1), h.apply(r2)
    e1, e2 = vcycle_error(z1, zr1, env1, terms), vcycle_error(z2, zr2, env2, terms)
    assert max(e1, e2) <= 1.0, (e1, e2)
    # a fixed symmetric linear operator
    a, b = 0.75, -1.25
    z12 = gpu.apply_preconditioner(lam, a * r1 + b * r2)
    env12 = h.apply(a * r1 + b * r2, envelope=True)
    lin = bound_ratio(np.abs(np.asarray(z12, LD) - a * np.asarray(z1, LD) - b * np.asarray(z2, LD)),
                      terms * U * (env12 + abs(a) * env1 + abs(b) * env2) + 4 * U * np.abs(z12))
    # symmetric up to rounding and to what the coarsest inverse's own asymmetry contributes (taken from the reference)
    sym = float(abs(r1 @ z2 - r2 @ z1) / (abs(np.asarray(r1, LD) @ zr2 - np.asarray(r2, LD) @ zr1) + terms * U * (
        np.abs(r1) @ env2 + np.abs(r2) @ env1) + 4 * n * U * (np.abs(r1) @ np.abs(z2) + np.abs(r2) @ np.abs(z1))))
    assert lin <= 1.0 and sym <= 1.0, (lin, sym)
    print(f"  lam {lam:.3e}: V-cycle application gate {max(e1, e2):.2e}, linearity {lin:.2e}, symmetry {sym:.2e} "
          f"(constant {terms})")


@pytest.mark.parametrize("name,switches,expect,operators", CASES, ids=[c[0] for c in CASES])
def test_preconditioner_against_host_reference(name, switches, expect, operators, request, monkeypatch):
    import torch
    import sim3opt_b200 as s3
    for k in ("S3O_KCYCLE", "S3O_KMASK", "S3O_COOP_ROWS"):
        monkeypatch.delenv(k, raising=False)
    for k, v in switches.items():
        monkeypatch.setenv(k, v)
    g, kind = case_graph(name, request)
    gpu = make_gpu(g, kind=kind, jac=1, math_mode=s3.MATH_CORRECTED)
    gpu.set_preconditioner(s3.PRECOND_MULTILEVEL)
    gpu.set_pcg(1e-10, 5000)
    colptr, rowidx = gpu.build_structure()
    H, _ = gpu.linearize()
    d, nf = gpu.d, gpu.num_free
    hidx = gpu.hessian_index()
    free2v = np.zeros(nf, np.int64)
    free2v[hidx[hidx >= 0]] = np.flatnonzero(hidx >= 0)
    est, aux = gpu.vertices(), g.get("aux")
    sizes, _, agg0 = s3.host_multilevel(len(g["est"]), g["fixed"], g["v0"], g["v1"])
    twin = ml_plan(sizes, nf, torch.cuda.get_device_properties(0).multi_processor_count, switches)
    md = gpu.max_diag()
    lams = (1e-4 * md, 1e-9 * md)
    before = gpu.solve(lams[1])
    rng = np.random.default_rng(17)
    prev = None
    print(f"\n{name} {switches}: {regime(twin)}")
    for lam in lams:
        plan = gpu.multilevel_prepare(lam)
        assert {k: plan[k] for k in PLAN_KEYS} == {k: twin[k] for k in PLAN_KEYS}, (plan, twin)
        assert {k: plan[k] for k in expect} == expect, plan
        nl = plan["n_levels"]
        Minv = fine_minv(gpu, lam, nf, d)
        gpu.multilevel_prepare(lam)
        levels = [gpu.multilevel_level(k) for k in range(nl)]
        inv = gpu.multilevel_coarsest_inverse() if nl and plan["dense"] else None
        if operators:
            check_operators(gpu, d, plan, levels, inv, Minv, lam, H, colptr, rowidx, est, aux, free2v, agg0)
            if prev is not None:
                check_reuse(d, prev[1], levels, prev[0], lam)
        check_application(gpu, plan, levels, inv, Minv, lam, d, rng)
        prev = (lam, levels)
    # the hooks leave nothing behind that a solve would see
    after = gpu.solve(lams[1])
    assert before[0] == after[0] == 0 and before[2] == after[2] and np.array_equal(before[1], after[1])
    assert np.array_equal(gpu.vertices(), est)


def test_hook_errors():
    import ctypes
    import sim3opt_b200 as s3
    from sim3opt_b200 import synth
    g = synth.sphere(4, 60, seed=2)
    p = make_gpu(g)
    p.set_preconditioner(s3.PRECOND_MULTILEVEL)
    p.build_structure()
    info = np.zeros(45, np.int32)
    ip = info.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))
    assert p.L.s3o_multilevel_prepare(p.h, 1.0, ip, 45) == -1                 # before s3o_linearize
    p.linearize_only()
    assert p.L.s3o_multilevel_prepare(p.h, 1.0, ip, 45) == 0 and info[0] >= 1
    assert p.L.s3o_get_multilevel_level(p.h, int(info[0]), None, None, None, None, None, None, None) == -1
    assert p.L.s3o_get_multilevel_level(p.h, -1, None, None, None, None, None, None, None) == -1
    assert p.L.s3o_multilevel_prepare(p.h, 1.0, ip, 9) == -1                  # info too short for the levels
    b = synth.ba_loop(8, 60, 4, seed=1)
    q = s3.BAProblem()
    q.set(b["cams"], b["points"], b["obs_cam"], b["obs_pt"], b["uv"], b["focal"], b["cx"], b["cy"])
    assert q.L.s3o_multilevel_prepare(q.h, 1.0, ip, 45) == -5
    assert q.L.s3o_apply_preconditioner(q.h, 1.0, None, None) == -5
