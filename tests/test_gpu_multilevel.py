"""Multilevel (aggregation) preconditioner of the pose-graph PCG -- GPU tests through the C ABI.

The preconditioner only changes how fast the PCG reaches the solution of (H + lambda I) x = b, never
the solution: the checks are the same backward-error / oracle gates as for block-Jacobi
(tests/test_gpu_parity.py), plus iteration counts and bitwise reproducibility.
"""
import numpy as np
import pytest

from conftest import make_gpu, make_oracle
from test_gpu_parity import dense_from_blocks
from test_gpu_spmv_shapes import backward_error

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sphere_mid():
    from sim3opt_b200 import synth
    return synth.sphere(n_laps=10, poses_per_lap=300, seed=11)


@pytest.fixture(params=["kitti_k1", "kitti_k118", "sphere_small", "sphere_mid", "manhattan_small"])
def graph(request):
    return request.getfixturevalue(request.param)


def test_solve_backward_error(graph):
    import sim3opt_b200 as s3
    gpu = make_gpu(graph, jac=1)
    colptr, rowidx = gpu.build_structure()
    H, b = gpu.linearize()
    lam = 1e-5 * gpu.max_diag()
    gpu.set_pcg(1e-11, 50000)
    gpu.set_preconditioner(s3.PRECOND_BLOCK_JACOBI)
    rc1, x1, it1, rel1 = gpu.solve(lam)
    gpu.set_preconditioner(s3.PRECOND_MULTILEVEL)
    rc2, x2, it2, rel2 = gpu.solve(lam)
    assert rc1 == 0 and rc2 == 0 and rel2 <= 1e-11
    A = dense_from_blocks(colptr, rowidx, H, 7) + lam * np.eye(len(b))
    assert np.linalg.norm(A @ x2 - b) <= 1e-10 * np.linalg.norm(b)
    assert it2 <= it1
    # reproducible to the bit: every sum runs in list order
    rc3, x3, it3, _ = gpu.solve(lam)
    assert it3 == it2 and np.array_equal(x2, x3)


def test_fewer_iterations_at_small_damping(sphere_mid):
    """The coarse-space correction pays when lambda is small (late LM iterations)."""
    import sim3opt_b200 as s3
    gpu = make_gpu(sphere_mid, jac=1, math_mode=s3.MATH_CORRECTED)
    gpu.linearize_only()
    lam = 1e-8 * gpu.max_diag()
    gpu.set_pcg(1e-8, 50000)
    gpu.set_preconditioner(s3.PRECOND_BLOCK_JACOBI)
    _, x1, it1, _ = gpu.solve(lam)
    gpu.set_preconditioner(s3.PRECOND_MULTILEVEL)
    _, x2, it2, _ = gpu.solve(lam)
    assert it2 * 3 <= it1, (it1, it2)
    assert np.abs(x1 - x2).max() <= 1e-3 * np.abs(x1).max()      # both stop at a 1e-8 residual; cond(H) bounds the error


def test_lm_matches_block_jacobi_and_oracle(sphere_small):
    """End-to-end LM with the multilevel PCG lands on the oracle's minimum (BASELINE tolerances)."""
    from oracle import oracle as orc
    import sim3opt_b200 as s3
    orc.set_math_mode(orc.MATH_CORRECTED)
    try:
        gpu = make_gpu(sphere_small, jac=1, math_mode=s3.MATH_CORRECTED)
        gpu.set_preconditioner(s3.PRECOND_MULTILEVEL)
        gpu.set_pcg(1e-10, 20000)
        cpu = make_oracle(sphere_small, jac=orc.JAC_ANALYTIC)
        n_g, chi_g, _, _ = gpu.optimize(40)
        n_c, chi_c, _, _ = cpu.optimize(40)
    finally:
        orc.set_math_mode(orc.MATH_REFERENCE)
    assert abs(chi_g - chi_c) <= 1e-4 * chi_c
    vg, vc = gpu.vertices(), cpu.vertices()
    assert np.abs(vg[:, 4:7] - vc[:, 4:7]).max() <= 1e-4
    dots = np.abs((vg[:, :4] * vc[:, :4]).sum(1) / (np.linalg.norm(vg[:, :4], axis=1) * np.linalg.norm(vc[:, :4], axis=1)))
    assert (2 * np.arccos(np.clip(dots, -1, 1))).max() <= 1e-5


def test_scale_trans_multilevel(kitti_k1, kitti_k118):
    """4-DoF scale+translation graph of the stepwise pipeline (kitti_surf.cpp:834-839,872-877): the
    coarse space is delta_i = (s_i/s_root) diag(1, R_i R_root^T) xi; same solution, far fewer iterations."""
    import sim3opt_b200 as s3
    from oracle import kitti_io
    for g in (kitti_k1, kitti_k118):
        st = kitti_io.to_scale_trans_graph(g)
        gpu = make_gpu(st, kind=s3.KIND_SCALE_TRANS, jac=1)
        colptr, rowidx = gpu.build_structure()
        H, b = gpu.linearize()
        lam = 1e-7 * gpu.max_diag()
        gpu.set_pcg(1e-11, 200000)
        gpu.set_preconditioner(s3.PRECOND_BLOCK_JACOBI)
        rc1, x1, it1, _ = gpu.solve(lam)
        gpu.set_preconditioner(s3.PRECOND_MULTILEVEL)
        rc2, x2, it2, rel2 = gpu.solve(lam)
        assert rc1 == 0 and rc2 == 0 and rel2 <= 1e-11
        A = dense_from_blocks(colptr, rowidx, H, 4) + lam * np.eye(len(b))
        assert np.linalg.norm(A @ x2 - b) <= 1e-10 * np.linalg.norm(b)
        assert it2 * 4 <= it1, (it1, it2)


def test_scale_null_vector_multilevel(kitti_k118):
    """1-DoF scale graph (kitti_surf.cpp:891-934): inverse iteration with the multilevel PCG finds the
    same null vector as numpy's dense SVD."""
    import sim3opt_b200 as s3
    g = kitti_k118
    n = len(g["est"])
    v0, v1, s = g["v0"], g["v1"], g["meas"][:, 7]
    A = np.zeros((len(v0), n))
    for r, (i, j, m) in enumerate(zip(v0, v1, s)):
        A[r, i] = m
        A[r, j] = -1.0
    _, sv, Vt = np.linalg.svd(A)
    ref = Vt[-1] / Vt[-1][0]
    p = s3.Problem(s3.KIND_SCALE)
    p.set_vertices(np.ones((n, 1)))
    p.set_edges(v0, v1, s.reshape(-1, 1))
    p.set_pcg(1e-13, 100000)
    p.set_preconditioner(s3.PRECOND_MULTILEVEL)
    x, lmin, lmax, its = p.smallest_eigenvector(60, 1e-13)
    x = x / x[0]
    assert np.abs(x - ref).max() <= 1e-6 * np.abs(ref).max()


def test_kcycle_fewer_iterations_same_solution():
    """K-cycle (two inner CG steps on the largest coarse levels, one cooperative kernel for the small ones)
    against the V-cycle on a 9k-pose sphere at a late-iteration linearisation point and damping: same solution
    (backward error against the same H and b, with a host product independent of the device SpMV the PCG uses), fewer
    iterations, bitwise reproducible."""
    import os
    import sim3opt_b200 as s3
    from sim3opt_b200 import synth
    g = dict(synth.sphere(n_laps=30, poses_per_lap=300, seed=42))
    warm = make_gpu(g, jac=1, math_mode=s3.MATH_CORRECTED)
    warm.set_pcg(1e-3, 20000)
    warm.optimize(5)                                         # a late-iteration linearisation point, shared by all runs
    g["est"] = warm.vertices()
    del warm
    res = {}
    for k in ("0", "1", "2"):
        os.environ["S3O_KCYCLE"] = k
        try:
            gpu = make_gpu(g, jac=1, math_mode=s3.MATH_CORRECTED)
            gpu.set_preconditioner(s3.PRECOND_MULTILEVEL)
            colptr, rowidx = gpu.build_structure()
            H, b = gpu.linearize()
            lam = 1e-10 * gpu.max_diag()
            gpu.set_pcg(1e-10, 50000)
            rc, x, it, rel = gpu.solve(lam)
            y = gpu.hessian_multiply(lam, x)
            rc2, x2, it2, _ = gpu.solve(lam)
        finally:
            del os.environ["S3O_KCYCLE"]
        assert rc == 0 and rel <= 1e-10
        assert backward_error(colptr, rowidx, H, lam, x, b) <= 1e-9
        assert np.linalg.norm(y - b) <= 1e-9 * np.linalg.norm(b)
        assert it2 == it and np.array_equal(x, x2)
        res[k] = (x, it)
    counts = {k: v[1] for k, v in res.items()}
    print("PCG iterations V / K1 / K2:", counts)
    for k in ("1", "2"):
        assert np.abs(res[k][0] - res["0"][0]).max() <= 1e-5 * np.abs(res["0"][0]).max()
    assert counts["1"] < counts["0"] and counts["2"] <= counts["1"], counts
    assert counts["2"] * 3 <= counts["0"] * 2, counts


def test_large_graph_kcycle_with_dense_coarsest_level():
    """Graphs of >= 20 000 free vertices take the production path of the 1M-pose benchmark: K-cycle levels inside the
    persistent kernel and a coarsest level of up to 128 vertices inverted by the row-resident block Gauss-Jordan.
    A wrong coarse inverse or Galerkin operator shows as a stalled PCG; the solution is checked against H itself, with a
    host product (the device SpMV is what the PCG runs, so it cannot be the judge)."""
    import sim3opt_b200 as s3
    from sim3opt_b200 import synth
    g = dict(synth.sphere(n_laps=30, poses_per_lap=1000, seed=7))
    warm = make_gpu(g, jac=1, math_mode=s3.MATH_CORRECTED)
    warm.set_pcg(0.1, 20000)
    warm.optimize(4)
    g["est"] = warm.vertices()
    del warm
    gpu = make_gpu(g, jac=1, math_mode=s3.MATH_CORRECTED)
    colptr, rowidx = gpu.build_structure()
    H, b = gpu.linearize()
    gpu.set_pcg(1e-10, 5000)
    out = []
    for lam_rel in (1e-4, 1e-9):
        lam = lam_rel * gpu.max_diag()
        rc, x, it, rel = gpu.solve(lam)
        assert rc == 0 and rel <= 1e-10, (lam_rel, rc, it, rel)
        assert backward_error(colptr, rowidx, H, lam, x, b) <= 1e-9
        y = gpu.hessian_multiply(lam, x)
        assert np.linalg.norm(y - b) <= 1e-9 * np.linalg.norm(b)
        assert it <= 600, (lam_rel, it)
        out.append((x, it))
    st = gpu.stats()
    assert st["multilevel_levels"] >= 2
    # same lambda again: the coarse operators are kept (only the diagonal shift is redone) and the solve is bitwise equal
    before = st["multilevel_reuses"]
    rc, x2, it2, _ = gpu.solve(1e-9 * gpu.max_diag())
    assert it2 == out[1][1] and np.array_equal(x2, out[1][0])
    assert gpu.stats()["multilevel_reuses"] == before + 1


def test_multilevel_rejected_for_ba():
    import sim3opt_b200 as s3
    from sim3opt_b200 import synth
    g = synth.ba_loop(8, 60, 4, seed=1)
    p = s3.BAProblem()
    p.set(g["cams"], g["points"], g["obs_cam"], g["obs_pt"], g["uv"], g["focal"], g["cx"], g["cy"])
    assert p.L.s3o_set_preconditioner(p.h, s3.PRECOND_MULTILEVEL) == -5      # S3O_ERR_UNSUPPORTED
