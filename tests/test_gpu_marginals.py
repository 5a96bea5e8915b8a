"""GPU tests of the marginal covariances (s3o_compute_marginals: g2o SparseOptimizer::computeMarginals), the selected
inverse of the device's sparse block Cholesky factor (csrc/direct.cu selinv_kernel).

Gates: a closed form (SCALE chain: Sigma_kl = min(k, l)); the dense inverse of the same H, read back with
Problem.linearize() at the same estimates, within 64 kappa(H) 2^-53 max|Sigma|; the backward error of whole block
columns (pairs off the pattern of L included), which does not depend on kappa; bitwise reproducibility; no change to
what the LM and s3o_solve compute; the error codes; the g2o-spelled facade."""
import os
import subprocess

import numpy as np
import pytest

from conftest import KITTI_DIR, ROOT, make_gpu

pytestmark = pytest.mark.gpu

EPS = 2.0 ** -53


def _s3():
    import sim3opt_b200 as s3
    return s3


def dense(gpu):
    from test_gpu_parity import dense_from_blocks
    H, _ = gpu.linearize()
    colptr, rowidx = gpu.build_structure()
    return dense_from_blocks(colptr, rowidx, H, gpu.d)


def edge_pairs(g, hidx):
    a, b = hidx[np.asarray(g["v0"])], hidx[np.asarray(g["v1"])]
    keep = (a >= 0) & (b >= 0)
    return np.stack([a[keep], b[keep]], 1)


def test_closed_form_scale_chain():
    """H of a SCALE chain at its measurements (s = 1, unit information, vertex 0 fixed) is the path Laplacian with a
    Dirichlet end: Sigma_kl = min(k, l) in vertex ids."""
    s3 = _s3()
    n = 40
    p = s3.Problem(s3.KIND_SCALE)
    fixed = np.zeros(n, np.uint8)
    fixed[0] = 1
    p.set_vertices(np.ones((n, 1)), fixed)
    v0 = np.arange(n - 1, dtype=np.int32)
    p.set_edges(v0, v0 + 1, np.ones((n - 1, 1)))
    p.set_jacobian_mode(s3.JAC_ANALYTIC)
    diag = p.marginals()[:, 0, 0]
    k = np.arange(1, n)
    assert np.abs(diag - k).max() <= 1e-12 * k.max()
    assert np.all(np.abs(diag - k) <= 1e-12 * k)
    pairs = np.array([(0, n - 2), (n - 2, 0), (3, 30), (30, 3), (10, 11), (20, 20), (5, 37)], np.int32)
    got = p.marginals(pairs)[:, 0, 0]
    ref = np.minimum(pairs[:, 0], pairs[:, 1]) + 1.0
    assert np.all(np.abs(got - ref) <= 1e-12 * ref), (got, ref)


@pytest.mark.parametrize("name", ["kitti_k1", "kitti_k118", "sphere_small", "manhattan_small", "k118_scale_trans"])
def test_against_dense_inverse(request, name):
    s3 = _s3()
    if name == "k118_scale_trans":
        from oracle import kitti_io
        g = kitti_io.to_scale_trans_graph(request.getfixturevalue("kitti_k118"))
        gpu = make_gpu(g, kind=s3.KIND_SCALE_TRANS, jac=1)
    else:
        g = request.getfixturevalue(name)
        gpu = make_gpu(g, jac=1)
    d = gpu.d
    A = dense(gpu)
    ref = np.linalg.inv(A)
    kappa = np.linalg.cond(A)
    hidx = gpu.hessian_index()
    diag = gpu.marginals()
    pairs = edge_pairs(g, hidx)
    offd = gpu.marginals(pairs)
    smax = np.abs(ref).max()
    err = 0.0
    for k in range(len(diag)):
        err = max(err, np.abs(diag[k] - ref[k * d:(k + 1) * d, k * d:(k + 1) * d]).max())
        assert np.array_equal(diag[k], diag[k].T)
    for (r, c), B in zip(pairs, offd):
        err = max(err, np.abs(B - ref[r * d:(r + 1) * d, c * d:(c + 1) * d]).max())
    gate = 64 * kappa * EPS * smax
    print(f"\nmarginals {name}: d {d} kappa {kappa:.3e} max|dSigma| {err:.3e} gate {gate:.3e} ratio {err / gate:.3e}")
    assert err <= gate
    # the same values again, bit for bit (one writer per block, fixed summation order)
    assert np.array_equal(gpu.marginals(), diag)
    assert np.array_equal(gpu.marginals(pairs), offd)


def _column_pairs(nf, c):
    return np.stack([np.arange(nf, dtype=np.int32), np.full(nf, c, np.int32)], 1)


def _backward_error(gpu, Hnorm, nf, cols):
    d = gpu.d
    worst = 0.0
    for c in cols:
        X = gpu.marginals(_column_pairs(nf, c)).reshape(nf * d, d)      # block column c of H^-1
        gpu.linearize_only()
        R = np.stack([gpu.hessian_multiply(0.0, X[:, m]) for m in range(d)], 1)
        R[c * d:(c + 1) * d] -= np.eye(d)
        ratio = np.linalg.norm(R) / (Hnorm * np.linalg.norm(X))
        worst = max(worst, ratio)
        assert ratio <= 1e-12, (c, ratio)
    return worst


def test_block_columns_backward_error(kitti_k118, sphere_small):
    """Whole block columns (far pairs solved with the factor, pairs on the pattern from the selected inverse)."""
    for g in (kitti_k118, sphere_small):
        gpu = make_gpu(g, jac=1)
        A = dense(gpu)
        nf = A.shape[0] // 7
        w = _backward_error(gpu, np.linalg.norm(A), nf, [0, nf // 3, nf - 1])
        print(f"\nblock-column backward error: {w:.3e}")


def test_s10k_columns():
    """s10k sphere (no dense inverse fits): backward error of block columns, and their blocks on the pattern against an
    independent exact solve of H X = E_c through the linear-solver handle, within the kappa-scaled gate."""
    import scipy.sparse as sp
    import scipy.sparse.linalg as spla
    s3 = _s3()
    from sim3opt_b200 import synth
    g = synth.sphere(10, 1000, seed=42)          # the bench's s10k graph
    gpu = make_gpu(g, jac=1)
    H, _ = gpu.linearize()
    colptr, rowidx = gpu.build_structure()
    nf, d = len(colptr) - 1, 7
    cols = np.repeat(np.arange(nf), np.diff(colptr))
    off = rowidx != cols
    low = sp.bsr_matrix((np.ascontiguousarray(H[off].transpose(0, 2, 1)), rowidx[off],
                         np.concatenate([[0], np.cumsum(np.bincount(cols[off], minlength=nf))])), shape=(nf * d, nf * d))
    dg = sp.block_diag([sp.csr_matrix(B) for B in H[~off]], format="csr")
    A = (dg + low + low.T).tocsc()
    lmax = spla.eigsh(A, k=1, which="LM", return_eigenvectors=False)[0]
    lmin = spla.eigsh(A, k=1, sigma=0, which="LM", return_eigenvectors=False)[0]
    kappa = lmax / lmin
    Hnorm = spla.norm(A)
    picks = [0, nf // 2, nf - 1]
    w = _backward_error(gpu, Hnorm, nf, picks)
    ls = s3.LinearSolver(7)
    ls.set_linear_solver(s3.LINSOLVER_DIRECT)
    worst = 0.0
    for c in picks:
        X = gpu.marginals(_column_pairs(nf, c))
        E = np.zeros((nf * d, d))
        E[c * d:(c + 1) * d] = np.eye(d)
        Y = np.stack([ls.solve(colptr, rowidx, H, E[:, m])[1] for m in range(d)], 1).reshape(nf, d, d)
        nb = set(rowidx[cols == c]) | set(cols[rowidx == c])          # the pattern of H around c (in L's pattern)
        for r in nb:
            worst = max(worst, np.abs(X[r] - Y[r]).max())
        gate = 64 * kappa * EPS * np.abs(Y).max()
        assert worst <= gate, (c, worst, gate)
    print(f"\ns10k: kappa {kappa:.3e} backward {w:.3e} on-pattern max|d| {worst:.3e}")


def test_no_change_to_the_lm(kitti_k1, sphere_small):
    s3 = _s3()
    # AUTO on a mesh picks the PCG; computing marginals (on a forced-cap plan) must not change that
    a, b = make_gpu(sphere_small, jac=1), make_gpu(sphere_small, jac=1)
    a.marginals()
    ra, rb = a.optimize(6), b.optimize(6)
    assert np.array_equal(ra[3], rb[3]) and ra[1] == rb[1]
    assert np.array_equal(a.vertices(), b.vertices())
    st = a.stats()
    assert st["direct_solves"] == 0 and st["pcg_iterations"] > 0 and st["direct_levels"] == 0
    # resumed LM on K1: optimize(3), marginals, optimize(3) == optimize(3), optimize(3)
    a, b = make_gpu(kitti_k1, jac=1), make_gpu(kitti_k1, jac=1)
    for p in (a, b):
        p.set_lm_resume(1)
    ha1, hb1 = a.optimize(3)[3], b.optimize(3)[3]
    a.marginals()
    ha2, hb2 = a.optimize(3)[3], b.optimize(3)[3]
    assert np.array_equal(ha1, hb1) and np.array_equal(ha2, hb2)
    assert np.array_equal(a.vertices(), b.vertices())
    # s3o_solve(lambda) with and without marginals computed in between (a PCG solve starts from the previous step)
    for solver in (s3.LINSOLVER_AUTO, s3.LINSOLVER_DIRECT, s3.LINSOLVER_PCG):
        a, b = make_gpu(kitti_k1, jac=1), make_gpu(kitti_k1, jac=1)
        xs = []
        for p, with_marginals in ((a, True), (b, False)):
            p.set_linear_solver(solver)
            p.linearize_only()
            _, x0, _, _ = p.solve(1e-3)
            if with_marginals:
                p.marginals()
            p.linearize_only()
            _, x1, _, _ = p.solve(1e-3)
            xs.append((x0, x1))
        assert np.array_equal(xs[0][0], xs[1][0]) and np.array_equal(xs[0][1], xs[1][1]), solver
        if solver != s3.LINSOLVER_PCG:
            assert np.array_equal(xs[0][0], xs[0][1])             # exact solves: the same system, the same answer


def test_errors(kitti_k1):
    s3 = _s3()
    from sim3opt_b200 import synth
    # gauge-free SCALE graph (test_scale_null_vector_exact_solver): no vertex fixed
    g = kitti_k1
    n = len(g["est"])
    p = s3.Problem(s3.KIND_SCALE)
    p.set_vertices(np.ones((n, 1)))
    p.set_edges(g["v0"], g["v1"], g["meas"][:, 7].reshape(-1, 1))
    with pytest.raises(s3.S3OError, match=r"error -6: .*no fixed vertex"):
        p.marginals()
    # fixed or out-of-range Hessian index
    gpu = make_gpu(kitti_k1, jac=1)
    nf = int((np.asarray(kitti_k1["fixed"]) == 0).sum())
    for bad in ([[-1, 0]], [[0, nf]], [[nf + 5, 2]]):
        with pytest.raises(s3.S3OError, match=r"error -1:"):
            gpu.marginals(bad)
    # bundle adjustment
    ba_g = synth.ba_loop(30, 900, 6, seed=21)
    ba = s3.BAProblem()
    ba.set(ba_g["cams"], ba_g["points"], ba_g["obs_cam"], ba_g["obs_pt"], ba_g["uv"], ba_g["focal"], ba_g["cx"], ba_g["cy"])
    with pytest.raises(s3.S3OError, match=r"error -5:"):
        ba.marginals()


def test_facade_kitti_pgo_marginals(tmp_path, kitti_k1):
    subprocess.run(["make", "-C", os.path.join(ROOT, "examples")], check=True, stdout=subprocess.DEVNULL)
    out_file, marg_file = str(tmp_path / "direct.txt"), str(tmp_path / "marg.txt")
    r = subprocess.run([os.path.join(ROOT, "examples", "bin", "kitti_pgo"), "direct", KITTI_DIR, out_file, "--iters", "5",
                        "--marginals", marg_file], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    rows = np.array([l.split() for l in open(marg_file) if not l.startswith("%")], float)
    assert rows.shape == (770, 50)
    assert np.array_equal(rows[:, 0].astype(int), kitti_k1["frame_ids"][1:])
    gpu = make_gpu(kitti_k1, jac=1)
    gpu.set_pcg(1e-13, 100000)
    gpu.optimize(5)
    ref = gpu.marginals().reshape(770, 49)
    rel = np.abs(rows[:, 1:] - ref).max() / np.abs(ref).max()
    print(f"\nkitti_pgo --marginals against the Python path: max rel {rel:.3e}")
    assert rel <= 1e-6
    # computeMarginals(spinv, vertex) is false for the fixed vertex 0: through a tiny driver of the facade
    src = tmp_path / "fixed_vertex.cpp"
    src.write_text(r'''
#include "sim3opt_b200/g2o_facade.hpp"
int main() {
    g2o::SparseOptimizer opt;
    for (int i = 0; i < 3; ++i) {
        auto *v = new vio::VertexSim3Expmap();
        v->setId(i);
        v->setFixed(i == 0);
        v->setEstimate(g2o::Sim3(g2o::Quaternion(1, 0, 0, 0), g2o::Vector3(i, 0, 0), 1.0));
        opt.addVertex(v);
    }
    for (int i = 1; i < 3; ++i) {
        auto *e = new vio::EdgeSim3();
        e->setVertex(0, opt.vertex(i));
        e->setVertex(1, opt.vertex(i - 1));
        e->setMeasurement(g2o::Sim3(g2o::Quaternion(1, 0, 0, 0), g2o::Vector3(-1, 0, 0), 1.0));
        opt.addEdge(e);
    }
    if (!opt.initializeOptimization()) return 2;
    g2o::SparseBlockMatrix<g2o::MatrixX> spinv;
    if (opt.computeMarginals(spinv, opt.vertex(0))) return 3;
    if (!opt.computeMarginals(spinv, opt.vertex(2)) || !spinv.block(1, 1) || spinv.block(0, 0)) return 4;
    std::printf("%.17g\n", (*spinv.block(1, 1))(6, 6));
    return 0;
}
''')
    exe = str(tmp_path / "fixed_vertex")
    subprocess.run(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), str(src), "-o", exe,
                    "-L", os.path.join(ROOT, "sim3opt_b200", "lib"), "-lsim3opt_b200",
                    "-Wl,-rpath," + os.path.join(ROOT, "sim3opt_b200", "lib")], check=True)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert float(r.stdout) > 0
