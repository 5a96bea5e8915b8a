"""Marginal covariances by the iterative route (csrc/marginals_pcg.cu): requested block columns of H^-1 by PCG solves
H x = e_(c,m) without damping, refined until the true residual |e - H x| <= S3O_MARGINALS_PCG_TOL.  The route serves
graphs whose sparse Cholesky factor exceeds the forced cap; S3O_MARGINALS_ROUTE=pcg forces it elsewhere, so that both
routes can be compared on the same H.

Gates: the forward bound |X_c - Sigma_c| <= |H^-1| |R_c| with |H^-1|_2 <= tr(Sigma) (R_c the true residual, recomputed
here with s3o_hessian_multiply) against the direct route; a closed form at scale (SCALE chain, Sigma_kl = min(k, l));
on s100k (beyond the cap) the backward error of whole block columns, the symmetry of Sigma across two columns,
determinism and the refusal of the NULL form; no change to what the LM computes; the error codes; the facade."""
import os
import subprocess
from contextlib import contextmanager

import numpy as np
import pytest

from conftest import ROOT, make_gpu

EPS = 2.0 ** -53
TAU = 1e-10      # S3O_MARGINALS_PCG_TOL


def _s3():
    import sim3opt_b200 as s3
    return s3


@contextmanager
def pcg_route():
    os.environ["S3O_MARGINALS_ROUTE"] = "pcg"
    try:
        yield
    finally:
        del os.environ["S3O_MARGINALS_ROUTE"]


def _column_pairs(nf, c):
    return np.stack([np.arange(nf, dtype=np.int32), np.full(nf, c, np.int32)], 1)


def _hnorm(gpu):
    """Frobenius norm of the symmetric H from its stored upper blocks."""
    H, _ = gpu.linearize()
    colptr, rowidx = gpu.build_structure()
    cols = np.repeat(np.arange(len(colptr) - 1), np.diff(colptr))
    off = rowidx != cols
    return np.sqrt((H[~off] ** 2).sum() + 2 * (H[off] ** 2).sum())


def _residual(gpu, X, c):
    """R = H X - E_c for a block column X (nf*d, d), H linearised at the current estimates."""
    d = gpu.d
    gpu.linearize_only()
    R = np.stack([gpu.hessian_multiply(0.0, X[:, m]) for m in range(d)], 1)
    R[c * d:(c + 1) * d] -= np.eye(d)
    return R


def _graph(request, name):
    if name == "s10k":
        from sim3opt_b200 import synth
        return synth.sphere(10, 1000, seed=42)
    return request.getfixturevalue(name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["sphere_small", "kitti_k118", "s10k"])
def test_forced_route_against_direct(request, name):
    g = _graph(request, name)
    gpu = make_gpu(g, jac=1)
    d = gpu.d
    nf = int((np.asarray(g["fixed"]) == 0).sum())
    Hn = _hnorm(gpu)
    diag = gpu.marginals()                       # the direct route's NULL call
    tr = float(np.trace(diag, axis1=1, axis2=2).sum())       # >= |H^-1|_2
    picks = np.unique(np.linspace(0, nf - 1, 7).astype(int))
    worst = worst_res = 0.0
    for c in picks:
        pairs = _column_pairs(nf, c)
        Sig = gpu.marginals(pairs)               # selected inverse on the pattern, column solves off it
        with pcg_route():
            X = gpu.marginals(pairs)
        assert not np.array_equal(X, Sig), "the iterative route did not run"
        R = _residual(gpu, X.reshape(nf * d, d), c)
        Rn = np.linalg.norm(R)
        direct_gate = 64 * Hn * tr * EPS * np.abs(Sig).max()       # kappa(H) <= |H|_F tr(Sigma)
        err = np.linalg.norm(X - Sig)
        gate = 2 * tr * Rn + direct_gate
        assert err <= gate, (c, err, gate)
        assert np.array_equal(X[c], X[c].T)
        worst, worst_res = max(worst, err / gate), max(worst_res, Rn)
    print(f"\n{name}: worst |X - Sigma| / gate {worst:.3e}, worst |R_c|_F {worst_res:.3e}, tr(Sigma) {tr:.3e}")


@pytest.mark.gpu
def test_closed_form_scale_chain_at_scale():
    """SCALE chain of 30 000 vertices, vertex 0 fixed, unit information: Sigma_kl = min(k, l) in vertex ids."""
    s3 = _s3()
    n = 30000
    p = s3.Problem(s3.KIND_SCALE)
    fixed = np.zeros(n, np.uint8)
    fixed[0] = 1
    p.set_vertices(np.ones((n, 1)), fixed)
    v0 = np.arange(n - 1, dtype=np.int32)
    p.set_edges(v0, v0 + 1, np.ones((n - 1, 1)))
    p.set_jacobian_mode(s3.JAC_ANALYTIC)
    nf = n - 1
    hinv = 1.0 / (4 * np.sin(np.pi / (2 * (2 * nf + 1))) ** 2)     # |H^-1|_2 of the path Laplacian, Dirichlet end
    worst_r = 0.0
    with pcg_route():
        for c in (0, 1, 9999, nf - 1):
            X = p.marginals(_column_pairs(nf, c))[:, 0, 0]
            R = np.linalg.norm(_residual(p, X.reshape(nf, 1), c))
            assert R <= max(TAU, 1e-13 * np.sqrt(6 * nf) * np.linalg.norm(X)), (c, R)
            ref = np.minimum(np.arange(nf), c) + 1.0
            err = np.abs(X - ref).max()
            assert err <= 2 * hinv * R, (c, err)
            worst_r = max(worst_r, R)
            print(f"\nchain column {c}: max |X - min(k, l)| {err:.3e} (max {ref.max():.0f}), |R| {R:.3e}")
        pairs = np.array([(0, nf - 1), (nf - 1, 0), (3, 30), (30, 3), (10, 11), (20, 20), (nf - 1, nf - 1), (5000, 29000)],
                         np.int32)
        got = p.marginals(pairs)[:, 0, 0]
    ref = np.minimum(pairs[:, 0], pairs[:, 1]) + 1.0
    assert np.all(np.abs(got - ref) <= 4 * hinv * max(worst_r, TAU)), (got, ref)


def _s100k():
    from sim3opt_b200 import synth
    return synth.sphere(100, 1000, seed=42)


def test_s100k_is_beyond_the_cap():
    s3 = _s3()
    g = _s100k()
    with pytest.raises(s3.S3OError, match=r"error -5:"):
        s3.host_direct_plan(len(g["est"]), g["fixed"], g["v0"], g["v1"], max_pairs=60000000)


@pytest.mark.gpu
def test_s100k_columns():
    s3 = _s3()
    g = _s100k()
    gpu = make_gpu(g, jac=1)
    d = gpu.d
    nf = int((np.asarray(g["fixed"]) == 0).sum())
    with pytest.raises(s3.S3OError, match=r"error -5: .*explicit pairs"):
        gpu.marginals()
    Hn = _hnorm(gpu)
    cols = [0, nf // 2, nf - 1]
    X, Rn = {}, {}
    for c in cols:
        X[c] = gpu.marginals(_column_pairs(nf, c))
        Xc = X[c].reshape(nf * d, d)
        R = _residual(gpu, Xc, c)
        Rn[c] = np.linalg.norm(R)
        back = Rn[c] / (Hn * np.linalg.norm(Xc))
        assert back <= 1e-10, (c, back)
        B = X[c][c]
        assert np.array_equal(B, B.T) and np.linalg.eigvalsh(B).min() > 0
        print(f"\ns100k column {c}: backward error {back:.3e}, |R|_F {np.linalg.norm(R):.3e}")
    # Sigma(r, c) from column c against Sigma(c, r)^T from column r: |H^-1|_2 = 1 / lambda_min(H)
    _, lmin, _, _ = gpu.smallest_eigenvector(50, 1e-8)
    assert lmin > 0
    a, b = cols[0], cols[-1]
    gap = np.abs(X[a][b] - X[b][a].T).max()
    gate = 2.0 / lmin * (Rn[a] + Rn[b])
    assert gap <= gate, (gap, gate)
    print(f"s100k: |Sigma(r,c) - Sigma(c,r)^T| {gap:.3e} (gate {gate:.3e}, lambda_min {lmin:.3e})")
    # bitwise determinism
    again = gpu.marginals(_column_pairs(nf, cols[1]))
    assert np.array_equal(again, X[cols[1]])


LM_STATS = ("pcg_iterations", "pcg_unconverged", "ms_spmv_sampled", "n_spmv_sampled", "direct_solves",
            "multilevel_rebuilds", "multilevel_reuses")


def _lm_twins(g, between, setup=None, its=2):
    a, b = make_gpu(g, jac=1), make_gpu(g, jac=1)
    out = []
    for p, with_marginals in ((a, True), (b, False)):
        if setup:
            setup(p)
        p.set_lm_resume(1)
        h1 = p.optimize(its)[3]
        if with_marginals:
            between(p)
        h2 = p.optimize(its)[3]
        out.append((h1, h2, p.vertices(), p.stats()))
    (ha1, ha2, va, sa), (hb1, hb2, vb, sb) = out
    assert np.array_equal(ha1, hb1) and np.array_equal(ha2, hb2)
    assert np.array_equal(va, vb)
    for k in LM_STATS:
        if k == "ms_spmv_sampled":
            assert sa["n_spmv_sampled"] == sb["n_spmv_sampled"]
            continue
        assert sa[k] == sb[k], (k, sa[k], sb[k])
    return sa


@pytest.mark.gpu
def test_no_change_to_the_lm(sphere_small):
    s3 = _s3()
    g = _s100k()
    nf = int((np.asarray(g["fixed"]) == 0).sum())
    _lm_twins(g, lambda p: p.marginals(np.array([[nf - 1, nf - 1], [0, nf - 1]], np.int32)))

    # AUTO on a small graph, PCG linear solver: block-Jacobi with the switch to the multilevel PCG once a solve gets
    # expensive (auto_multilevel), batches sized by the previous solve (last_pcg_iters)
    def setup(p):
        p.set_linear_solver(s3.LINSOLVER_PCG)
        p.set_pcg(1e-10, 5000)

    def between(p):
        with pcg_route():
            p.marginals(np.array([[5, 5], [100, 5]], np.int32))

    st = _lm_twins(sphere_small, between, setup, its=4)
    assert st["pcg_iterations"] > 0


@pytest.mark.gpu
def test_errors(kitti_k1):
    s3 = _s3()
    from sim3opt_b200 import synth
    gpu = make_gpu(kitti_k1, jac=1)
    nf = int((np.asarray(kitti_k1["fixed"]) == 0).sum())
    with pcg_route():
        for bad in ([[-1, 0]], [[0, nf]], [[nf + 5, 2]]):
            with pytest.raises(s3.S3OError, match=r"error -1:"):
                gpu.marginals(bad)
        with pytest.raises(s3.S3OError, match=r"error -5: .*explicit pairs"):
            gpu.marginals()
        ba_g = synth.ba_loop(30, 900, 6, seed=21)
        ba = s3.BAProblem()
        ba.set(ba_g["cams"], ba_g["points"], ba_g["obs_cam"], ba_g["obs_pt"], ba_g["uv"], ba_g["focal"], ba_g["cx"], ba_g["cy"])
        with pytest.raises(s3.S3OError, match=r"error -5:"):
            ba.marginals()


FACADE_DRIVER = r'''
#include <cstdio>
#include "sim3opt_b200/g2o_facade.hpp"
int main(int argc, char **argv) {
    FILE *f = std::fopen(argv[1], "r");
    int n = 0, ne = 0, m = 0;
    if (std::fscanf(f, "%d %d %d", &n, &ne, &m) != 3) return 2;
    g2o::SparseOptimizer opt;
    std::vector<vio::VertexSim3Expmap *> vs;
    for (int i = 0; i < n; ++i) {
        double x[8];
        int fx = 0;
        for (double &v : x) if (std::fscanf(f, "%lf", &v) != 1) return 2;
        if (std::fscanf(f, "%d", &fx) != 1) return 2;
        auto *v = new vio::VertexSim3Expmap();
        v->setId(i);
        v->setFixed(fx != 0);
        v->setEstimate(g2o::Sim3::unpack(x));
        opt.addVertex(v);
        vs.push_back(v);
    }
    for (int k = 0; k < ne; ++k) {
        int a = 0, b = 0;
        double x[8];
        if (std::fscanf(f, "%d %d", &a, &b) != 2) return 2;
        for (double &v : x) if (std::fscanf(f, "%lf", &v) != 1) return 2;
        auto *e = new vio::EdgeSim3();
        e->setVertex(0, opt.vertex(a));
        e->setVertex(1, opt.vertex(b));
        e->setMeasurement(g2o::Sim3::unpack(x));
        for (int i = 0; i < 49; ++i) if (std::fscanf(f, "%lf", &e->information().data()[i]) != 1) return 2;
        opt.addEdge(e);
    }
    std::vector<std::pair<int, int>> idx(m);
    for (auto &q : idx) if (std::fscanf(f, "%d %d", &q.first, &q.second) != 2) return 2;
    if (!opt.initializeOptimization()) return 3;
    g2o::SparseBlockMatrix<g2o::MatrixX> spinv;
    if (!opt.computeMarginals(spinv, idx)) { std::fprintf(stderr, "%s\n", opt.lastError().c_str()); return 4; }
    for (auto &q : idx) {
        const g2o::MatrixX *B = spinv.block(q.first, q.second);
        if (!B) return 5;
        for (int r = 0; r < 7; ++r)
            for (int c = 0; c < 7; ++c) std::printf("%.17g\n", (*B)(r, c));
    }
    return 0;
}
'''


@pytest.mark.gpu
def test_facade_pcg_route(tmp_path, sphere_small):
    g = sphere_small
    gpu = make_gpu(g, jac=1)
    nf = int((np.asarray(g["fixed"]) == 0).sum())
    gpu.build_structure()
    hidx = gpu.hessian_index()
    pairs = np.array([(0, 0), (nf - 1, 0), (17, 200), (200, 200), (nf - 1, nf - 1)], np.int32)
    with pcg_route():
        ref = gpu.marginals(pairs)
    est, fixed = np.asarray(g["est"]).reshape(-1, 8), np.asarray(g["fixed"])
    info = np.asarray(g["info"]).reshape(-1, 49)
    meas = np.asarray(g["meas"]).reshape(-1, 8)
    v_of = {int(h): v for v, h in enumerate(hidx) if h >= 0}
    lines = [f"{len(est)} {len(meas)} {len(pairs)}"]
    lines += [" ".join(f"{x:.17g}" for x in est[i]) + f" {int(fixed[i])}" for i in range(len(est))]
    lines += [f"{int(g['v0'][k])} {int(g['v1'][k])} " + " ".join(f"{x:.17g}" for x in np.concatenate([meas[k], info[k]]))
              for k in range(len(meas))]
    # the facade takes Hessian indices as g2o does; the driver's vertex ids equal the graph's
    lines += [f"{r} {c}" for r, c in pairs]
    data = tmp_path / "graph.txt"
    data.write_text("\n".join(lines) + "\n")
    src = tmp_path / "drv.cpp"
    src.write_text(FACADE_DRIVER)
    exe = str(tmp_path / "drv")
    subprocess.run(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), str(src), "-o", exe,
                    "-L", os.path.join(ROOT, "sim3opt_b200", "lib"), "-lsim3opt_b200",
                    "-Wl,-rpath," + os.path.join(ROOT, "sim3opt_b200", "lib")], check=True)
    env = dict(os.environ, S3O_MARGINALS_ROUTE="pcg")
    r = subprocess.run([exe, str(data)], capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0, r.stdout + r.stderr
    got = np.array(r.stdout.split(), float).reshape(len(pairs), 7, 7)
    rel = np.abs(got - ref).max() / np.abs(ref).max()
    print(f"\nfacade computeMarginals (iterative route) against the Python path: max rel {rel:.3e}")
    assert len(v_of) == nf and rel <= 1e-6
