"""GPU tests of the bundle-adjustment marginal covariances (s3o_ba_compute_marginals / BAProblem.ba_marginals): camera
blocks from the selected inverse of the Schur complement (csrc/direct.cu selinv_kernel<6>), point and camera-point
blocks from the point phase (csrc/ba.cu ba_marginal_points_kernel).

Gates: the dense inverse of the same H (assembled from the CPU oracle's linearisation at the same estimates) within
64 kappa(H) 2^-53 max|Sigma|, as in test_gpu_marginals.py; at the bench size, the backward error of camera block columns
against the device's Schur complement and the numpy twin (test_ba_marginals_host.py) fed with the device's Sigma_cc;
exact symmetry and transposition; bitwise reproducibility; no change to what the LM and s3o_solve compute; the error
codes; the g2o-spelled facade."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from sim3opt_b200 import synth
from test_ba_marginals_host import (HUBER, ba_fixings, dense_h, dense_schur, dense_scc, hessian_indices,
                                    oracle_system, point_observations, random_info, twin)

pytestmark = pytest.mark.gpu

EPS = 2.0 ** -53


def _s3():
    import sim3opt_b200 as s3
    return s3


@pytest.fixture(scope="module")
def ba_small():
    return synth.ba_loop(24, 300, 5, seed=11)


@pytest.fixture(scope="module")
def ba_medium():
    return synth.ba_loop(120, 6000, 8, seed=5)


def make_ba(g, cf, pf, info=None, robust=True):
    s3 = _s3()
    p = s3.BAProblem()
    p.set(g["cams"], g["points"], g["obs_cam"], g["obs_pt"], g["uv"], g["focal"], g["cx"], g["cy"],
          cam_fixed=cf, pt_fixed=pf, info=info)
    if robust:
        p.set_robust(HUBER, 2.5)
    p.build_structure()
    return p


def observed_pairs(g, ch, ph):
    """Distinct (camera, point) Hessian-index pairs of observations between free vertices."""
    c, q = ch[g["obs_cam"]], ph[g["obs_pt"]]
    keep = (c >= 0) & (q >= 0)
    return np.unique(np.stack([c[keep], q[keep]], 1), axis=0)


def sparse_h(Hpp, Hll, Hpl, g, ch, ph):
    import scipy.sparse as sp
    ncf, npf = len(Hpp), len(Hll)
    n = 6 * ncf + 3 * npf
    r6, c6 = np.meshgrid(np.arange(6), np.arange(6), indexing="ij")
    r3, c3 = np.meshgrid(np.arange(3), np.arange(3), indexing="ij")
    rows, cols, vals = [], [], []
    i = np.arange(ncf)[:, None, None] * 6
    rows.append((i + r6).ravel()); cols.append((i + c6).ravel()); vals.append(Hpp.ravel())
    i = 6 * ncf + np.arange(npf)[:, None, None] * 3
    rows.append((i + r3).ravel()); cols.append((i + c3).ravel()); vals.append(Hll.ravel())
    c, q = ch[g["obs_cam"]], ph[g["obs_pt"]]
    keep = (c >= 0) & (q >= 0)
    ci = c[keep][:, None, None] * 6
    qi = 6 * ncf + (q[keep][:, None, None] - ncf) * 3
    rr, cc = np.meshgrid(np.arange(6), np.arange(3), indexing="ij")
    B = Hpl[keep]
    rows += [(ci + rr).ravel(), (qi + cc).ravel()]
    cols += [(qi + cc).ravel(), (ci + rr).ravel()]
    vals += [B.ravel(), B.ravel()]
    return sp.csc_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(n, n))


def kappa_sparse(A):
    import scipy.sparse.linalg as spla
    lmax = spla.eigsh(A, k=1, which="LM", return_eigenvectors=False)[0]
    lmin = spla.eigsh(A, k=1, sigma=0, which="LM", return_eigenvectors=False)[0]
    return lmax / lmin


def on_pattern_of_l(colptr, rowidx, pairs):
    """Which camera pairs are blocks of the factor L of S (the plan AUTO / DIRECT factorises with)."""
    s3 = _s3()
    nf = len(colptr) - 1
    cols = np.repeat(np.arange(nf), np.diff(colptr))
    off = rowidx != cols
    plan = s3.host_direct_plan(nf, np.zeros(nf, np.uint8), rowidx[off].astype(np.int32), cols[off].astype(np.int32),
                               max_pairs=60000000)
    pos = np.empty(nf, int)
    pos[plan["perm"]] = np.arange(nf)
    bcol = np.repeat(np.arange(plan["n"]), np.diff(plan["cptr"]))
    blocks = set(zip(plan["brow"].tolist(), bcol.tolist()))
    a, b = pos[pairs[:, 0]], pos[pairs[:, 1]]
    return np.array([(max(x, y), min(x, y)) in blocks for x, y in zip(a, b)])


def test_dense_truth_small(ba_small):
    g = ba_small
    cf, pf = ba_fixings(g)
    info = random_info(g)
    gpu = make_ba(g, cf, pf, info)
    _, _, _, Hpp, Hll, Hpl = oracle_system(g, cf, pf, info)
    ch, ph = hessian_indices(cf, pf)
    A = dense_h(Hpp, Hll, Hpl, g, ch, ph)
    ref = np.linalg.inv(A)
    kappa = np.linalg.cond(A)
    ncf, npf = gpu.ncf, gpu.npf
    assert (ncf, npf) == (len(Hpp), len(Hll))
    cams, pts = gpu.ba_marginals()
    err = 0.0
    for i in range(ncf):
        assert np.array_equal(cams[i], cams[i].T)
        err = max(err, np.abs(cams[i] - ref[6 * i:6 * i + 6, 6 * i:6 * i + 6]).max())
    for li in range(npf):
        assert np.array_equal(pts[li], pts[li].T)
        o = 6 * ncf + 3 * li
        err = max(err, np.abs(pts[li] - ref[o:o + 3, o:o + 3]).max())
    # every camera-camera pair, on and off the pattern of L
    cc = np.array([(i, j) for i in range(ncf) for j in range(ncf)], np.int32)
    on = on_pattern_of_l(*gpu.build_structure(), cc)
    assert on.any() and not on.all()
    for (i, j), B in zip(cc, gpu.ba_marginals(cc)):
        err = max(err, np.abs(B - ref[6 * i:6 * i + 6, 6 * j:6 * j + 6]).max())
    # every observed camera-point pair, both orientations; (point, camera) is the transpose bit for bit
    cl = observed_pairs(g, ch, ph)
    both = np.concatenate([cl, cl[:, ::-1]])
    res = gpu.ba_marginals(both)
    for k, (c, q) in enumerate(cl):
        B, Bt = res[k], res[len(cl) + k]
        assert B.shape == (6, 3) and Bt.shape == (3, 6)
        assert np.array_equal(Bt, B.T)
        o = 6 * ncf + 3 * (q - ncf)
        err = max(err, np.abs(B - ref[6 * c:6 * c + 6, o:o + 3]).max())
    gate = 64 * kappa * EPS * np.abs(ref).max()
    print(f"\nba marginals ba_small: kappa {kappa:.3e} max|dSigma| {err:.3e} gate {gate:.3e} ratio {err / gate:.3e}")
    assert err <= gate


def test_medium_against_schur_inverse(ba_medium):
    g = ba_medium
    cf, pf = ba_fixings(g)
    info = random_info(g)
    gpu = make_ba(g, cf, pf, info)
    o, colptr, rowidx, Hpp, Hll, Hpl = oracle_system(g, cf, pf, info)
    ch, ph = hessian_indices(cf, pf)
    rc, S, _ = o.schur(0.0)
    assert rc == 0
    Sinv = np.linalg.inv(dense_schur(colptr, rowidx, S))
    kappa = kappa_sparse(sparse_h(Hpp, Hll, Hpl, g, ch, ph))
    pdiag, clref = twin(dense_scc(Sinv), Hll, Hpl, g, ch, ph)
    ncf, npf = gpu.ncf, gpu.npf
    cams, pts = gpu.ba_marginals()
    smax = max(np.abs(Sinv).max(), max(np.abs(B).max() for B in pdiag.values()))
    err = max(np.abs(cams[i] - Sinv[6 * i:6 * i + 6, 6 * i:6 * i + 6]).max() for i in range(ncf))
    err = max(err, max(np.abs(pts[li] - pdiag[li]).max() for li in range(npf)))
    cl = observed_pairs(g, ch, ph)
    for (c, q), B in zip(cl, gpu.ba_marginals(cl)):
        err = max(err, np.abs(B - clref[(int(c), int(q) - ncf)]).max())
    gate = 64 * kappa * EPS * smax
    print(f"\nba marginals ba_medium: kappa {kappa:.3e} max|dSigma| {err:.3e} gate {gate:.3e} ratio {err / gate:.3e}")
    assert err <= gate


def test_bench_size():
    """ba_loop(1000, 500000, 10): backward error of camera block columns against the device's Schur complement, and a
    sample of 1000 points against the twin fed with the device's Sigma_cc and linearisation."""
    import scipy.sparse as sp
    g = synth.ba_loop(1000, 500000, 10, seed=42)
    cf, pf = ba_fixings(g)
    gpu = make_ba(g, cf, pf)
    ncf, npf = gpu.ncf, gpu.npf
    cams, pts = gpu.ba_marginals()
    assert cams.shape == (ncf, 6, 6) and pts.shape == (npf, 3, 3)
    Hpp, Hll, Hpl, _ = gpu.linearize()
    S, _ = gpu.schur(0.0)
    colptr, rowidx = gpu.build_structure()
    A = dense_schur(colptr, rowidx, S)
    Ssp = sp.csr_matrix(A)
    Snorm = np.linalg.norm(A)
    worst = 0.0
    for c in (0, ncf // 2, ncf - 1):
        pairs = np.stack([np.arange(ncf), np.full(ncf, c)], 1).astype(np.int32)
        X = np.concatenate(gpu.ba_marginals(pairs))                 # (6 ncf, 6): block column c of S^-1
        assert np.array_equal(X[6 * c:6 * c + 6], cams[c])
        R = Ssp @ X
        R[6 * c:6 * c + 6] -= np.eye(6)
        ratio = np.linalg.norm(R) / (Snorm * np.linalg.norm(X))
        worst = max(worst, ratio)
        assert ratio <= 1e-12, (c, ratio)
    # 1000 points: Sigma_cc blocks among their cameras from the device, then the twin
    ch, ph = hessian_indices(cf, pf)
    rng = np.random.default_rng(0)
    sample = np.sort(rng.choice(npf, 1000, replace=False))
    obs = point_observations(g, ch, ph)
    need = set()
    for li in sample:
        cs = np.unique(ch[g["obs_cam"][obs[li]]])
        need.update((int(a), int(b)) for a in cs for b in cs)
    need = np.array(sorted(need), np.int32)
    blocks = dict(zip(map(tuple, need.tolist()), gpu.ba_marginals(need)))

    def scc(cs):
        return np.block([[blocks[(int(a), int(b))] for b in cs] for a in cs])

    pdiag, clref = twin(scc, Hll, Hpl, g, ch, ph, points=sample)
    cl = np.array([(c, ncf + li) for (c, li) in clref], np.int32)
    got = gpu.ba_marginals(cl)
    scale = max(max(np.abs(B).max() for B in pdiag.values()), max(np.abs(B).max() for B in clref.values()))
    err = max(np.abs(pts[li] - pdiag[li]).max() for li in sample)
    err = max(err, max(np.abs(B - clref[(int(c), int(q) - ncf)]).max() for (c, q), B in zip(cl, got)))
    print(f"\nba marginals bench size: ncf {ncf} npf {npf} column backward error {worst:.3e} "
          f"sample max|d| / max|Sigma| {err / scale:.3e}")
    assert err <= 1e-10 * scale


def test_degenerate_fixings(ba_small):
    g = ba_small
    cf, pf = ba_fixings(g)
    # all cameras fixed: Sigma(l, l) = Hll^-1, no factorisation
    gpu = make_ba(g, np.ones_like(cf), pf)
    _, Hll, _, _ = gpu.linearize()
    cams, pts = gpu.ba_marginals()
    assert cams.shape == (0, 6, 6)
    for li in range(gpu.npf):
        ref = np.linalg.inv(Hll[li])
        assert np.abs(pts[li] - ref).max() <= 64 * np.linalg.cond(Hll[li]) * EPS * np.abs(ref).max(), li
    # all points fixed: S = Hpp, the camera blocks are its inverse
    gpu = make_ba(g, cf, np.ones_like(pf))
    Hpp, _, _, _ = gpu.linearize()
    S, _ = gpu.schur(0.0)
    A = dense_schur(*gpu.build_structure(), S)
    ref = np.linalg.inv(A)
    cams, pts = gpu.ba_marginals()
    assert pts.shape == (0, 3, 3)
    gate = 64 * np.linalg.cond(A) * EPS * np.abs(ref).max()
    assert max(np.abs(cams[i] - ref[6 * i:6 * i + 6, 6 * i:6 * i + 6]).max() for i in range(gpu.ncf)) <= gate


def test_determinism(ba_small):
    g = ba_small
    cf, pf = ba_fixings(g)
    info = random_info(g)
    a, b = make_ba(g, cf, pf, info), make_ba(g, cf, pf, info)
    ch, ph = hessian_indices(cf, pf)
    pairs = np.concatenate([observed_pairs(g, ch, ph), [[0, 5], [5, 0], [3, 3]]]).astype(np.int32)
    ca, pa = a.ba_marginals()
    ra = a.ba_marginals(pairs)
    for p in (a, b):
        c, q = p.ba_marginals()
        assert np.array_equal(c, ca) and np.array_equal(q, pa)
        assert all(np.array_equal(x, y) for x, y in zip(p.ba_marginals(pairs), ra))


@pytest.mark.parametrize("solver", ["AUTO", "PCG"])
def test_no_change_to_the_lm(ba_small, solver):
    s3 = _s3()
    g = ba_small
    cf, pf = ba_fixings(g)
    kind = getattr(s3, "LINSOLVER_" + solver)
    a, b = make_ba(g, cf, pf), make_ba(g, cf, pf)
    for p in (a, b):
        p.set_linear_solver(kind)
        p.set_lm_resume(1)
    ha1, hb1 = a.optimize(3)[3], b.optimize(3)[3]
    d0 = a.stats()["direct_solves"]
    a.ba_marginals()
    assert a.stats()["direct_solves"] == d0
    ha2, hb2 = a.optimize(3)[3], b.optimize(3)[3]
    assert np.array_equal(ha1, hb1) and np.array_equal(ha2, hb2)
    assert np.array_equal(a.cameras(), b.cameras()) and np.array_equal(a.points(), b.points())
    # s3o_solve with and without marginals computed in between
    a, b = make_ba(g, cf, pf), make_ba(g, cf, pf)
    xs = []
    for p, with_marginals in ((a, True), (b, False)):
        p.set_linear_solver(kind)
        p.linearize_only()
        _, x0, _, _ = p.solve(1e-3)
        if with_marginals:
            p.ba_marginals()
        p.linearize_only()
        _, x1, _, _ = p.solve(1e-3)
        xs.append((x0, x1))
    assert np.array_equal(xs[0][0], xs[1][0]) and np.array_equal(xs[0][1], xs[1][1])


def two_view(g):
    """The graph restricted to points seen by at least two distinct cameras (no point needs fixing)."""
    seen = np.unique(np.stack([g["obs_pt"], g["obs_cam"]], 1), axis=0)
    keep_pt = np.bincount(seen[:, 0], minlength=len(g["points"])) >= 2
    new = -np.ones(len(g["points"]), int)
    new[keep_pt] = np.arange(int(keep_pt.sum()))
    ko = keep_pt[g["obs_pt"]]
    h = dict(g)
    h.update(points=g["points"][keep_pt], obs_cam=g["obs_cam"][ko], obs_pt=new[g["obs_pt"][ko]], uv=g["uv"][ko])
    return h


def test_errors(ba_small):
    s3 = _s3()
    g = ba_small
    h = two_view(g)
    nc, npts = len(h["cams"]), len(h["points"])
    # gauge-free: no fixed vertex, then one fixed camera and no second anchor
    for cf in (np.zeros(nc, np.uint8), np.eye(1, nc, 0, np.uint8).ravel()):
        p = make_ba(h, cf, np.zeros(npts, np.uint8))
        with pytest.raises(s3.S3OError, match=r"error -6: .*connected component of camera [01] "):
            p.ba_marginals()
    # a free point seen by one camera: keep one observation of point 4
    cf, pf = ba_fixings(g)
    ko = (g["obs_pt"] != 4) | (np.arange(len(g["uv"])) == np.nonzero(g["obs_pt"] == 4)[0][0])
    h = dict(g, obs_cam=g["obs_cam"][ko], obs_pt=g["obs_pt"][ko], uv=g["uv"][ko])
    p = make_ba(h, cf, pf)
    with pytest.raises(s3.S3OError, match=r"error -6: .*free point 4 is seen by 1 distinct"):
        p.ba_marginals()
    # unsupported pairs: two distinct points, a camera that does not see the point
    p = make_ba(g, cf, pf)
    ncf, n = p.ncf, p.ncf + p.npf
    ch, ph = hessian_indices(cf, pf)
    seen = set(map(tuple, observed_pairs(g, ch, ph).tolist()))
    unseen = next((c, q) for c in range(ncf) for q in range(ncf, n) if (c, q) not in seen)
    for bad in ([[ncf, ncf + 1]], [unseen], [unseen[::-1]]):
        with pytest.raises(s3.S3OError, match=r"error -5:"):
            p.ba_marginals(bad)
    # negative, out-of-range (fixed vertices have no index) indices
    for bad in ([[-1, 0]], [[0, n]], [[n + 3, 1]]):
        with pytest.raises(s3.S3OError, match=r"error -1:"):
            p.ba_marginals(bad)
    # wrong n_pairs with NULL rows
    out = np.zeros(36 * ncf + 9 * p.npf)
    assert p.L.s3o_ba_compute_marginals(p.h, n - 1, None, None, out.ctypes.data_as(C.POINTER(C.c_double))) == -1
    # a pose-graph problem and a linear-solver handle
    q = s3.Problem(s3.KIND_SIM3)
    assert q.L.s3o_ba_compute_marginals(q.h, 1, None, None, out.ctypes.data_as(C.POINTER(C.c_double))) == -1
    ls = s3.LinearSolver(6)
    assert ls.L.s3o_ba_compute_marginals(ls.h, 1, None, None, out.ctypes.data_as(C.POINTER(C.c_double))) == -1
    # the call that failed left the problem usable
    cams, _ = p.ba_marginals()
    assert cams.shape == (ncf, 6, 6)


FACADE_DRIVER = r'''
#include <cstdio>
#include <fstream>
#include "sim3opt_b200/g2o_facade.hpp"
int main(int argc, char **argv) {
    std::ifstream in(argv[1]);
    int nc, np, no;
    in >> nc >> np >> no;
    g2o::SparseOptimizer opt;
    double f, cx, cy;
    in >> f >> cx >> cy;
    auto *cam = new g2o::CameraParameters(f, g2o::Matrix<double, 2, 1>{ cx, cy }, 0.);
    cam->setId(0);
    opt.addParameter(cam);
    std::vector<g2o::VertexSE3Expmap *> cams;
    std::vector<g2o::VertexSBAPointXYZ *> pts;
    for (int i = 0; i < nc; ++i) {
        double q[7];
        int fixed;
        for (double &v : q) in >> v;
        in >> fixed;
        auto *v = new g2o::VertexSE3Expmap();
        v->setId(i);
        v->setFixed(fixed != 0);
        v->setEstimate(g2o::SE3Quat(g2o::Quaternion(q[3], q[0], q[1], q[2]), g2o::Vector3(q[4], q[5], q[6])));
        opt.addVertex(v);
        cams.push_back(v);
    }
    for (int i = 0; i < np; ++i) {
        double x, y, z;
        int fixed;
        in >> x >> y >> z >> fixed;
        auto *v = new g2o::VertexSBAPointXYZ();
        v->setId(nc + i);
        v->setMarginalized(true);
        v->setFixed(fixed != 0);
        v->setEstimate(g2o::Vector3(x, y, z));
        opt.addVertex(v);
        pts.push_back(v);
    }
    for (int k = 0; k < no; ++k) {
        int c, l;
        double u, w;
        in >> c >> l >> u >> w;
        auto *e = new g2o::EdgeProjectXYZ2UV();
        e->setVertex(0, pts[l]);
        e->setVertex(1, cams[c]);
        e->setMeasurement(g2o::Matrix<double, 2, 1>{ u, w });
        e->setParameterId(0, 0);
        opt.addEdge(e);
    }
    int ic, ip;
    in >> ic >> ip;
    if (!opt.initializeOptimization()) return 2;
    for (auto *v : cams) {                          // the estimates as the facade holds them (normalised rotations)
        double q[7];
        v->packEstimate(q);
        for (double x : q) std::printf("%.17g\n", x);
    }
    g2o::SparseBlockMatrix<g2o::MatrixX> spinv;
    if (opt.computeMarginals(spinv, cams[0])) return 3;                       // fixed camera
    const int hc = cams[ic]->hessianIndex(), hp = pts[ip]->hessianIndex();
    auto dump = [](const g2o::MatrixX *b) {
        for (int r = 0; r < b->rows(); ++r)
            for (int c = 0; c < b->cols(); ++c) std::printf("%.17g\n", (*b)(r, c));
    };
    if (!opt.computeMarginals(spinv, cams[ic]) || !spinv.block(hc, hc)) return 4;
    if (spinv.rowsOfBlock(hc) != 6) return 5;
    dump(spinv.block(hc, hc));
    if (!opt.computeMarginals(spinv, pts[ip]) || !spinv.block(hp, hp)) return 6;
    if (spinv.rowsOfBlock(hp) != 3 || spinv.colsOfBlock(hp) != 3) return 7;
    dump(spinv.block(hp, hp));
    if (!opt.computeMarginals(spinv, std::vector<std::pair<int, int>>{ { hc, hp }, { hp, hc } })) return 8;
    const g2o::MatrixX *a = spinv.block(hc, hp), *b = spinv.block(hp, hc);
    if (!a || !b || a->rows() != 6 || a->cols() != 3 || b->rows() != 3 || b->cols() != 6) return 9;
    dump(a);
    dump(b);
    return 0;
}
'''


def test_facade_ba_marginals(tmp_path, ba_small):
    g = ba_small
    cf, pf = ba_fixings(g, cams=(0, 1))
    ch, ph = hessian_indices(cf, pf)
    ic = 5
    ip = int(next(l for l in g["obs_pt"][g["obs_cam"] == ic] if ph[l] >= 0))
    data = tmp_path / "ba.txt"
    with open(data, "w") as f:
        f.write(f"{len(g['cams'])} {len(g['points'])} {len(g['uv'])}\n{g['focal']!r} {g['cx']!r} {g['cy']!r}\n")
        for q, x in zip(g["cams"], cf):
            f.write(" ".join(repr(float(v)) for v in q) + f" {int(x)}\n")
        for q, x in zip(g["points"], pf):
            f.write(" ".join(repr(float(v)) for v in q) + f" {int(x)}\n")
        for c, l, uv in zip(g["obs_cam"], g["obs_pt"], g["uv"]):
            f.write(f"{int(c)} {int(l)} {float(uv[0])!r} {float(uv[1])!r}\n")
        f.write(f"{ic} {ip}\n")
    src, exe = tmp_path / "ba_marginals.cpp", str(tmp_path / "ba_marginals")
    src.write_text(FACADE_DRIVER)
    subprocess.run(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), str(src), "-o", exe,
                    "-L", os.path.join(ROOT, "sim3opt_b200", "lib"), "-lsim3opt_b200",
                    "-Wl,-rpath," + os.path.join(ROOT, "sim3opt_b200", "lib")], check=True)
    r = subprocess.run([exe, str(data)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    vals = np.array(r.stdout.split(), float)
    nc7 = 7 * len(g["cams"])
    got = vals[nc7:]
    gpu = make_ba(dict(g, cams=vals[:nc7].reshape(-1, 7)), cf, pf, robust=False)
    hc, hp = int(ch[ic]), int(ph[ip])
    ref = np.concatenate([B.ravel() for B in gpu.ba_marginals([[hc, hc], [hp, hp], [hc, hp], [hp, hc]])])
    rel = np.abs(got - ref).max() / np.abs(ref).max()
    print(f"\nfacade BA computeMarginals against the Python path: max rel {rel:.3e}")
    assert rel <= 1e-12
