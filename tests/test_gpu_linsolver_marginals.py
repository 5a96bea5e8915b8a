"""Marginal covariances at the LinearSolver cut (s3o_linsolver_solve_pattern, g2o LinearSolver::solvePattern /
solveBlocks): blocks of A^-1 for an upper block-CCS A uploaded to a s3o_linsolver handle.

Gates: the H of a problem, read back with s3o_get_hessian and fed to a handle, gives s3o_compute_marginals' blocks bit
for bit (same H bits, same plan, same kernels); the dense inverse within 64 kappa eps max|Sigma|, also for the 6x6 BA
Hpp and the BA Schur complement (whose camera blocks equal s3o_ba_compute_marginals'); row- and column-major blocks
alike; the PCG route on a handle (block-Jacobi, within the bound of test_gpu_marginals_pcg.py, true residuals); no
effect on later solves or on the solver statistics; pattern changes; the error codes; reproducibility."""
import ctypes as C
import os
from contextlib import contextmanager

import numpy as np
import pytest

from conftest import make_gpu

EPS = 2.0 ** -53
TAU = 1e-10      # S3O_MARGINALS_PCG_TOL


def _s3():
    import sim3opt_b200 as s3
    return s3


@contextmanager
def env(**kw):
    old = {k: os.environ.get(k) for k in kw}
    os.environ.update(kw)
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v


def _graph(request, name):
    """(graph, kind) of a named test graph: K1, K118 and sphere_small at Sim3, K118 at scale-trans and at scale."""
    s3 = _s3()
    if name == "k118_scale_trans":
        from oracle import kitti_io
        return kitti_io.to_scale_trans_graph(request.getfixturevalue("kitti_k118")), s3.KIND_SCALE_TRANS
    if name == "k118_scale":
        g = request.getfixturevalue("kitti_k118")
        return dict(est=np.ascontiguousarray(g["est"][:, 7:8]), fixed=g["fixed"], v0=g["v0"], v1=g["v1"],
                    meas=np.ascontiguousarray(g["meas"][:, 7:8])), s3.KIND_SCALE
    return request.getfixturevalue(name), s3.KIND_SIM3


def _system(request, name):
    """A problem linearised at its estimates and its H in g2o's block-CCS order."""
    g, kind = _graph(request, name)
    p = make_gpu(g, kind=kind, jac=1)
    H, _ = p.linearize()
    colptr, rowidx = p.build_structure()
    return g, p, colptr, rowidx, H


def _pairs(g, p, nf, seed=0):
    """Every edge pair between free vertices, both orientations of a few, and far pairs (mostly off the factor's
    pattern)."""
    hidx = p.hessian_index()
    a, b = hidx[np.asarray(g["v0"])], hidx[np.asarray(g["v1"])]
    keep = (a >= 0) & (b >= 0)
    edges = np.stack([a[keep], b[keep]], 1)
    rng = np.random.default_rng(seed)
    far = rng.choice(nf, 12, replace=False)
    far = np.stack([far, (far + nf // 2) % nf], 1)
    return np.concatenate([edges, edges[:5, ::-1], far, far[:, ::-1]]).astype(np.int32)


def _dense(colptr, rowidx, H, d):
    from test_gpu_parity import dense_from_blocks
    return dense_from_blocks(colptr, rowidx, H, d)


GRAPHS = ["kitti_k1", "kitti_k118", "sphere_small", "k118_scale_trans", "k118_scale"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", GRAPHS)
def test_same_h_same_answer(request, name):
    s3 = _s3()
    g, p, colptr, rowidx, H = _system(request, name)
    d, nf = p.d, len(colptr) - 1
    pairs = _pairs(g, p, nf)
    ls = s3.LinearSolver(d)
    diag = ls.marginals(colptr, rowidx, H)
    offd = ls.marginals(colptr, rowidx, H, pairs)
    assert np.array_equal(diag, p.marginals())
    assert np.array_equal(offd, p.marginals(pairs))
    assert all(np.array_equal(B, B.T) for B in diag)


@pytest.mark.gpu
@pytest.mark.parametrize("name", GRAPHS)
def test_against_dense_inverse(request, name):
    s3 = _s3()
    g, p, colptr, rowidx, H = _system(request, name)
    d, nf = p.d, len(colptr) - 1
    A = _dense(colptr, rowidx, H, d)
    ref, kappa = np.linalg.inv(A), np.linalg.cond(A)
    pairs = _pairs(g, p, nf)
    ls = s3.LinearSolver(d)
    diag = ls.marginals(colptr, rowidx, H)
    offd = ls.marginals(colptr, rowidx, H, pairs)
    err = max(np.abs(diag - np.stack([ref[k * d:(k + 1) * d, k * d:(k + 1) * d] for k in range(nf)])).max(),
              max(np.abs(B - ref[r * d:(r + 1) * d, c * d:(c + 1) * d]).max() for (r, c), B in zip(pairs, offd)))
    gate = 64 * kappa * EPS * np.abs(ref).max()
    print(f"\n{name}: d {d} kappa {kappa:.3e} max|dSigma| {err:.3e} gate {gate:.3e}")
    assert err <= gate


def _ba():
    from sim3opt_b200 import synth
    from test_ba_marginals_host import ba_fixings
    from test_gpu_ba_marginals import make_ba
    g = synth.ba_loop(24, 300, 5, seed=11)
    cf, pf = ba_fixings(g)
    return make_ba(g, cf, pf)


@pytest.mark.gpu
def test_ba_hpp_and_schur_complement():
    """g2o's BlockSolver_6_3 hands solvePattern the camera block Hpp of H: block diagonal, so its inverse is the
    blocks' inverses.  The Schur complement at lambda = 0 gives the true camera marginals, bit for bit those of
    s3o_ba_compute_marginals."""
    s3 = _s3()
    ba = _ba()
    Hpp, _, _, _ = ba.linearize()
    ncf = len(Hpp)
    ls = s3.LinearSolver(6)
    ident = np.arange(ncf + 1, dtype=np.int32)
    got = ls.marginals(ident, ident[:-1], Hpp)
    ref = np.linalg.inv(Hpp)
    kappa = max(np.linalg.cond(B) for B in Hpp)
    assert np.abs(got - ref).max() <= 64 * kappa * EPS * np.abs(ref).max()
    # 6x6 blocks on the PCG route: block-Jacobi is the exact inverse of a block-diagonal Hpp
    with env(S3O_MARGINALS_ROUTE="pcg"):
        X = ls.marginals(ident, ident[:-1], Hpp, np.stack([ident[:-1], ident[:-1]], 1))
    tr = float(np.trace(ref, axis1=1, axis2=2).sum())
    assert np.abs(X - ref).max() <= 2 * tr * np.sqrt(6) * TAU + 64 * kappa * EPS * np.abs(ref).max()
    assert all(np.array_equal(B, B.T) for B in X)
    colptr, rowidx = ba.build_structure()
    S, _ = ba.schur(0.0)
    cams, _ = ba.ba_marginals()
    assert np.array_equal(ls.marginals(colptr, rowidx, S), cams)
    cols = np.repeat(np.arange(ncf), np.diff(colptr))
    cc = np.stack([rowidx, cols], 1)[rowidx != cols].astype(np.int32)
    cc = np.concatenate([cc, cc[:, ::-1], [[0, ncf - 1], [ncf - 1, 1]]]).astype(np.int32)
    assert all(np.array_equal(a, b) for a, b in zip(ls.marginals(colptr, rowidx, S, cc), ba.ba_marginals(cc)))
    A = _dense(colptr, rowidx, S, 6)
    ref = np.linalg.inv(A)
    err = max(np.abs(cams[k] - ref[6 * k:6 * k + 6, 6 * k:6 * k + 6]).max() for k in range(ncf))
    assert err <= 64 * np.linalg.cond(A) * EPS * np.abs(ref).max()


@pytest.mark.gpu
def test_layouts(kitti_k118):
    s3 = _s3()
    p = make_gpu(kitti_k118, jac=1)
    H, _ = p.linearize()
    colptr, rowidx = p.build_structure()
    pairs = _pairs(kitti_k118, p, len(colptr) - 1)
    ls = s3.LinearSolver(7)
    Ht = np.ascontiguousarray(H.transpose(0, 2, 1))
    assert np.array_equal(ls.marginals(colptr, rowidx, H), ls.marginals(colptr, rowidx, Ht, column_major=True))
    assert np.array_equal(ls.marginals(colptr, rowidx, H, pairs), ls.marginals(colptr, rowidx, Ht, pairs, column_major=True))


def _column_pairs(nf, c):
    return np.stack([np.arange(nf, dtype=np.int32), np.full(nf, c, np.int32)], 1)


# K118 (kappa ~4e12): block-Jacobi does not bring every column to the tolerance within the 20 000-iteration cap.  Such
# a column is refused with the residual it reached (S3O_ERR_SOLVE, as documented); the route is deterministic, so which
# columns are served is fixed.
@pytest.mark.gpu
@pytest.mark.parametrize("name,served,missed", [("sphere_small", (0, 159, 478), ()), ("kitti_k118", (0,), (256,))])
def test_pcg_route(request, capfd, name, served, missed):
    """S3O_MARGINALS_ROUTE=pcg on a handle: block-Jacobi (no hierarchy: a handle has no estimates), the forward bound
    of test_gpu_marginals_pcg.py against the direct route, and the true residual of every right-hand side."""
    s3 = _s3()
    g, p, colptr, rowidx, H = _system(request, name)
    d, nf = p.d, len(colptr) - 1
    import scipy.sparse as sp
    Ad = _dense(colptr, rowidx, H, d)
    A, Hn = sp.csr_matrix(Ad), np.linalg.norm(Ad)
    ls = s3.LinearSolver(d)
    diag = ls.marginals(colptr, rowidx, H)
    tr = float(np.trace(diag, axis1=1, axis2=2).sum())       # >= |A^-1|_2
    for c in served:
        pairs = _column_pairs(nf, c)
        Sig = ls.marginals(colptr, rowidx, H, pairs)
        capfd.readouterr()
        with env(S3O_MARGINALS_ROUTE="pcg", S3O_MARGINALS_TRACE="1"):
            X = ls.marginals(colptr, rowidx, H, pairs)
        trace = capfd.readouterr().err
        assert "s3o_linsolver_solve_pattern: preconditioner block-Jacobi" in trace, trace[-2000:]
        assert "multilevel" not in trace
        print(f"\n{name}: " + "".join(line for line in trace.splitlines() if "PCG iterations" in line))
        assert not np.array_equal(X, Sig), "the iterative route did not run"
        Xc = X.reshape(nf * d, d)
        R = A @ Xc
        R[c * d:(c + 1) * d] -= np.eye(d)
        for m in range(d):          # each right-hand side: the tolerance, or the backward-error fallback
            res, xn = np.linalg.norm(R[:, m]), np.linalg.norm(Xc[:, m])
            floor = 8 * EPS * Hn * xn       # rounding of this host product against the device's
            assert res <= TAU + floor or res <= (1e-13 + 8 * EPS) * Hn * xn, (c, m, res, res / (Hn * xn))
        gate = 2 * tr * np.linalg.norm(R) + 64 * Hn * tr * EPS * np.abs(Sig).max()
        assert np.linalg.norm(X - Sig) <= gate, (c, np.linalg.norm(X - Sig), gate)
        assert np.array_equal(X[c], X[c].T)
    for c in missed:
        pairs = _column_pairs(nf, c)
        with env(S3O_MARGINALS_ROUTE="pcg"):
            with pytest.raises(s3.S3OError, match=rf"error -6: s3o_linsolver_solve_pattern: the PCG solve of column "
                                                  rf"vertex {c} .* after 20000 iterations"):
                ls.marginals(colptr, rowidx, H, pairs)
        assert np.array_equal(ls.marginals(colptr, rowidx, H, pairs)[c], diag[c])      # the direct route, unaffected
    # the NULL form by PCG: n d solves, refused as on a problem
    with env(S3O_MARGINALS_ROUTE="pcg"):
        with pytest.raises(s3.S3OError, match=r"error -5: s3o_linsolver_solve_pattern: "):
            ls.marginals(colptr, rowidx, H)


def _stats(ls):
    from sim3opt_b200 import _lib
    st = _lib.Stats()
    assert ls.L.s3o_get_stats(ls.h, C.byref(st)) == 0
    return st.direct_solves, st.pcg_iterations


# The PCG route takes the two better-conditioned graphs: block-Jacobi does not bring K1 (kappa 1e11) to the tolerance.
@pytest.mark.gpu
@pytest.mark.parametrize("route,graphs", [("direct", ("kitti_k1", "kitti_k118")), ("pcg", ("sphere_small", "manhattan_small"))])
def test_no_side_effects(request, route, graphs):
    """solve -> solve_pattern -> solve gives the x of solve -> solve, bit for bit, with the same statistics, on every
    linear solver; a pattern change between the calls; solve_pattern as the first call on a fresh handle."""
    s3 = _s3()
    systems = []
    for name in graphs:
        p = make_gpu(request.getfixturevalue(name), jac=1)
        H, b = p.linearize()
        colptr, rowidx = p.build_structure()
        systems.append((colptr, rowidx, H, b))
    (cp, ri, H, b), (cp2, ri2, H2, _) = systems
    n, n2 = len(cp) - 1, len(cp2) - 1
    with env(S3O_MARGINALS_ROUTE=route):
        for solver in (s3.LINSOLVER_AUTO, s3.LINSOLVER_DIRECT, s3.LINSOLVER_PCG):
            a, z = s3.LinearSolver(7), s3.LinearSolver(7)
            for ls in (a, z):
                ls.set_linear_solver(solver)
                ls.set_pcg(1e-12, 5000)
            xa0 = a.solve(cp, ri, H, b, 1e-3)
            before = _stats(a)
            a.marginals(cp, ri, H, [(0, 0), (5, n // 2), (n - 1, 3)])
            assert _stats(a) == before, solver
            xa1 = a.solve(cp, ri, H, b, 1e-3)
            xz0, xz1 = z.solve(cp, ri, H, b, 1e-3), z.solve(cp, ri, H, b, 1e-3)
            for u, v in ((xa0, xz0), (xa1, xz1)):
                assert u[0] == v[0] and np.array_equal(u[1], v[1]) and u[2:] == v[2:], solver
            assert _stats(a) == _stats(z), solver
            # pattern change: the second graph's A in between, then the first one's again
            a.marginals(cp2, ri2, H2, [(1, 1), (n2 // 8, 3 * n2 // 4)])
            xa2 = a.solve(cp, ri, H, b, 1e-3)
            fresh = s3.LinearSolver(7)
            fresh.set_linear_solver(solver)
            fresh.set_pcg(1e-12, 5000)
            xf = fresh.solve(cp, ri, H, b, 1e-3)
            assert np.array_equal(xa2[1], xf[1]), solver
    # solve_pattern first on a fresh handle, then a solve: as on a handle that only solves
    a, z = s3.LinearSolver(7), s3.LinearSolver(7)
    first = a.marginals(cp, ri, H)
    assert np.array_equal(a.solve(cp, ri, H, b, 1e-3)[1], z.solve(cp, ri, H, b, 1e-3)[1])
    assert np.array_equal(a.marginals(cp, ri, H), first)


@pytest.mark.gpu
def test_errors(kitti_k1):
    s3 = _s3()
    from sim3opt_b200 import _lib
    p = make_gpu(kitti_k1, jac=1)
    H, b = p.linearize()
    cp, ri = p.build_structure()
    n = len(cp) - 1
    ls = s3.LinearSolver(7)
    x_ref = s3.LinearSolver(7).solve(cp, ri, H, b, 1e-3)[1]
    # not positive definite: one diagonal block negated
    Hbad = H.copy()
    Hbad[cp[300 + 1] - 1] *= -1
    with pytest.raises(s3.S3OError, match=r"error -6: s3o_linsolver_solve_pattern: .*not positive definite"):
        ls.marginals(cp, ri, Hbad)
    assert np.array_equal(ls.solve(cp, ri, H, b, 1e-3)[1], x_ref)
    # malformed CCS: rows of column 1 out of order (the checks and messages of s3o_linsolver_solve)
    ri_bad = ri.copy()
    k = cp[1]
    ri_bad[k:cp[2]] = ri_bad[k:cp[2]][::-1]
    with pytest.raises(s3.S3OError, match=r"error -1: s3o_linsolver_solve_pattern: column 1 is not an upper block-CCS"):
        ls.marginals(cp, ri_bad, H)
    assert np.array_equal(ls.solve(cp, ri, H, b, 1e-3)[1], x_ref)
    for bad in ([[-1, 0]], [[0, n]], [[n + 5, 2]]):
        with pytest.raises(s3.S3OError, match=r"error -1: s3o_linsolver_solve_pattern: pair 0"):
            ls.marginals(cp, ri, H, bad)
    ip = C.POINTER(C.c_int32)
    out = np.zeros((n, 7, 7))
    args = (n, cp.ctypes.data_as(ip), ri.ctypes.data_as(ip), H.ctypes.data_as(C.POINTER(C.c_double)), 0)
    assert ls.L.s3o_linsolver_solve_pattern(ls.h, *args, n - 1, None, None, out.ctypes.data_as(C.POINTER(C.c_double))) == -1
    assert b"n_pairs = n_block_cols" in _lib.load().s3o_last_error()
    assert ls.L.s3o_linsolver_solve_pattern(p.h, *args, n, None, None, out.ctypes.data_as(C.POINTER(C.c_double))) == -1
    # and a handle is still refused by the problem's entry
    rows = np.zeros(1, np.int32)
    assert ls.L.s3o_compute_marginals(ls.h, 1, rows.ctypes.data_as(ip), rows.ctypes.data_as(ip),
                                      out.ctypes.data_as(C.POINTER(C.c_double))) == -5
    assert np.array_equal(ls.solve(cp, ri, H, b, 1e-3)[1], x_ref)


@pytest.mark.gpu
def test_reproducible(sphere_small):
    s3 = _s3()
    p = make_gpu(sphere_small, jac=1)
    H, _ = p.linearize()
    cp, ri = p.build_structure()
    pairs = _pairs(sphere_small, p, len(cp) - 1)
    runs = []
    for _ in range(2):
        ls = s3.LinearSolver(7)
        for _ in range(2):
            runs.append((ls.marginals(cp, ri, H), ls.marginals(cp, ri, H, pairs)))
    assert all(np.array_equal(r[0], runs[0][0]) and np.array_equal(r[1], runs[0][1]) for r in runs)
