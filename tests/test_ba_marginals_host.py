"""CPU tests of the bundle-adjustment marginal covariances (s3o_ba_compute_marginals): a numpy twin of the point phase,
evaluated on the CPU oracle's undamped system, against np.linalg.inv of the dense H.  This pins the index, sign and
transpose conventions the device kernels follow:
    Y_a = Hpl_a Hll^-1,  Z_a = sum_b Sigma_cc(c_a, c_b) Y_b,  Sigma(c_a, l) = -Z_a,  Sigma(l, l) = Hll^-1 + sum_a Y_a^T Z_a
over the observations of a free point by free cameras, with Sigma_cc = S^-1, S = Hpp - Hpl Hll^-1 Hpl^T."""
import os
import subprocess

import numpy as np

from conftest import ROOT
from oracle import oracle as orc
from sim3opt_b200 import synth

HUBER = 1


def ba_fixings(g, cams=(0, 7)):
    """Fixed cameras `cams`, and every point seen by fewer than two distinct cameras (its Hll would be singular)."""
    nc, npts = len(g["cams"]), len(g["points"])
    cf = np.zeros(nc, np.uint8)
    cf[list(cams)] = 1
    seen = np.unique(np.stack([g["obs_pt"], g["obs_cam"]], 1), axis=0)
    pf = (np.bincount(seen[:, 0], minlength=npts) < 2).astype(np.uint8)
    return cf, pf


def random_info(g, seed=3):
    rng = np.random.default_rng(seed)
    n = len(g["uv"])
    return np.stack([rng.uniform(0.5, 2.0, n), rng.uniform(-0.2, 0.2, n), rng.uniform(0.5, 2.0, n)], axis=1)


def hessian_indices(cf, pf):
    """Camera and point Hessian indices (free cameras first, then free points; -1 for fixed vertices)."""
    ncf = int((cf == 0).sum())
    ch, ph = -np.ones(len(cf), int), -np.ones(len(pf), int)
    ch[cf == 0] = np.arange(ncf)
    ph[pf == 0] = ncf + np.arange(int((pf == 0).sum()))
    return ch, ph


def point_observations(g, ch, ph):
    """Free point index li -> observation indices (caller order) by free cameras."""
    keep = (ch[g["obs_cam"]] >= 0) & (ph[g["obs_pt"]] >= 0)
    ks = np.nonzero(keep)[0]
    li = ph[g["obs_pt"][ks]] - int((ch >= 0).sum())
    order = np.argsort(li, kind="stable")
    ks, li = ks[order], li[order]
    npf = int((ph >= 0).sum())
    ptr = np.concatenate([[0], np.cumsum(np.bincount(li, minlength=npf))])
    return [ks[ptr[i]:ptr[i + 1]] for i in range(npf)]


def twin(scc, Hll, Hpl, g, ch, ph, points=None):
    """Point blocks from Sigma_cc: scc(cams) -> the (6n, 6n) matrix of Sigma_cc blocks between the listed free cameras.
    Returns {li: Sigma(l, l)} and {(ci, li): Sigma(c, l)} for the free points `points` (default: all)."""
    obs = point_observations(g, ch, ph)
    pdiag, cl = {}, {}
    for li in (range(len(obs)) if points is None else points):
        Dinv = np.linalg.inv(Hll[li])
        ks = obs[li]
        if len(ks) == 0:
            pdiag[li] = Dinv
            continue
        cams = ch[g["obs_cam"][ks]]
        Y = (Hpl[ks] @ Dinv).reshape(-1, 3)                   # (6n, 3): Y_a stacked
        Z = scc(cams) @ Y
        pdiag[li] = Dinv + Y.T @ Z
        for a, c in enumerate(cams):
            cl.setdefault((int(c), li), -Z[6 * a:6 * a + 6])
    return pdiag, cl


def dense_scc(Sinv):
    def scc(cams):
        idx = (np.asarray(cams)[:, None] * 6 + np.arange(6)).reshape(-1)
        return Sinv[np.ix_(idx, idx)]
    return scc


def dense_schur(colptr, rowidx, S):
    nf = len(colptr) - 1
    A = np.zeros((nf * 6, nf * 6))
    for c in range(nf):
        for k in range(colptr[c], colptr[c + 1]):
            r = rowidx[k]
            A[r * 6:r * 6 + 6, c * 6:c * 6 + 6] = S[k]
            A[c * 6:c * 6 + 6, r * 6:r * 6 + 6] = S[k].T
    return A


def dense_h(Hpp, Hll, Hpl, g, ch, ph):
    ncf, npf = len(Hpp), len(Hll)
    n = 6 * ncf + 3 * npf
    H = np.zeros((n, n))
    for i in range(ncf):
        H[6 * i:6 * i + 6, 6 * i:6 * i + 6] = Hpp[i]
    for li in range(npf):
        o = 6 * ncf + 3 * li
        H[o:o + 3, o:o + 3] = Hll[li]
    for k, (c, l) in enumerate(zip(g["obs_cam"], g["obs_pt"])):
        ci, pi = ch[c], ph[l]
        if ci < 0 or pi < 0:
            continue
        o = 6 * ncf + 3 * (pi - ncf)
        H[6 * ci:6 * ci + 6, o:o + 3] += Hpl[k]
        H[o:o + 3, 6 * ci:6 * ci + 6] += Hpl[k].T
    return H


def oracle_system(g, cf, pf, info):
    o = orc.BAProblem()
    o.set(g["cams"], g["points"], g["obs_cam"], g["obs_pt"], g["uv"], g["focal"], g["cx"], g["cy"],
          cam_fixed=cf, pt_fixed=pf, info=info)
    o.set_robust(HUBER, 2.5)
    colptr, rowidx = o.build_structure()
    Hpp, Hll, Hpl, _ = o.linearize()
    return o, colptr, rowidx, Hpp, Hll, Hpl


def check_against_dense(g, cf, pf, info):
    o, colptr, rowidx, Hpp, Hll, Hpl = oracle_system(g, cf, pf, info)
    ch, ph = hessian_indices(cf, pf)
    ncf, npf = len(Hpp), len(Hll)
    ref = np.linalg.inv(dense_h(Hpp, Hll, Hpl, g, ch, ph))
    scale = np.abs(ref).max()
    if ncf > 0:
        rc, S, _ = o.schur(0.0)
        assert rc == 0
        Sinv = np.linalg.inv(dense_schur(colptr, rowidx, S))
        assert np.abs(Sinv - ref[:6 * ncf, :6 * ncf]).max() <= 1e-10 * scale
    else:
        Sinv = np.zeros((0, 0))
    pdiag, cl = twin(dense_scc(Sinv), Hll, Hpl, g, ch, ph)
    assert len(pdiag) == npf
    for li, B in pdiag.items():
        o3 = 6 * ncf + 3 * li
        assert np.abs(B - ref[o3:o3 + 3, o3:o3 + 3]).max() <= 1e-10 * scale, li
    for (ci, li), B in cl.items():
        o3 = 6 * ncf + 3 * li
        assert np.abs(B - ref[6 * ci:6 * ci + 6, o3:o3 + 3]).max() <= 1e-10 * scale, (ci, li)
    return ncf, npf, len(cl)


def test_twin_matches_dense_inverse():
    g = synth.ba_loop(24, 300, 5, seed=11)
    cf, pf = ba_fixings(g)
    ncf, npf, ncl = check_against_dense(g, cf, pf, random_info(g))
    assert ncf == 22 and npf > 200 and ncl > 2 * npf


def test_twin_all_cameras_fixed():
    g = synth.ba_loop(24, 300, 5, seed=11)
    cf, pf = ba_fixings(g)
    cf[:] = 1
    ncf, npf, ncl = check_against_dense(g, cf, pf, random_info(g))
    assert ncf == 0 and npf > 200 and ncl == 0


def test_ba_marginals_declaration_compiles_as_c(tmp_path):
    src = os.path.join(ROOT, "tests", "cpp", "ba_marginals_snippet.c")
    subprocess.run(["gcc", "-std=c11", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"),
                    "-c", src, "-o", str(tmp_path / "ba_marginals_snippet.o")], check=True)
