"""CPU tests of the marginal covariances' schedule (s3o_compute_marginals, csrc/direct.cu selinv_kernel): a numpy twin of
the selected inverse (Takahashi recurrences, rounds of the DIRECT plan in reverse, off-diagonal blocks before diagonal
blocks) on the plan of api.host_direct_plan, checked against np.linalg.inv, and the two facts the kernel's schedule
relies on."""
import os
import subprocess

import numpy as np

import sim3opt_b200 as s3
from conftest import ROOT
from test_direct_host import bsr_upper


def plan_of(g):
    nv = len(g["est"])
    fixed = np.asarray(g["fixed"], np.uint8)
    plan = s3.host_direct_plan(nv, fixed, g["v0"], g["v1"], max_pairs=60000000)
    hidx = -np.ones(nv, int)
    hidx[fixed == 0] = np.arange(int((fixed == 0).sum()))
    return plan, hidx


def pattern(plan):
    """bcol of every block, round of every column, and (row, col) -> block index of L (elimination positions)."""
    n, cptr, brow = plan["n"], plan["cptr"], plan["brow"]
    bcol = np.repeat(np.arange(n), np.diff(cptr))
    rnd = np.repeat(np.arange(plan["rounds"]), np.diff(plan["lev_ptr"]))
    where = {(int(brow[t]), int(bcol[t])): t for t in range(len(brow))}
    return bcol, rnd, where


def spd_with_pattern(nf, blocks, d, seed):
    rng = np.random.default_rng(seed)
    A = np.zeros((nf * d, nf * d))
    for r, c in blocks:
        B = rng.standard_normal((d, d))
        if r == c:
            A[r * d:(r + 1) * d, r * d:(r + 1) * d] = B @ B.T + 4 * len(blocks) / nf * d * np.eye(d)
        else:
            A[r * d:(r + 1) * d, c * d:(c + 1) * d] = B
            A[c * d:(c + 1) * d, r * d:(r + 1) * d] = B.T
    return A


def selinv_twin(plan, Lfull, d):
    """Sigma on the pattern of L from the block factor Lfull (elimination order), the way selinv_kernel computes it."""
    n, cptr, brow, lp = plan["n"], plan["cptr"], plan["brow"], plan["lev_ptr"]
    bcol, rnd, where = pattern(plan)
    blk = lambda M, i, j: M[i * d:(i + 1) * d, j * d:(j + 1) * d]
    Linv = [np.linalg.inv(blk(Lfull, j, j)) for j in range(n)]
    Sig = np.zeros((len(brow), d, d))
    done = np.zeros(len(brow), bool)

    def sigma(i, k):                      # Sigma_ik from its stored block (max, min)
        t = where[(max(i, k), min(i, k))]
        assert done[t], "an operand is read before it is written"
        return Sig[t].T if i < k else Sig[t]

    for lev in range(plan["rounds"] - 1, -1, -1):
        cols = range(lp[lev], lp[lev + 1])
        for j in cols:                    # phase 1: off-diagonal blocks
            S = brow[cptr[j] + 1:cptr[j + 1]]
            for t in range(cptr[j] + 1, cptr[j + 1]):
                acc = sum((sigma(brow[t], k) @ blk(Lfull, k, j) for k in S), np.zeros((d, d)))
                Sig[t] = -acc @ Linv[j]
        for j in cols:
            done[cptr[j] + 1:cptr[j + 1]] = True
        for j in cols:                    # phase 2: diagonal blocks
            W = Linv[j].copy()
            for t in range(cptr[j] + 1, cptr[j + 1]):
                W -= blk(Lfull, brow[t], j).T @ Sig[t]
            D = Linv[j].T @ W
            Sig[cptr[j]] = np.tril(D) + np.tril(D, -1).T          # one triangle, mirrored
            done[cptr[j]] = True
    return Sig


def check_graph(g, d, seed=0):
    plan, hidx = plan_of(g)
    nf = plan["n"]
    A = spd_with_pattern(nf, bsr_upper(nf, hidx, g["v0"], g["v1"]), d, seed)
    perm = plan["perm"]
    idx = (perm[:, None] * d + np.arange(d)).reshape(-1)       # elimination order -> scalar rows of A
    Lfull = np.linalg.cholesky(A[np.ix_(idx, idx)])
    Sig = selinv_twin(plan, Lfull, d)
    ref = np.linalg.inv(A)
    bcol, _, _ = pattern(plan)
    scale = np.abs(ref).max()
    for t in range(len(plan["brow"])):
        i, j = perm[plan["brow"][t]], perm[bcol[t]]                # Hessian indices of the block
        assert np.abs(Sig[t] - ref[i * d:(i + 1) * d, j * d:(j + 1) * d]).max() <= 1e-10 * scale, t
    for j in range(nf):
        D = Sig[plan["cptr"][j]]
        assert np.array_equal(D, D.T)
    return plan


def test_selected_inverse_twin_matches_dense_inverse(kitti_k1, kitti_k118, sphere_small, manhattan_small):
    check_graph(kitti_k1, d=3)
    check_graph(kitti_k118, d=3)
    check_graph(sphere_small, d=2)
    check_graph(manhattan_small, d=2)


def test_schedule_facts(kitti_k1, kitti_k118, sphere_small, manhattan_small):
    """Every (max, min) pair of S(j) is a block of L (S(j) is a clique of the filled graph), and every Sigma operand of
    column j belongs to a strictly later round than j -- so the rounds can run in reverse, one writer per block."""
    for g in (kitti_k1, kitti_k118, sphere_small, manhattan_small):
        plan, _ = plan_of(g)
        cptr, brow = plan["cptr"], plan["brow"]
        _, rnd, where = pattern(plan)
        products = 0
        for j in range(plan["n"]):
            S = [int(k) for k in brow[cptr[j] + 1:cptr[j + 1]]]
            products += len(S) * len(S) + len(S)
            for i in S:
                for k in S:
                    t = where.get((max(i, k), min(i, k)))
                    assert t is not None, (j, i, k)
                    assert rnd[max(i, k)] > rnd[j] and rnd[min(i, k)] > rnd[j]
        assert products == 2 * plan["n_pairs"]          # the selected inverse costs twice the factor's products


def test_marginals_declaration_compiles_as_c(tmp_path):
    src = os.path.join(ROOT, "tests", "cpp", "marginals_snippet.c")
    subprocess.run(["gcc", "-std=c11", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"),
                    "-c", src, "-o", str(tmp_path / "marginals_snippet.o")], check=True)
