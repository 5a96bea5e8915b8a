"""Host reference of the multilevel preconditioner (csrc/amg.cu), piece by piece, and the gates the GPU tests apply.

Every piece is recomputed in numpy with long double accumulation: the transfer frames, the Galerkin operators
A_{k+1} = P_k^T A_k P_k, the smoother inverses, the coarsest inverse and one application z = M^-1 r in each cycle
regime.  tests/test_gpu_multilevel_reference.py compares the device's read-outs (s3o_multilevel_prepare,
s3o_get_multilevel_level, ...) with them one level at a time.  The tests here need no device: they check that each
gate accepts an honest fp64 evaluation and rejects the bugs it is there for by at least 100x, pin the adjoint
convention with the oracle, and check the twin of the regime choice against the host hierarchy.
"""
import numpy as np
import pytest

LD = np.longdouble
U = 2.0 ** -53
OMEGA = 0.7                 # kOmega: damping of the coarse-level block-Jacobi sweeps
COARSEST_MAX, COARSEST_MAX_BIG, BIG_GRAPH = 16, 128, 20000
TAIL_ROWS, COOP_ROWS, COOP_THREADS = 1024, 24000, 512


# ---- twin of the regime choice (amg_setup and apply_t) ---------------------------------------------------------
def ml_plan(level_sizes, n_free, sms, env=None):
    """The cycle a problem takes, from its coarse level sizes (host_multilevel), its free vertices, the SM count and
    the S3O_KCYCLE / S3O_KMASK / S3O_COOP_ROWS switches.  Same keys as Problem.multilevel_prepare."""
    env = env or {}
    n = [int(v) for v in level_sizes]
    nl = len(n)
    if nl == 0:
        return dict(n_levels=0, kdepth=0, kmask=0, coop_first=0, lt=0, dense=0, dense_coop=0, coop_grid=0, grid=0,
                    n=[], G=[])
    dense = n[-1] <= COARSEST_MAX_BIG
    dense_coop = dense and n[-1] > COARSEST_MAX
    kdepth = nl - 1 if (nl >= 2 and n_free >= BIG_GRAPH) else 0
    kmask = (1 << kdepth) - 1
    if kdepth >= 2:
        kmask &= ~1
    if "S3O_KCYCLE" in env:
        kdepth = max(0, min(int(env["S3O_KCYCLE"]), nl - 1))
        kmask = (1 << kdepth) - 1
    if "S3O_KMASK" in env:
        kmask = int(env["S3O_KMASK"], 0) & ((1 << (nl - 1)) - 1)
        kdepth = max([l + 1 for l in range(nl - 1) if (kmask >> l) & 1] or [0])
        if kdepth == 0 and n_free >= BIG_GRAPH:
            kdepth = 1
    coop_rows = int(env.get("S3O_COOP_ROWS", COOP_ROWS))
    coop_first = 0
    while coop_first < nl - 1 and n[coop_first] > coop_rows:
        coop_first += 1
    coop_grid = sms if (kdepth > 0 or dense_coop) else 0
    lt = next((l for l in range(nl) if n[l] <= TAIL_ROWS), nl - 1)
    grid, G = 0, [0] * nl
    if kdepth > 0:
        grid = max(8, min(-(-n[coop_first] * 8 // COOP_THREADS), coop_grid))
        lanes = grid * COOP_THREADS
        G = [0 if l < coop_first else (4 if n[l] * 32 <= lanes else (2 if n[l] * 16 <= lanes else 1)) for l in range(nl)]
    return dict(n_levels=nl, kdepth=kdepth, kmask=kmask, coop_first=coop_first, lt=lt, dense=int(dense),
                dense_coop=int(dense_coop), coop_grid=coop_grid, grid=grid, n=n, G=G)


def regime(plan):
    """One line naming the path the plan takes."""
    if plan["n_levels"] == 0:
        return "no coarse levels: D^-1 r"
    coarsest = ("shared-memory inverse" if plan["dense"] and not plan["dense_coop"] else
                "cooperative inverse" if plan["dense"] else "five damped sweeps (no dense inverse)")
    if plan["kdepth"] == 0:
        above = f"levels 0..{plan['lt'] - 1} by ordinary launches, " if plan["lt"] else ""
        return f"V-cycle, {above}tail kernel from level {plan['lt']}, {coarsest}; levels {plan['n']}"
    return (f"K-cycle mask {plan['kmask']:#x}, cooperative kernel from level {plan['coop_first']} on grid "
            f"{plan['grid']} (G {plan['G']}), {coarsest}; levels {plan['n']}")


# ---- transfer frames ---------------------------------------------------------------------------------------------
def quat_rot(q, normalise):
    """Rotation matrices of quaternions [x y z w] (quat_to_rot); normalise as the device does for Sim3 products."""
    q = np.asarray(q, LD)
    if normalise:
        q = q / np.sqrt((q * q).sum(1, keepdims=True))
    x, y, z, w = q.T
    return np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w),
                     2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w),
                     2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)], 1).reshape(-1, 3, 3)


def frames_ref(d, est, aux, vid, rvid):
    """rel of every fine vertex: S_i S_root^-1 as [R (row-major), t, s] (n, 13), for vertex ids vid (fine) and rvid
    (the root of each one's aggregate).  Sim3: (R_i R_r^T, t_i - (s_i/s_r) R_i R_r^T t_r, s_i/s_r); scale-trans:
    (R_i R_r^T from the fixed rotations, 0, s_i/s_r); scale: (I, 0, s_i/s_r)."""
    est = np.asarray(est, LD)
    n = len(vid)
    rel = np.zeros((n, 13), LD)
    R = np.broadcast_to(np.eye(3, dtype=LD), (n, 3, 3))
    if d == 7:
        Ri, Rr = quat_rot(est[vid, :4], True), quat_rot(est[rvid, :4], True)
        R = Ri @ np.transpose(Rr, (0, 2, 1))
        s = est[vid, 7] / est[rvid, 7]
        rel[:, 9:12] = est[vid, 4:7] - s[:, None] * np.einsum("nij,nj->ni", R, est[rvid, 4:7])
    elif d == 4:
        Ri, Rr = quat_rot(aux[vid], False), quat_rot(aux[rvid], False)
        R = Ri @ np.transpose(Rr, (0, 2, 1))
        s = est[vid, 0] / est[rvid, 0]
    else:
        s = est[vid, 0] / est[rvid, 0]
    rel[:, :9] = R.reshape(n, 9)
    rel[:, 12] = s
    return rel


def frame_error(rel, ref, est, vid, rvid, d):
    """Worst |rel - ref| over the 13 entries, relative to the size of what was computed: 1 for R, |t_i| + s|t_r| for
    t (a relative translation is a difference of two large ones), s for the scale.  About 1e-15 when both agree."""
    rel, ref = np.asarray(rel, LD), np.asarray(ref, LD)
    scale = np.ones_like(ref)
    scale[:, 12] = np.abs(ref[:, 12])
    if d == 7:
        est = np.asarray(est, LD)
        tsz = np.linalg.norm(est[vid, 4:7].astype(float), axis=1) + \
            np.abs(ref[:, 12]).astype(float) * np.linalg.norm(est[rvid, 4:7].astype(float), axis=1)
        scale[:, 9:12] = np.maximum(tsz, 1.0)[:, None]
    return float((np.abs(rel - ref) / scale).max())


def prolongation(rel, d):
    """P_i (n, d, d) of every fine vertex from its frame: Ad(S) = [[R,0,0],[[t]x R, sR, -t],[0,0,1]] (d = 7),
    s diag(1, R) (d = 4), s (d = 1)."""
    rel = np.asarray(rel, LD)
    n = len(rel)
    R, t, s = rel[:, :9].reshape(n, 3, 3), rel[:, 9:12], rel[:, 12]
    if d == 1:
        return s.reshape(n, 1, 1).copy()
    P = np.zeros((n, d, d), LD)
    if d == 4:
        P[:, 0, 0] = s
        P[:, 1:, 1:] = s[:, None, None] * R
        return P
    T = np.zeros((n, 3, 3), LD)
    T[:, 0, 1], T[:, 0, 2], T[:, 1, 2] = -t[:, 2], t[:, 1], -t[:, 0]
    T[:, 1, 0], T[:, 2, 0], T[:, 2, 1] = t[:, 2], -t[:, 1], t[:, 0]
    P[:, :3, :3] = R
    P[:, 3:6, :3] = T @ R
    P[:, 3:6, 3:6] = s[:, None, None] * R
    P[:, 3:6, 6] = -t
    P[:, 6, 6] = 1
    return P


# ---- Galerkin operators --------------------------------------------------------------------------------------------
def full_pattern_from_upper(colptr, rowidx, H, lam):
    """Every block (row, col, B) of H + lam I from its upper block-CCS (s3o_get_hessian)."""
    nf = len(colptr) - 1
    col = np.repeat(np.arange(nf), np.diff(colptr))
    row = np.asarray(rowidx, np.int64)
    off = row != col
    H = np.asarray(H, LD).copy()
    d = H.shape[-1]
    H[~off] += LD(lam) * np.eye(d, dtype=LD)
    return (np.concatenate([row, col[off]]), np.concatenate([col, row[off]]),
            np.concatenate([H, np.transpose(H[off], (0, 2, 1))]))


def bsr_blocks(rowptr, colidx, A):
    rowptr = np.asarray(rowptr)
    return np.repeat(np.arange(len(rowptr) - 1), np.diff(rowptr)), np.asarray(colidx, np.int64), np.asarray(A)


def galerkin_ref(rows, cols, B, agg, P, nc, dtype=LD):
    """P^T A P for the fine operator given by its blocks (rows, cols, B).  Returns (keys, A, env, n): the coarse blocks
    I * nc + J in ascending order (the expected BSR pattern), their values, |P|^T |A| |P|, and the number of products
    summed into every entry (d^2 per contributing fine block)."""
    agg = np.asarray(agg, np.int64)
    key = agg[rows] * nc + agg[cols]
    keys, inv = np.unique(key, return_inverse=True)
    B = np.asarray(B, dtype)
    P = np.asarray(P, dtype)
    d = B.shape[-1]
    out = np.zeros((len(keys), d, d), dtype)
    np.add.at(out, inv, np.einsum("kac,kcm->kam", np.einsum("kba,kbc->kac", P[rows], B), P[cols]))
    if dtype is not LD:
        return keys, out, None, None
    env = np.zeros((len(keys), d, d), LD)
    aP = np.abs(P)
    np.add.at(env, inv, np.einsum("kac,kcm->kam", np.einsum("kba,kbc->kac", aP[rows], np.abs(B)), aP[cols]))
    return keys, out, env, np.bincount(inv, minlength=len(keys))[:, None, None] * d * d


def bound_ratio(err, bound):
    """Worst err / bound (inf where the bound is 0 and the error is not)."""
    err, bound = np.asarray(err, LD), np.asarray(bound, LD)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(bound > 0, err / bound, np.where(err > 0, np.inf, 0.0))
    return float(r.max())


def galerkin_error(A, ref):
    """Worst |A - A_ref| / (2 n u |P|^T |A| |P|): at most 1 for the product summed in any order in fp64."""
    _, Aref, env, n = ref
    return bound_ratio(np.abs(np.asarray(A, LD) - Aref), 2 * n * U * env)


def mass_ref(agg, P, Mf, nc):
    """M = P^T Mf P (block diagonal: one nonzero block per row of P); Mf None: identity."""
    P = np.asarray(P, LD)
    X = np.einsum("kba,kbc->kac", P, P) if Mf is None else np.einsum("kba,kbm,kmc->kac", P, np.asarray(Mf, LD), P)
    M = np.zeros((nc,) + X.shape[1:], LD)
    np.add.at(M, np.asarray(agg, np.int64), X)
    return M


# ---- smoother and coarsest inverses --------------------------------------------------------------------------------
def inverse_residual(B, X):
    """(|B X - I|_2, kappa_2(B)) per block of a stack (or of one matrix)."""
    B, X = np.asarray(B, float), np.asarray(X, float)
    Rm = np.asarray(B, LD) @ np.asarray(X, LD) - np.eye(B.shape[-1], dtype=LD)
    return np.linalg.norm(Rm.astype(float), 2, axis=(-2, -1)), np.linalg.cond(B)


def inverse_error(B, X, c=10):
    """Worst |B X - I|_2 / (c d u kappa(B)): at most 1 for a backward-stable inverse of a matrix of order d."""
    res, kap = inverse_residual(B, X)
    return float(np.max(res / (c * np.asarray(B).shape[-1] * U * kap)))


def dense_of(rowptr, colidx, A):
    rows, cols, A = bsr_blocks(rowptr, colidx, A)
    n, d = len(rowptr) - 1, A.shape[-1]
    out = np.zeros((n, d, n, d))
    out[rows, :, cols, :] = A
    return out.reshape(n * d, n * d)


# ---- one application z = M^-1 r -------------------------------------------------------------------------------------
class Hierarchy:
    """Operators of a hierarchy as the device holds them: fine block-Jacobi inverses Minv (nf, d, d), and per coarse
    level k its transfer (agg, P from the fine level) and operator (rowptr, colidx, A, Dinv); inv: dense inverse of
    the coarsest level or None.  apply() runs the cycle of plan (ml_plan keys kdepth, kmask) in long double;
    with envelope=True it runs it on absolute values with every subtraction made an addition (the rounding
    envelope of the V-cycle)."""

    def __init__(self, Minv, levels, inv, plan, omega=OMEGA, sweeps=5):
        self.Minv, self.levels, self.inv, self.plan = Minv, levels, inv, plan
        self.omega, self.sweeps = omega, sweeps
        self.omega_at = {}          # (level, sweep) -> damping, for the self-tests' bugs

    def _mv(self, L, x, env):
        y = np.zeros_like(x)
        np.add.at(y, L["rows"], np.einsum("kij,kj->ki", L["aA"] if env else L["A"], x[L["colidx"]]))
        return y

    def _jac(self, L, r, env, k, sweep):
        om = LD(self.omega_at.get((k, sweep), self.omega))
        return om * np.einsum("nij,nj->ni", L["aDinv"] if env else L["Dinv"], r)

    def _sub(self, a, b, env):
        return a + b if env else a - b

    def _restrict(self, L, t, env):
        rc = np.zeros((L["n"], t.shape[1]), LD)
        np.add.at(rc, L["agg"], np.einsum("nji,nj->ni", L["aP"] if env else L["P"], t))
        return rc

    def _prolong(self, L, xc, env):
        return np.einsum("nij,nj->ni", L["aP"] if env else L["P"], xc[L["agg"]])

    def vcycle(self, k, r, env):
        L = self.levels[k]
        if k == len(self.levels) - 1:
            if self.inv is not None:
                inv = np.abs(self.inv) if env else self.inv
                return (inv @ r.reshape(-1)).reshape(r.shape)
            x = self._jac(L, r, env, k, 0)
            for s in range(1, self.sweeps):
                x = x + self._jac(L, self._sub(r, self._mv(L, x, env), env), env, k, s)
            return x
        x = self._jac(L, r, env, k, 0)
        t = self._sub(r, self._mv(L, x, env), env)
        x = x + self._prolong(self.levels[k + 1], self.solve(k + 1, self._restrict(self.levels[k + 1], t, env), env), env)
        return x + self._jac(L, self._sub(r, self._mv(L, x, env), env), env, k, 1)

    def solve(self, k, r, env):
        p = self.plan
        if p["kdepth"] > 0 and (p["kmask"] >> k) & 1 and k < len(self.levels) - 1:
            assert not env, "a K-cycle level has no rounding envelope"
            L = self.levels[k]
            z1 = self.vcycle(k, r, False)
            q1 = self._mv(L, z1, False)
            ks = kstep_first((z1 * q1).sum(), (z1 * r).sum())
            rp = r - ks["alpha1"] * q1
            z2 = self.vcycle(k, rp, False)
            q2 = self._mv(L, z2, False)
            kstep_second(ks, (z2 * q2).sum(), (z2 * rp).sum(), (z2 * q1).sum())
            return ks["c1"] * z1 + ks["c2"] * z2
        return self.vcycle(k, r, env)

    def apply(self, r, envelope=False):
        d = self.Minv.shape[-1]
        r = np.asarray(r, LD).reshape(-1, d)
        if envelope:
            r = np.abs(r)
        Minv = np.abs(self.Minv) if envelope else self.Minv
        z = np.einsum("nij,nj->ni", Minv, r)
        if self.levels:
            L0 = self.levels[0]
            z = z + self._prolong(L0, self.solve(0, self._restrict(L0, r, envelope), envelope), envelope)
        return z.reshape(-1)

    def terms(self):
        """Fixed constant of the V-cycle gate: 2 x (longest sum in any one step) x (steps on the longest path)."""
        d = self.Minv.shape[-1]
        longest = [d + 1]
        for L in self.levels:
            longest += [int(np.diff(L["rowptr"]).max()) * d + 1, int(np.bincount(L["agg"]).max()) * d]
        if self.inv is not None:
            longest.append(self.inv.shape[0])
        return 2 * max(longest) * (6 * len(self.levels) + 2 * self.sweeps + 4)


def make_level(agg, P, rowptr, colidx, A, Dinv):
    L = dict(agg=np.asarray(agg, np.int64), P=np.asarray(P, LD), rowptr=np.asarray(rowptr),
             colidx=np.asarray(colidx, np.int64), A=np.asarray(A, LD), Dinv=np.asarray(Dinv, LD))
    L["n"] = len(L["rowptr"]) - 1
    L["rows"] = np.repeat(np.arange(L["n"]), np.diff(L["rowptr"]))
    L["aP"], L["aA"], L["aDinv"] = np.abs(L["P"]), np.abs(L["A"]), np.abs(L["Dinv"])
    return L


def kstep_first(zq, zr):
    """kscal_first: the first inner step's scalars, guarded against zq <= 0."""
    ok = zq > 0 and np.isfinite(float(zq))
    return dict(rho1=zq if ok else LD(1), alpha1=zr / zq if ok else LD(0), c1=zr / zq if ok else LD(0), c2=LD(0))


def kstep_second(ks, beta, alpha2, gamma, guard=True):
    """kscal_second: coefficients of x = c1 z1 + c2 z2; with rho2 <= 0 (or not finite) the one-step result."""
    rho2 = beta - gamma * gamma / ks["rho1"]
    if not guard or (rho2 > 0 and np.isfinite(float(rho2))):
        with np.errstate(divide="ignore", invalid="ignore"):
            ks["c1"] = ks["alpha1"] - alpha2 * gamma / (ks["rho1"] * rho2)
            ks["c2"] = alpha2 / rho2
    else:
        ks["c1"], ks["c2"] = ks["alpha1"], LD(0)
    return ks


def vcycle_error(z, zref, env, terms):
    """Worst |z - z_ref| / (terms u envelope): at most 1 for the V-cycle evaluated in fp64."""
    return bound_ratio(np.abs(np.asarray(z, LD) - zref), terms * U * env)


def kcycle_error(z, zref):
    """Relative 2-norm difference: the K-cycle's coefficients divide by dot products, so no componentwise envelope."""
    zref = np.asarray(zref, LD)
    return float(np.linalg.norm((np.asarray(z, LD) - zref).astype(float)) / np.linalg.norm(zref.astype(float)))


KCYCLE_TOL = 1e-10
FRAME_TOL = 2e-14           # frame_error of the device's frames (fp64 products of a few terms)


# =====================================================================================================================
# CPU tests
# =====================================================================================================================
def _random_sim3(rng, n):
    from scipy.spatial.transform import Rotation
    q = Rotation.random(n, random_state=rng.integers(1 << 31)).as_quat()
    t = rng.normal(scale=20.0, size=(n, 3))
    s = np.exp(rng.normal(scale=0.3, size=n))
    return np.concatenate([q, t, s[:, None]], 1)


def test_adjoint_convention_against_oracle():
    """P_i = Ad(S_i S_r^-1) with the oracle's conventions: exp(Ad(S) v) S == S exp(v), and the frame built here equals
    orc.sim3_adjoint(orc.sim3_mul(S_i, orc.sim3_inv(S_r)))."""
    from oracle import oracle as orc
    rng = np.random.default_rng(3)
    est = _random_sim3(rng, 12)
    vid, rvid = np.arange(12), np.array([0, 0, 0, 3, 3, 5, 5, 5, 5, 9, 9, 9])
    P = prolongation(frames_ref(7, est, None, vid, rvid), 7).astype(float)
    for i in range(12):
        S = orc.sim3_mul(est[vid[i]], orc.sim3_inv(est[rvid[i]]))
        assert np.abs(P[i] - orc.sim3_adjoint(S)).max() <= 1e-12 * max(1.0, np.abs(P[i]).max())
        Sq = S[:4] / np.linalg.norm(S[:4])
        Ad = prolongation(np.concatenate([orc.quat_to_rot(Sq).reshape(9), S[4:7], S[7:8]])[None], 7)[0].astype(float)
        v = rng.normal(scale=0.1, size=7)
        lhs = orc.sim3_mul(orc.sim3_exp(Ad @ v), S)
        rhs = orc.sim3_mul(S, orc.sim3_exp(v))
        assert np.abs(orc.quat_to_rot(lhs[:4]) - orc.quat_to_rot(rhs[:4])).max() <= 1e-12
        assert np.abs(lhs[4:] - rhs[4:]).max() <= 1e-11 * max(1.0, np.abs(rhs[4:]).max())


def _toy(d=7, seed=0, nf=60, agg_size=3, lam=1e-3):
    """A chain of nf poses with second-neighbour blocks, aggregates of agg_size consecutive poses, a second level of
    pairs of aggregates: the operators of a real hierarchy, built here in long double."""
    rng = np.random.default_rng(seed)
    est = _random_sim3(rng, nf)
    if d == 4:
        est_k, aux = np.concatenate([est[:, 7:8], est[:, 4:7]], 1), est[:, :4]
    elif d == 1:
        est_k, aux = est[:, 7:8], None
    else:
        est_k, aux = est, None
    row = np.concatenate([np.arange(nf), np.arange(nf - 1), np.arange(nf - 2)])
    col = np.concatenate([np.arange(nf), np.arange(1, nf), np.arange(2, nf)])
    order = np.lexsort((row, col))
    row, col = row[order], col[order]
    colptr = np.concatenate([[0], np.cumsum(np.bincount(col, minlength=nf))])
    H = rng.normal(size=(len(row), d, d))
    diag = row == col
    H[diag] = np.einsum("kij,klj->kil", H[diag], H[diag]) + 6 * d * np.eye(d)
    rows, cols, B = full_pattern_from_upper(colptr, row, H, lam)
    agg = np.arange(nf) // agg_size
    nc = agg.max() + 1
    rvid = agg * agg_size
    rel = frames_ref(d, est_k, aux, np.arange(nf), rvid)
    P = prolongation(rel, d)
    keys, A1, env, n = galerkin_ref(rows, cols, B, agg, P, nc)
    return dict(d=d, est=est_k, aux=aux, rvid=rvid, rows=rows, cols=cols, B=B, agg=agg, nc=nc, rel=rel, P=P, keys=keys,
                A1=A1, ref=(keys, A1, env, n), colptr=colptr, rowidx=row, H=H, lam=lam)


@pytest.mark.parametrize("d", [7, 4, 1])
def test_frame_and_galerkin_gates(d):
    t = _toy(d)
    nf = len(t["agg"])
    assert frame_error(t["rel"].astype(float), t["rel"], t["est"], np.arange(nf), t["rvid"], d) <= 1e-15
    # an honest fp64 product (other order, fp64 frames) passes
    P64 = prolongation(t["rel"].astype(float), d).astype(float)
    _, A64, _, _ = galerkin_ref(t["rows"][::-1], t["cols"][::-1], t["B"][::-1].astype(float), t["agg"], P64, t["nc"],
                                dtype=np.float64)
    assert galerkin_error(A64, t["ref"]) <= 1.0
    keys = t["keys"]
    nc = t["nc"]
    I, J = keys // nc, keys % nc
    # a transposed coarse off-diagonal block
    bad = A64.copy()
    k = int(np.flatnonzero(I != J)[0])
    bad[k] = bad[k].T
    if d > 1:
        assert galerkin_error(bad, t["ref"]) >= 100
    # a dropped contributor
    drop = np.ones(len(t["rows"]), bool)
    drop[int(np.flatnonzero(t["rows"] != t["cols"])[3])] = False
    _, Ad, _, _ = galerkin_ref(t["rows"][drop], t["cols"][drop], t["B"][drop], t["agg"], t["P"], nc)
    assert galerkin_error(Ad.astype(float), t["ref"]) >= 100
    # ... and the mirror of a coarse block is its exact transpose
    pos = np.searchsorted(keys, J * nc + I)
    assert np.array_equal(keys[pos], J * nc + I)
    if d == 7:
        # a flipped translation sign in one frame: caught by the frame gate and by the Galerkin gate
        rel = t["rel"].copy()
        i = 4
        rel[i, 9:12] = -rel[i, 9:12]
        assert frame_error(rel, t["rel"], t["est"], np.arange(nf), t["rvid"], d) >= 100 * FRAME_TOL
        _, Af, _, _ = galerkin_ref(t["rows"], t["cols"], t["B"], t["agg"], prolongation(rel, d), nc)
        assert galerkin_error(Af.astype(float), t["ref"]) >= 100


def _toy_hierarchy(d=7, dense=True, seed=1):
    t = _toy(d, seed=seed, nf=90, lam=1e-2)
    nc = t["nc"]
    rowptr = np.searchsorted(t["keys"] // nc, np.arange(nc + 1))
    A1 = t["A1"]
    diag1 = t["keys"] // nc == t["keys"] % nc
    Dinv1 = np.linalg.inv(A1[diag1].astype(float))
    agg2 = np.arange(nc) // 3
    nc2 = agg2.max() + 1
    rng = np.random.default_rng(seed + 7)
    rel2 = frames_ref(7, _random_sim3(rng, nc), None, np.arange(nc), agg2 * 3)
    if d != 7:
        rel2[:, :12] = np.concatenate([np.eye(3).reshape(9), np.zeros(3)])
    P2 = prolongation(rel2, d)
    rows, cols, B = bsr_blocks(rowptr, t["keys"] % nc, A1)
    keys2, A2, _, _ = galerkin_ref(rows, cols, B, agg2, P2, nc2)
    rowptr2 = np.searchsorted(keys2 // nc2, np.arange(nc2 + 1))
    diag2 = keys2 // nc2 == keys2 % nc2
    Dinv2 = np.linalg.inv(A2[diag2].astype(float))
    inv = np.linalg.inv(dense_of(rowptr2, keys2 % nc2, A2.astype(float))) if dense else None
    diag0 = t["rows"] == t["cols"]
    Minv = np.linalg.inv(t["B"][diag0].astype(float))
    levels = [make_level(t["agg"], t["P"], rowptr, t["keys"] % nc, A1, Dinv1),
              make_level(agg2, P2, rowptr2, keys2 % nc2, A2, Dinv2)]
    return Minv, levels, inv


@pytest.mark.parametrize("dense", [True, False])
def test_cycle_gates(dense):
    """The V-cycle gate accepts the cycle evaluated in fp64 and rejects omega = 0.75 in one sweep and, without a dense
    coarsest inverse, four sweeps instead of five."""
    Minv, levels, inv = _toy_hierarchy(dense=dense)
    plan = dict(kdepth=0, kmask=0)
    h = Hierarchy(Minv, levels, inv, plan)
    rng = np.random.default_rng(5)
    r = rng.normal(size=Minv.shape[0] * 7)
    zref, env = h.apply(r), h.apply(r, envelope=True)
    terms = h.terms()
    # honest fp64: the same cycle with every operand rounded to fp64 and fp64 arithmetic
    h64 = Hierarchy(Minv, [dict(L, **{k: L[k].astype(float) for k in ("P", "A", "Dinv", "aP", "aA", "aDinv")})
                           for L in levels], inv, plan)
    with np.errstate(all="ignore"):
        z64 = _apply_fp64(h64, r)
    assert vcycle_error(z64, zref, env, terms) <= 1.0
    for k in range(len(levels) - (1 if dense else 0)):      # a dense coarsest level has no sweep
        hb = Hierarchy(Minv, levels, inv, plan)
        hb.omega_at[(k, 1)] = 0.75
        assert vcycle_error(hb.apply(r), zref, env, terms) >= 100, k
    if not dense:
        assert vcycle_error(Hierarchy(Minv, levels, inv, plan, sweeps=4).apply(r), zref, env, terms) >= 100
    # K-cycle on level 0: the relative gate rejects omega = 0.75 in one sweep as well
    pk = dict(kdepth=1, kmask=1)
    zk = Hierarchy(Minv, levels, inv, pk).apply(r)
    hb = Hierarchy(Minv, levels, inv, pk)
    hb.omega_at[(0, 0)] = 0.75
    assert kcycle_error(hb.apply(r), zk) >= 100 * KCYCLE_TOL


def _apply_fp64(h, r):
    """Hierarchy.apply with fp64 operands and arithmetic (the long double class with its dtype swapped)."""
    global LD
    saved = LD
    LD = np.float64
    try:
        return h.apply(r)
    finally:
        LD = saved


def test_kcycle_guard():
    """kscal_second keeps the one-step result when rho2 = beta - gamma^2 / rho1 is not positive: an unguarded step
    differs from it by far more than the K-cycle tolerance."""
    rng = np.random.default_rng(9)
    z1, z2 = rng.normal(size=50), rng.normal(size=50)
    ks = kstep_first(LD(2.0), LD(0.5))
    guarded = kstep_second(dict(ks), LD(1.0), LD(0.3), LD(1.5))          # rho2 = 1 - 2.25 / 2 < 0
    unguarded = kstep_second(dict(ks), LD(1.0), LD(0.3), LD(1.5), guard=False)
    zg = guarded["c1"] * z1 + guarded["c2"] * z2
    zu = unguarded["c1"] * z1 + unguarded["c2"] * z2
    assert guarded["c2"] == 0 and guarded["c1"] == ks["alpha1"]
    assert kcycle_error(zu, zg) >= 100 * KCYCLE_TOL
    # first step: zq <= 0 gives alpha1 = 0
    assert kstep_first(LD(-1.0), LD(1.0))["alpha1"] == 0


def test_inverse_gates():
    rng = np.random.default_rng(2)
    X = rng.normal(size=(40, 7, 7))
    B = np.einsum("kij,klj->kil", X, X) + 1e-3 * np.eye(7)
    Bi = np.linalg.inv(B)
    assert inverse_error(B, Bi) <= 1.0
    Bi[3, 2, 5] *= 1 + 1e-6
    assert inverse_error(B, Bi) >= 100


def chains(n_chains, length, seed=0):
    """n_chains disconnected odometry chains of `length` poses, the first pose of each fixed: aggregation stalls at one
    vertex per chain, which gives coarsest levels too large for the dense inverse on purpose."""
    from sim3opt_b200 import synth
    g = synth.sphere(n_laps=1, poses_per_lap=n_chains * length, seed=seed)
    v0, v1 = g["v0"], g["v1"]
    keep = (v1 - v0 == 1) & (v1 % length != 0)
    fixed = (np.arange(n_chains * length) % length == 0).astype(np.uint8)
    return dict(est=g["est"], fixed=fixed, v0=v0[keep], v1=v1[keep], meas=g["meas"][keep], info=g["info"][keep])


TWIN_CASES = [
    # graph, expected coarse level sizes (host_multilevel on this tree)
    ("chains_40x50", [680, 240, 80, 40]),
    ("chains_200x50", [3400, 1200, 400, 200]),
    ("chains_300x80", [8100, 2700, 900, 300]),
    ("sphere_10x300", [240, 40, 7]),
]


def twin_graph(name):
    from sim3opt_b200 import synth
    if name.startswith("chains"):
        a, b = name.split("_")[1].split("x")
        return chains(int(a), int(b))
    a, b = name.split("_")[1].split("x")
    return synth.sphere(int(a), int(b), seed=11)


@pytest.mark.parametrize("name,sizes", TWIN_CASES)
def test_twin_levels(name, sizes):
    """The regime twin works from host_multilevel's levels; the graphs of the GPU cases have the levels they are
    chosen for."""
    import sim3opt_b200 as s3
    g = twin_graph(name)
    lv, _, _ = s3.host_multilevel(len(g["est"]), g["fixed"], g["v0"], g["v1"])
    assert list(lv) == sizes
    nf = int((g["fixed"] == 0).sum())
    plan = ml_plan(lv, nf, 148)
    if name == "chains_300x80":         # large graph, coarsest without inverse, G = 1, 2, 4 on one grid
        assert nf == 23700 and plan["kdepth"] == 3 and plan["kmask"] == 6 and not plan["dense"]
        assert plan["grid"] == 127 and plan["G"] == [1, 2, 4, 4]
    if name == "chains_200x50":
        assert nf == 9800 and plan["kdepth"] == 0 and plan["lt"] == 2 and not plan["dense"]
    if name == "chains_40x50":
        assert plan["kdepth"] == 0 and plan["lt"] == 0 and plan["dense_coop"]


def test_twin_switches():
    sizes, nf = [2004, 265, 44], 29999
    p = ml_plan(sizes, nf, 148)
    assert (p["kdepth"], p["kmask"], p["coop_first"], p["dense_coop"], p["grid"], p["G"]) == (2, 2, 0, 1, 32, [1, 4, 4])
    p = ml_plan(sizes, nf, 148, {"S3O_KCYCLE": "0"})
    assert (p["kdepth"], p["lt"], p["dense_coop"]) == (0, 1, 1)
    p = ml_plan(sizes, nf, 148, {"S3O_KMASK": "3", "S3O_COOP_ROWS": "1000"})
    assert (p["kdepth"], p["kmask"], p["coop_first"], p["G"]) == (2, 3, 1, [0, 1, 4])
    p = ml_plan([240, 40, 7], 2999, 148, {"S3O_KCYCLE": "2"})
    assert (p["kdepth"], p["kmask"], p["coop_first"], p["dense"], p["dense_coop"]) == (2, 3, 0, 1, 0)
    assert ml_plan([], 11, 148)["n_levels"] == 0
