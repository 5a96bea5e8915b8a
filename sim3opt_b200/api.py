"""Thin Python mirror of the C ABI (include/sim3opt_b200.h) used by tests and bench.py.

Every method is one C call; no arithmetic happens in Python.  The object plays the role of
g2o::SparseOptimizer + OptimizationAlgorithmLevenberg for one graph (kitti_surf.cpp:552-558).
"""
import ctypes as C

import numpy as np

from . import _lib

KIND_SIM3, KIND_SCALE_TRANS, KIND_SCALE, KIND_BA = 0, 1, 2, 3
JAC_NUMERIC, JAC_ANALYTIC = 0, 1
MATH_REFERENCE, MATH_CORRECTED = 0, 1
PRECOND_AUTO, PRECOND_BLOCK_JACOBI, PRECOND_MULTILEVEL = 0, 1, 2
LINSOLVER_AUTO, LINSOLVER_PCG, LINSOLVER_DIRECT = 0, 1, 2
SCALE_MODEL_DIFFERENCE, SCALE_MODEL_LOGRATIO = 0, 1
ROBUST_NONE, ROBUST_HUBER, ROBUST_PTAM_TUKEY, ROBUST_PTAM_CAUCHY, ROBUST_PTAM_HUBER, ROBUST_PTAM_LS = range(6)

_EST_DIM = {KIND_SIM3: 8, KIND_SCALE_TRANS: 4, KIND_SCALE: 1, KIND_BA: 7}
_DIM = {KIND_SIM3: 7, KIND_SCALE_TRANS: 4, KIND_SCALE: 1, KIND_BA: 6}

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)
_up = C.POINTER(C.c_uint8)


class S3OError(RuntimeError):
    pass


def _d(a):
    return a.ctypes.data_as(_dp)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


class Problem:
    def __init__(self, kind=KIND_SIM3, device=0, stream=None):
        self.L = _lib.load()
        self.kind = kind
        if kind not in _DIM:
            raise S3OError(f"unsupported kind {kind}")
        self.d = _DIM[kind]
        self.est_dim = _EST_DIM[kind]
        h = C.c_void_p()
        self._check(self.L.s3o_create(kind, device, C.byref(h)))
        self.h = h
        self.nv = self.ne = 0
        if stream is not None:
            self.set_stream(stream)

    def _check(self, rc):
        if rc != 0:
            raise S3OError(f"s3o error {rc}: {self.L.s3o_last_error().decode()}")

    def close(self):
        if getattr(self, "h", None):
            self.L.s3o_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_comm(self, rank, world, unique_id):
        """Partitioned solve: call before set_edges on every rank with the id rank 0 generated."""
        self._check(self.L.s3o_set_comm(self.h, int(rank), int(world), bytes(unique_id) if unique_id else None))

    def set_stream(self, cuda_stream_handle):
        self._check(self.L.s3o_set_stream(self.h, C.c_void_p(int(cuda_stream_handle) if cuda_stream_handle else None)))

    # ---- graph -------------------------------------------------------------------
    def set_vertices(self, est, fixed=None, aux=None):
        est = _f64(est).reshape(-1, self.est_dim)
        self.nv = est.shape[0]
        fx = np.zeros(self.nv, np.uint8) if fixed is None else np.ascontiguousarray(fixed, np.uint8)
        auxp = None
        if aux is not None:
            aux = _f64(aux).reshape(self.nv, 4)
            auxp = _d(aux)
        self._check(self.L.s3o_set_vertices(self.h, self.nv, _d(est), fx.ctypes.data_as(_up), auxp))

    def set_edges(self, v0, v1, meas, info=None):
        v0 = np.ascontiguousarray(v0, np.int32)
        v1 = np.ascontiguousarray(v1, np.int32)
        meas = _f64(meas).reshape(-1, self.est_dim)
        self.ne = len(v0)
        infop = None
        if info is not None:
            info = _f64(info).reshape(self.ne, self.d, self.d)
            infop = _d(info)
        self._check(self.L.s3o_set_edges(self.h, self.ne, v0.ctypes.data_as(_ip), v1.ctypes.data_as(_ip), _d(meas), infop))

    def set_estimates(self, est):
        est = _f64(est).reshape(self.nv, self.est_dim)
        self._check(self.L.s3o_set_estimates(self.h, _d(est)))

    # ---- sharded host round trip of the estimates in the partitioned solve (s3o_*_slice)
    def estimate_slice(self):
        first, count = C.c_int(0), C.c_int(0)
        self._check(self.L.s3o_estimate_slice(self.h, C.byref(first), C.byref(count)))
        return first.value, count.value

    def set_estimates_slice(self, est_slice):
        """Collective: this rank's slice (estimate_slice()) of the caller-ordered estimates, C-contiguous float64."""
        assert est_slice.dtype == np.float64 and est_slice.flags["C_CONTIGUOUS"]
        self._check(self.L.s3o_set_estimates_slice(self.h, _d(est_slice)))

    def vertices_slice(self, out):
        assert out.dtype == np.float64 and out.flags["C_CONTIGUOUS"]
        self._check(self.L.s3o_get_vertices_slice(self.h, _d(out)))
        return out

    def set_robust(self, kind, param=0.0): self._check(self.L.s3o_set_robust(self.h, kind, float(param)))
    def set_jacobian_mode(self, mode, h=0.0): self._check(self.L.s3o_set_jacobian_mode(self.h, mode, float(h)))
    def set_math_mode(self, mode): self._check(self.L.s3o_set_math_mode(self.h, int(mode)))
    def set_scale_model(self, model): self._check(self.L.s3o_set_scale_model(self.h, int(model)))
    def set_lm(self, tau=0.0, lambda_init=0.0, max_trials=0): self._check(self.L.s3o_set_lm(self.h, tau, lambda_init, max_trials))
    def set_pcg(self, rel_tol=0.0, max_iter=0): self._check(self.L.s3o_set_pcg(self.h, rel_tol, max_iter))
    def set_stop_rules(self, max_abs_step=0.0, min_rel_predicted_decrease=0.0):
        self._check(self.L.s3o_set_stop_rules(self.h, float(max_abs_step), float(min_rel_predicted_decrease)))
    def set_preconditioner(self, kind): self._check(self.L.s3o_set_preconditioner(self.h, int(kind)))
    def set_linear_solver(self, kind): self._check(self.L.s3o_set_linear_solver(self.h, int(kind)))

    # ---- structure ---------------------------------------------------------------
    def build_structure(self):
        nf, nb = C.c_int(0), C.c_int(0)
        self._check(self.L.s3o_build_structure(self.h, C.byref(nf), C.byref(nb)))
        self.num_free, self.num_blocks = nf.value, nb.value
        colptr = np.zeros(nf.value + 1, np.int32)
        rowidx = np.zeros(max(nb.value, 1), np.int32)
        self._check(self.L.s3o_get_structure(self.h, colptr.ctypes.data_as(_ip), rowidx.ctypes.data_as(_ip)))
        return colptr, rowidx[:nb.value]

    def hessian_index(self):
        h = np.zeros(self.nv, np.int32)
        self._check(self.L.s3o_get_hessian_index(self.h, h.ctypes.data_as(_ip)))
        return h

    # ---- lock-step pieces --------------------------------------------------------
    def chi2(self):
        out = C.c_double(0)
        self._check(self.L.s3o_chi2(self.h, C.byref(out)))
        return out.value

    def edge_errors(self):
        e = np.zeros((self.ne, self.d))
        self._check(self.L.s3o_edge_errors(self.h, _d(e)))
        return e

    def linearize(self):
        self._check(self.L.s3o_linearize(self.h))
        st = self.stats()
        H = np.zeros((st["n_blocks"], self.d, self.d))
        b = np.zeros(st["n_free"] * self.d)
        self._check(self.L.s3o_get_hessian(self.h, _d(H), _d(b)))
        return H, b

    def linearize_only(self):
        self._check(self.L.s3o_linearize(self.h))

    def max_diag(self):
        out = C.c_double(0)
        self._check(self.L.s3o_max_diag(self.h, C.byref(out)))
        return out.value

    def solve(self, lam):
        st = self.stats()
        x = np.zeros(st["n_free"] * self.d)
        it, rel = C.c_int(0), C.c_double(0)
        rc = self.L.s3o_solve(self.h, float(lam), _d(x), C.byref(it), C.byref(rel))
        if rc not in (0, -6):            # -6 = S3O_ERR_SOLVE: reported to the caller like g2o's solve() == false
            self._check(rc)
        return rc, x, it.value, rel.value

    def hessian_multiply(self, lam, x):
        x = _f64(x)
        y = np.zeros_like(x)
        self._check(self.L.s3o_hessian_multiply(self.h, float(lam), _d(x), _d(y)))
        return y

    def update(self, x):
        x = _f64(x)
        self._check(self.L.s3o_update(self.h, _d(x)))

    def smallest_eigenvector(self, max_iter=50, tol=1e-12):
        """(x, lambda_min, lambda_max, iterations) of H at the current estimates (stepwise scale init)."""
        self.build_structure()
        x = np.zeros(self.num_free * self.d)
        lmin, lmax, it = C.c_double(0), C.c_double(0), C.c_int(0)
        self._check(self.L.s3o_smallest_eigenvector(self.h, max_iter, tol, _d(x), C.byref(lmin), C.byref(lmax), C.byref(it)))
        return x, lmin.value, lmax.value, it.value

    def marginals(self, pairs=None):
        """Marginal covariances (g2o SparseOptimizer::computeMarginals): blocks of H^-1, H the undamped Gauss-Newton
        Hessian at the current estimates.  pairs=None: the (n_free, d, d) diagonal blocks in Hessian order; otherwise
        an (m, 2) array of Hessian-index pairs (row, col) -> (m, d, d).
        Within the sparse Cholesky's forced cap the blocks come from the selected inverse of its factor.  Beyond it
        (s100k, S1M) only explicit pairs are served, by d PCG solves per distinct column vertex, each refined to a
        true residual |e - H x| <= 1e-10 (S3O_MARGINALS_PCG_TOL); pairs=None raises there.  S3O_MARGINALS_ROUTE=pcg
        in the environment takes the iterative route on any graph."""
        self.build_structure()
        if pairs is None:
            out = np.zeros((self.num_free, self.d, self.d))
            self._check(self.L.s3o_compute_marginals(self.h, self.num_free, None, None, _d(out)))
            return out
        pairs = np.ascontiguousarray(np.asarray(pairs, np.int32).reshape(-1, 2))
        rows, cols = np.ascontiguousarray(pairs[:, 0]), np.ascontiguousarray(pairs[:, 1])
        out = np.zeros((len(pairs), self.d, self.d))
        self._check(self.L.s3o_compute_marginals(self.h, len(pairs), rows.ctypes.data_as(_ip), cols.ctypes.data_as(_ip),
                                                 _d(out)))
        return out

    # ---- the hot call ------------------------------------------------------------
    def optimize(self, max_iter, stop_rel_gain=0.0):
        hist = np.zeros((max(max_iter, 1), 5))
        n, chi2, lam = C.c_int(0), C.c_double(0), C.c_double(0)
        self._check(self.L.s3o_optimize(self.h, max_iter, stop_rel_gain, C.byref(n), C.byref(chi2), C.byref(lam),
                                        _d(hist), max_iter))
        return n.value, chi2.value, lam.value, hist[:max(n.value, 0)]

    def set_lm_resume(self, resume=1): self._check(self.L.s3o_set_lm_resume(self.h, int(resume)))
    def snapshot_estimates(self): self._check(self.L.s3o_snapshot_estimates(self.h))
    def restore_estimates(self): self._check(self.L.s3o_restore_estimates(self.h))

    def vertices(self, out=None):
        if out is not None:
            self._check(self.L.s3o_get_vertices(self.h, _d(out)))
            return out
        return self._vertices()

    def _vertices(self):
        est = np.zeros((self.nv, self.est_dim))
        self._check(self.L.s3o_get_vertices(self.h, _d(est)))
        return est

    def stats(self):
        st = _lib.Stats()
        self._check(self.L.s3o_get_stats(self.h, C.byref(st)))
        return {name: getattr(st, name) for name, _ in _lib.Stats._fields_}

    def reset_stats(self): self._check(self.L.s3o_reset_stats(self.h))

    def estimate_sigma_squared(self, robust_kind):
        out = C.c_double(0)
        self._check(self.L.s3o_estimate_sigma_squared(self.h, robust_kind, C.byref(out)))
        return out.value


def comm_unique_id():
    """128-byte NCCL unique id (rank 0 creates it; broadcast it to the other ranks)."""
    L = _lib.load()
    buf = C.create_string_buffer(128)
    rc = L.s3o_comm_unique_id(buf)
    if rc != 0:
        raise S3OError(f"s3o error {rc}: {L.s3o_last_error().decode()}")
    return buf.raw


def host_partition(n_vertices, fixed, v0, v1, rank, world):
    """Partition plan of one rank, computed on the host (no device needed)."""
    L = _lib.load()
    v0 = np.ascontiguousarray(v0, np.int32)
    v1 = np.ascontiguousarray(v1, np.int32)
    fx = np.zeros(n_vertices, np.uint8) if fixed is None else np.ascontiguousarray(fixed, np.uint8)
    scal = [C.c_int32(0) for _ in range(4)]
    ghosts = np.zeros(max(n_vertices, 1), np.int32)
    send_idx = np.zeros(max(n_vertices * max(world - 1, 1), 1), np.int32)
    send_count = np.zeros(world, np.int32)
    recv_count = np.zeros(world, np.int32)
    rc = L.s3o_host_partition(n_vertices, fx.ctypes.data_as(_up), len(v0), v0.ctypes.data_as(_ip),
                              v1.ctypes.data_as(_ip), rank, world, *[C.byref(x) for x in scal],
                              ghosts.ctypes.data_as(_ip), send_count.ctypes.data_as(_ip),
                              recv_count.ctypes.data_as(_ip), send_idx.ctypes.data_as(_ip))
    if rc != 0:
        raise S3OError(f"s3o error {rc}: {L.s3o_last_error().decode()}")
    n_own, n_ghost, n_local, n_primary = (x.value for x in scal)
    return dict(n_own=n_own, n_ghost=n_ghost, n_local_edges=n_local, n_primary=n_primary,
                ghosts=ghosts[:n_ghost].copy(), send_count=send_count, recv_count=recv_count,
                send_idx=send_idx[:int(send_count.sum())].copy())


def align_similarity(query_xyz, train_xyz, only_scale=False, device=0):
    """Umeyama similarity of the query positions onto the train positions (kitti_surf.cpp:1091-1161) and the
    RMSE / max deviation of the aligned points (:1432-1452).  Returns (S221 4x4, rmse, max_dev)."""
    L = _lib.load()
    q = _f64(query_xyz).reshape(-1, 3)
    t = _f64(train_xyz).reshape(-1, 3)
    if len(q) != len(t):
        raise S3OError("align_similarity: trajectories differ in length")
    S = np.zeros(16)
    rmse, mx = C.c_double(0), C.c_double(0)
    rc = L.s3o_align_similarity(int(device), len(q), _d(q), _d(t), 1 if only_scale else 0, _d(S), C.byref(rmse), C.byref(mx))
    if rc != 0:
        raise S3OError(f"s3o error {rc}: {L.s3o_last_error().decode()}")
    return S.reshape(4, 4), rmse.value, mx.value


def host_multilevel(n_vertices, fixed, v0, v1, world=1):
    """Aggregation hierarchy of the multilevel preconditioner (host only): per-level vertex counts,
    per-level block counts, and the finest-level aggregate of every free vertex."""
    L = _lib.load()
    v0 = np.ascontiguousarray(v0, np.int32)
    v1 = np.ascontiguousarray(v1, np.int32)
    fx = np.zeros(n_vertices, np.uint8) if fixed is None else np.ascontiguousarray(fixed, np.uint8)
    nl = C.c_int(0)
    nvert, nblk = np.zeros(16, np.int32), np.zeros(16, np.int32)
    agg = np.full(max(int((fx == 0).sum()), 1), -1, np.int32)
    rc = L.s3o_host_multilevel(n_vertices, fx.ctypes.data_as(_up), len(v0), v0.ctypes.data_as(_ip),
                               v1.ctypes.data_as(_ip), int(world), 16, C.byref(nl), nvert.ctypes.data_as(_ip),
                               nblk.ctypes.data_as(_ip), agg.ctypes.data_as(_ip))
    if rc != 0:
        raise S3OError(f"s3o error {rc}: {L.s3o_last_error().decode()}")
    return nvert[:nl.value].copy(), nblk[:nl.value].copy(), agg[:int((fx == 0).sum())]


def host_structure(n_vertices, fixed, v0, v1):
    """g2o-order upper block-CCS from plain arrays, computed on the host (no device needed)."""
    L = _lib.load()
    v0 = np.ascontiguousarray(v0, np.int32)
    v1 = np.ascontiguousarray(v1, np.int32)
    fx = np.zeros(n_vertices, np.uint8) if fixed is None else np.ascontiguousarray(fixed, np.uint8)
    nf, nb = C.c_int(0), C.c_int(0)
    colptr = np.zeros(n_vertices + 1, np.int32)
    rowidx = np.zeros(n_vertices + len(v0) + 1, np.int32)
    hidx = np.zeros(max(n_vertices, 1), np.int32)
    rc = L.s3o_host_structure(n_vertices, fx.ctypes.data_as(_up), len(v0), v0.ctypes.data_as(_ip),
                              v1.ctypes.data_as(_ip), C.byref(nf), C.byref(nb), colptr.ctypes.data_as(_ip),
                              rowidx.ctypes.data_as(_ip), hidx.ctypes.data_as(_ip))
    if rc != 0:
        raise S3OError(f"s3o error {rc}: {L.s3o_last_error().decode()}")
    return colptr[:nf.value + 1].copy(), rowidx[:nb.value].copy(), hidx[:n_vertices].copy()


class LinearSolver:
    """LinearSolver-level plug-in (s3o_linsolver_*): solve (A + lambda I) x = b for an upper block-CCS matrix, the
    slot of g2o::LinearSolver<M>::solve(A, x, b) (kitti_surf.cpp:553-557)."""

    def __init__(self, block_dim, device=0):
        self.L = _lib.load()
        self.d = int(block_dim)
        self.h = C.c_void_p()
        rc = self.L.s3o_linsolver_create(int(device), self.d, C.byref(self.h))
        if rc != 0:
            raise S3OError(f"s3o error {rc}: {self.L.s3o_last_error().decode()}")

    def close(self):
        if getattr(self, "h", None):
            self.L.s3o_linsolver_destroy(self.h)
            self.h = None

    __del__ = close

    def set_linear_solver(self, kind):
        if self.L.s3o_set_linear_solver(self.h, int(kind)) != 0:
            raise S3OError(self.L.s3o_last_error().decode())

    def set_pcg(self, rel_tol=0.0, max_iter=0):
        self.L.s3o_set_pcg(self.h, rel_tol, max_iter)

    def solve(self, colptr, rowidx, blocks, b, lam=0.0, column_major=False):
        """Returns (rc, x, method, pcg_iterations); rc 0 ok, -6 (S3O_ERR_SOLVE) not positive definite / not converged."""
        colptr = np.ascontiguousarray(colptr, np.int32)
        rowidx = np.ascontiguousarray(rowidx, np.int32)
        blocks = _f64(blocks)
        b = _f64(b).reshape(-1)
        n = len(colptr) - 1
        x = np.zeros(n * self.d)
        method, its = C.c_int(0), C.c_int(0)
        rc = self.L.s3o_linsolver_solve(self.h, n, colptr.ctypes.data_as(_ip), rowidx.ctypes.data_as(_ip), _d(blocks),
                                        1 if column_major else 0, float(lam), _d(b), _d(x), C.byref(method), C.byref(its))
        if rc not in (0, -6):
            raise S3OError(f"s3o error {rc}: {self.L.s3o_last_error().decode()}")
        return rc, x, method.value, its.value


def host_direct_plan(n_vertices, fixed, v0, v1, max_pairs=0):
    """Factorisation plan of the DIRECT linear solver (host only): dict with perm, lev_ptr, cptr, brow, src,
    upd_ptr, upd_a, upd_b and the counts n, rounds, n_pairs."""
    L = _lib.load()
    v0 = np.ascontiguousarray(v0, np.int32)
    v1 = np.ascontiguousarray(v1, np.int32)
    fx = np.zeros(n_vertices, np.uint8) if fixed is None else np.ascontiguousarray(fixed, np.uint8)
    counts = (C.c_int64 * 5)()
    null = C.POINTER(C.c_int32)()

    def call(*arrs):
        rc = L.s3o_host_direct_plan(n_vertices, fx.ctypes.data_as(_up), len(v0), v0.ctypes.data_as(_ip),
                                    v1.ctypes.data_as(_ip), int(max_pairs), counts, *arrs)
        if rc != 0:
            raise S3OError(f"s3o error {rc}: {L.s3o_last_error().decode()}")

    call(*([null] * 8))
    n, nlev, nL, nupd, pairs = (int(c) for c in counts)
    out = {"perm": np.zeros(n, np.int32), "lev_ptr": np.zeros(nlev + 1, np.int32), "cptr": np.zeros(n + 1, np.int32),
           "brow": np.zeros(nL, np.int32), "src": np.zeros(nL, np.int32), "upd_ptr": np.zeros(nL + 1, np.int32),
           "upd_a": np.zeros(max(nupd, 1), np.int32), "upd_b": np.zeros(max(nupd, 1), np.int32)}
    call(*(out[k].ctypes.data_as(_ip) for k in ("perm", "lev_ptr", "cptr", "brow", "src", "upd_ptr", "upd_a", "upd_b")))
    out["upd_a"], out["upd_b"] = out["upd_a"][:nupd], out["upd_b"][:nupd]
    out.update(n=n, rounds=nlev, n_pairs=pairs)
    return out


class BAProblem(Problem):
    """Bundle adjustment (kind S3O_KIND_BA): the g2o calls of ba_demo (bal_example.cpp:44-243).

    Shares chi2 / linearize_only / max_diag / optimize / stats / set_robust / set_lm / set_pcg /
    snapshot / restore with Problem; x of solve / update is [6 n_free_cameras | 3 n_free_points]."""

    def __init__(self, device=0, stream=None):
        super().__init__(KIND_BA, device, stream)
        self.nc = self.npts = self.no = 0

    def set(self, cams, points, obs_cam, obs_pt, uv, focal, cx, cy, cam_fixed=None, pt_fixed=None, info=None):
        cams = _f64(cams).reshape(-1, 7)
        points = _f64(points).reshape(-1, 3)
        oc = np.ascontiguousarray(obs_cam, np.int32)
        op = np.ascontiguousarray(obs_pt, np.int32)
        uv = _f64(uv).reshape(-1, 2)
        self.nc, self.npts, self.no = len(cams), len(points), len(oc)
        self.ne = self.no
        cf = None if cam_fixed is None else np.ascontiguousarray(cam_fixed, np.uint8)
        pf = None if pt_fixed is None else np.ascontiguousarray(pt_fixed, np.uint8)
        self._check(self.L.s3o_ba_set_cameras(self.h, self.nc, _d(cams), None if cf is None else cf.ctypes.data_as(_up)))
        self._check(self.L.s3o_ba_set_points(self.h, self.npts, _d(points), None if pf is None else pf.ctypes.data_as(_up)))
        infop = None
        if info is not None:
            info = _f64(info).reshape(self.no, 3)
            infop = _d(info)
        self._check(self.L.s3o_ba_set_observations(self.h, self.no, oc.ctypes.data_as(_ip), op.ctypes.data_as(_ip), _d(uv), infop))
        self._check(self.L.s3o_ba_set_intrinsics(self.h, float(focal), float(cx), float(cy)))

    def build_structure(self):
        colptr, rowidx = super().build_structure()
        ncf, npf, nb, ncon = C.c_int(0), C.c_int(0), C.c_int(0), C.c_int64(0)
        self._check(self.L.s3o_ba_get_sizes(self.h, C.byref(ncf), C.byref(npf), C.byref(nb), C.byref(ncon)))
        self.ncf, self.npf, self.nb, self.ncon = ncf.value, npf.value, nb.value, ncon.value
        return colptr, rowidx

    def set_estimates(self, cams=None, points=None):
        c = None if cams is None else _f64(cams).reshape(self.nc, 7)
        q = None if points is None else _f64(points).reshape(self.npts, 3)
        self._check(self.L.s3o_ba_set_estimates(self.h, None if c is None else _d(c), None if q is None else _d(q)))

    def cameras(self, out=None):
        c = np.zeros((self.nc, 7)) if out is None else out
        self._check(self.L.s3o_ba_get_cameras(self.h, _d(c)))
        return c

    def points(self, out=None):
        q = np.zeros((self.npts, 3)) if out is None else out
        self._check(self.L.s3o_ba_get_points(self.h, _d(q)))
        return q

    def edge_errors(self):
        e = np.zeros((self.no, 2))
        self._check(self.L.s3o_ba_edge_errors(self.h, _d(e)))
        return e

    def linearize(self):
        self.build_structure()
        self._check(self.L.s3o_linearize(self.h))
        Hpp, Hll = np.zeros((self.ncf, 6, 6)), np.zeros((self.npf, 3, 3))
        Hpl, b = np.zeros((self.no, 6, 3)), np.zeros(6 * self.ncf + 3 * self.npf)
        self._check(self.L.s3o_ba_get_system(self.h, _d(Hpp), _d(Hll), _d(Hpl), _d(b)))
        return Hpp, Hll, Hpl, b

    def schur(self, lam):
        S, bs = np.zeros((self.nb, 6, 6)), np.zeros(6 * self.ncf)
        self._check(self.L.s3o_ba_get_schur(self.h, float(lam), _d(S), _d(bs)))
        return S, bs

    def ba_marginals(self, pairs=None):
        """Marginal covariances of BA (s3o_ba_compute_marginals): blocks of H^-1, H the full undamped Gauss-Newton Hessian
        at the current estimates.  Hessian indices: free cameras 0..ncf-1, then free points ncf..ncf+npf-1.
        pairs=None: (cams (ncf, 6, 6), points (npf, 3, 3)), the diagonal blocks; otherwise an (m, 2) array of index
        pairs (row, col) -> a list of m arrays, (6 or 3) x (6 or 3) by the kinds of row and col."""
        self.build_structure()
        if pairs is None:
            out = np.zeros(36 * self.ncf + 9 * self.npf)
            self._check(self.L.s3o_ba_compute_marginals(self.h, self.ncf + self.npf, None, None, _d(out)))
            return out[:36 * self.ncf].reshape(self.ncf, 6, 6), out[36 * self.ncf:].reshape(self.npf, 3, 3)
        pairs = np.ascontiguousarray(np.asarray(pairs, np.int32).reshape(-1, 2))
        rows, cols = np.ascontiguousarray(pairs[:, 0]), np.ascontiguousarray(pairs[:, 1])
        dims = [(6 if r < self.ncf else 3, 6 if c < self.ncf else 3) for r, c in pairs]
        out = np.zeros(max(sum(a * b for a, b in dims), 1))
        self._check(self.L.s3o_ba_compute_marginals(self.h, len(pairs), rows.ctypes.data_as(_ip), cols.ctypes.data_as(_ip),
                                                    _d(out)))
        res, o = [], 0
        for a, b in dims:
            res.append(out[o:o + a * b].reshape(a, b).copy())
            o += a * b
        return res

    def solve(self, lam):
        x = np.zeros(6 * self.ncf + 3 * self.npf)
        it, rel = C.c_int(0), C.c_double(0)
        rc = self.L.s3o_solve(self.h, float(lam), _d(x), C.byref(it), C.byref(rel))
        return rc, x, it.value, rel.value

    def vertices(self, out=None):
        raise S3OError("BAProblem: use cameras() / points()")
