"""The tiled SpMV and the PCG at multi-tile shapes, checked against an independent host product.

Every PCG step, s3o_hessian_multiply and every backward-error check goes through the tiled SpMV (csrc/spmv.cu).  The
d = 7 kernel (spmv4) stages a CTA's tile descriptors in shared memory (up to KMAX), prefetches the block indices of
tile n+2 and the vectors of tile n+1 into registers, reuses an NS-deep TMA ring and grows the grid in waves above
grid_cap * KMAX tiles.  None of that runs while every CTA owns one tile, which is the case on all small fixtures.  The
per-problem switches S3O_SPMV_GRID, S3O_SPMV_VERSION and S3O_SPMV4_CFG force the other regimes on graphs of a few
thousand vertices; a Python twin of the tile builder tells which regime each case reaches, and the case asserts it.

Products are compared with (A + lambda I) x accumulated in long double, component by component, under the rounding
bound of an fp64 sum in any order; solutions by their backward error against the same host product.
"""
import contextlib
import os

import numpy as np
import pytest
from scipy.spatial.transform import Rotation

from conftest import KITTI_DIR, make_gpu, make_oracle

U = 2.0 ** -53
KMAX = 384                  # Spmv4Cfg::KMAX: tile descriptors per CTA
DEFAULT_CAP = 148 * 2       # s3o_problem::spmv_grid_cap
MAX_PARTIALS = 4096         # kMaxPartials
SPMV4_TB = (112, 80, 56)    # S3O_SPMV4_CFG 0, 1, 2
SPMV4_NS = (2, 3, 4)


# ---- host reference product ---------------------------------------------------------------------------------------
def host_product(colptr, rowidx, H, lam, x):
    """(A + lam I) x for the symmetric matrix whose upper block-CCS is (colptr, rowidx, H), accumulated in long double.

    Returns (y, m, n): y the product, m = (|A| + lam I)|x|, and n the number of products summed into each component
    (d per block of the full symmetric block row, plus the lambda term)."""
    H = np.asarray(H)
    d = H.shape[-1]
    nf = len(colptr) - 1
    col = np.repeat(np.arange(nf), np.diff(colptr))
    row = np.asarray(rowidx, np.int64)
    off = row != col

    def apply(B, X, lam):
        Y = lam * X
        np.add.at(Y, row, np.einsum("kij,kj->ki", B, X[col]))
        np.add.at(Y, col[off], np.einsum("kji,kj->ki", B[off], X[row[off]]))
        return Y.reshape(-1)

    X = np.asarray(x, np.longdouble).reshape(nf, d)
    B = H.astype(np.longdouble)
    y = apply(B, X, np.longdouble(lam))
    m = apply(np.abs(B), np.abs(X), np.longdouble(abs(lam)))
    nblk = np.bincount(row, minlength=nf) + np.bincount(col[off], minlength=nf)
    return y, m, np.repeat(d * nblk + 1, d)


def product_error(y, ref):
    """Worst |y - y_ref| / (2 n u m) over the components: at most 1 for an fp64 product summed in any order.  A dropped,
    duplicated, transposed or misrouted block exceeds it by orders of magnitude, also in rows whose values are small."""
    y_ref, m, n = ref
    err = np.abs(np.asarray(y, np.longdouble) - y_ref)
    bound = 2 * n * U * m
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(bound > 0, err / bound, np.where(err > 0, np.inf, 0.0))
    return float(r.max())


def backward_error(colptr, rowidx, H, lam, x, b):
    """|(A + lam I) x - b| / |b| with the host product."""
    y, _, _ = host_product(colptr, rowidx, H, lam, x)
    return float(np.linalg.norm((y - np.asarray(b, np.longdouble)).astype(np.float64)) / np.linalg.norm(b))


# ---- twin of the tile builder and of the kernel choice ------------------------------------------------------------
def build_tiles(row_blocks, cap):
    """Mirrors build_tiles (csrc/structure.cpp): first row of every tile, then nf."""
    nf = len(row_blocks)
    tile_row = [0]
    r = 0
    while r < nf:
        start, blocks = r, 0
        while r < nf:
            nb = int(row_blocks[r])
            if blocks + nb > cap and r > start:
                break
            blocks += nb
            r += 1
            if blocks >= cap:
                break
        tile_row.append(r)
    return np.array(tile_row)


def spmv4_grid(ntiles, grid_cap):
    """Mirrors spmv4_grid (csrc/spmv.cu): grid_cap CTAs, times the number of waves that keeps ntl <= KMAX."""
    if ntiles <= grid_cap:
        return ntiles
    return grid_cap * (-(-ntiles // (grid_cap * KMAX)))


def spmv_plan(row_blocks, d, version=4, cfg=0, cap=DEFAULT_CAP):
    """Which SpMV a problem runs (run_spmv in csrc/problem.cu), its tiles, grid and tiles per CTA."""
    if version == 4 and d == 7:
        tb = SPMV4_TB[cfg]
    elif version >= 3:
        tb = {7: 112, 6: 128}.get(d, 256)
    else:
        tb = 128 if d >= 6 else 256
    tile_row = build_tiles(row_blocks, tb)
    nt = len(tile_row) - 1
    longest = int(np.max(row_blocks))
    grid = None
    if version == 1:
        kernel = "v1"
    elif version == 4 and d == 7 and longest <= tb and 0 < spmv4_grid(nt, cap) <= MAX_PARTIALS \
            and -(-nt // spmv4_grid(nt, cap)) <= KMAX:
        kernel, grid = "v4", spmv4_grid(nt, cap)
    elif version >= 3 and longest <= tb:
        kernel, grid = "v3", min(nt, cap)
    else:
        kernel, grid = "v2", min(nt, 148 * 24)
    return dict(kernel=kernel, tb=tb, tile_row=tile_row, ntiles=nt, grid=grid,
                per_cta=None if grid is None else -(-nt // grid))


def row_blocks_of(colptr, rowidx):
    """Blocks per BSR-upper row (the tile builder's input) from the upper block-CCS."""
    return np.bincount(rowidx, minlength=len(colptr) - 1)


# ---- graphs -------------------------------------------------------------------------------------------------------
def _with_edges(g, v0, v1, seed):
    """g's vertices with the edges (v0, v1) and measurements C = exp(noise) S_j S_i^-1 (identity information)."""
    from sim3opt_b200 import synth
    est = g["est"]
    R, t, s = Rotation.from_quat(est[:, :4]), est[:, 4:7], est[:, 7]
    Sji = synth._mul(R[v1], t[v1], s[v1], *synth._inv(R[v0], t[v0], s[v0]))
    noise = synth.sim3_exp(0.01 * np.random.default_rng(seed).standard_normal((len(v0), 7)))
    meas = synth._pack(*synth._mul(*noise, *Sji))
    return dict(est=est, fixed=g["fixed"], v0=np.asarray(v0, np.int32), v1=np.asarray(v1, np.int32), meas=meas)


def chain(n_free):
    """One fixed vertex followed by n_free free ones, edges (k, k+1): every BSR-upper row has two blocks but the last."""
    from sim3opt_b200 import synth
    g = synth.sphere(n_laps=1, poses_per_lap=n_free + 1, seed=3)
    keep = g["v1"] - g["v0"] == 1
    return dict(est=g["est"], fixed=g["fixed"], v0=g["v0"][keep], v1=g["v1"][keep], meas=g["meas"][keep],
                info=g["info"][keep])


def hub(n_hub_edges, n=1500):
    """A chain of n vertices (vertex 0 fixed) whose vertex 1, Hessian index 0, also links to vertices 2 .. n_hub_edges+1:
    the first BSR-upper row has n_hub_edges + 1 blocks."""
    from sim3opt_b200 import synth
    g = synth.sphere(n_laps=1, poses_per_lap=n, seed=4)
    k = np.arange(n - 1)
    v0 = np.concatenate([k, np.ones(n_hub_edges - 1, np.int64)])
    v1 = np.concatenate([k + 1, np.arange(3, n_hub_edges + 2)])
    return _with_edges(g, v0, v1, seed=n_hub_edges)


def kitti_k118():
    from oracle import kitti_io
    return kitti_io.build_kitti_sim3_graph(KITTI_DIR, use_one_constraint=False)


def _sphere(*args, **kw):
    from sim3opt_b200 import synth
    return lambda: synth.sphere(*args, **kw)


GRAPHS = {
    "sphere_mid": _sphere(n_laps=10, poses_per_lap=300, seed=11),       # test_gpu_multilevel's sphere_mid
    "s10k": _sphere(100, 100, seed=42),                                  # bench parity graph
    "s30k": _sphere(n_laps=30, poses_per_lap=1000, seed=7),              # test_large_graph_kcycle_with_dense_coarsest_level
    "s100k": _sphere(100, 1000, seed=42),
    "chain21504": lambda: chain(21504),
    "chain21505": lambda: chain(21505),
    "kitti_k118": kitti_k118,
}
for _h in sorted({tb - 1 for tb in SPMV4_TB} | set(SPMV4_TB) | {300}):
    GRAPHS[f"hub{_h}"] = (lambda h: lambda: hub(h))(_h)


def as_kind(g, kind):
    """The Sim3 graph, or its 4-DoF scale+translation / 1-DoF scale twin (as in tests/test_gpu_parity.py)."""
    import sim3opt_b200 as s3
    from oracle import kitti_io
    if kind == s3.KIND_SIM3:
        return g
    st = kitti_io.to_scale_trans_graph(g)
    if kind == s3.KIND_SCALE_TRANS:
        return st
    return dict(est=st["est"][:, :1].copy(), fixed=st["fixed"], v0=st["v0"], v1=st["v1"], meas=st["meas"][:, :1].copy())


@pytest.fixture(scope="module")
def graph_of():
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = GRAPHS[name]()
        return cache[name]
    yield get
    cache.clear()


@contextlib.contextmanager
def spmv_env(version=None, cfg=None, cap=None):
    """The SpMV switches, read once by s3o_create: set them only around Problem creation."""
    keys = {"S3O_SPMV_VERSION": version, "S3O_SPMV4_CFG": cfg, "S3O_SPMV_GRID": cap}
    old = {k: os.environ.get(k) for k in keys}
    try:
        for k, v in keys.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = str(v)
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def make_linearized(g, kind, version=None, cfg=None, cap=None):
    with spmv_env(version, cfg, cap):
        gpu = make_gpu(g, kind=kind, jac=1)
    colptr, rowidx = gpu.build_structure()
    H, b = gpu.linearize()
    return gpu, colptr, rowidx, H, b


# ---- 1. the host reference and its gate (CPU) ---------------------------------------------------------------------
def _random_block_system(nf=40, d=7, seed=0):
    rng = np.random.default_rng(seed)
    colptr, rowidx = [0], []
    for c in range(nf):
        rows = [r for r in range(c) if rng.random() < 0.15] + [c]
        rowidx += rows
        colptr.append(len(rowidx))
    H = rng.standard_normal((len(rowidx), d, d))
    diag = np.array(colptr[1:]) - 1                 # diagonal blocks are symmetric, as in a Hessian
    H[diag] = H[diag] + H[diag].transpose(0, 2, 1)
    return np.array(colptr, np.int32), np.array(rowidx, np.int32), H, rng.standard_normal(nf * d)


def _loop_product(colptr, rowidx, H, lam, x, corrupt=None, at=None):
    """Plain fp64 loop over the blocks, written independently of host_product; `corrupt` injects one defect at block
    `at` (an off-diagonal block)."""
    d = H.shape[-1]
    X = x.reshape(-1, d)
    Y = lam * X
    for c in range(len(colptr) - 1):
        for k in range(colptr[c], colptr[c + 1]):
            r, B = rowidx[k], H[k]
            if k == at and corrupt == "drop":
                continue
            if k == at and corrupt == "lambda_offdiag":
                B = B + lam * np.eye(d)
            src = c + 1 if k == at and corrupt == "neighbour_column" else c
            for i in range(d):
                Y[r, i] += sum(B[i, j] * X[src, j] for j in range(d))
            if r != c:
                Bt = B if k == at and corrupt == "untransposed" else B.T
                for i in range(d):
                    Y[c, i] += sum(Bt[i, j] * X[r, j] for j in range(d))
    return Y.reshape(-1)


def test_reference_is_more_precise_than_fp64():
    assert np.finfo(np.longdouble).eps < 1e-18


def test_host_product_gate_accepts_fp64_and_rejects_corruptions():
    colptr, rowidx, H, x = _random_block_system()
    lam = 0.7
    ref = host_product(colptr, rowidx, H, lam, x)
    assert product_error(_loop_product(colptr, rowidx, H, lam, x), ref) <= 1.0
    # and a dense fp64 product, summed in yet another order
    nf, d = len(colptr) - 1, H.shape[-1]
    A = np.zeros((nf * d, nf * d))
    for c in range(nf):
        for k in range(colptr[c], colptr[c + 1]):
            r = rowidx[k]
            A[c * d:(c + 1) * d, r * d:(r + 1) * d] = H[k].T
            A[r * d:(r + 1) * d, c * d:(c + 1) * d] = H[k]
    assert product_error(A @ x + lam * x, ref) <= 1.0
    col = np.repeat(np.arange(nf), np.diff(colptr))
    at = int(np.flatnonzero((rowidx != col) & (col < nf - 1))[3])
    for corrupt in ("drop", "untransposed", "lambda_offdiag", "neighbour_column"):
        y = _loop_product(colptr, rowidx, H, lam, x, corrupt=corrupt, at=at)
        assert product_error(y, ref) > 1e6, corrupt


def test_host_product_gate_catches_a_wrong_small_row():
    """A relative-to-max|y| tolerance lets a wrong row of tiny values through; the componentwise gate does not."""
    colptr, rowidx, H, x = _random_block_system(seed=1)
    d = H.shape[-1]
    x = x * np.repeat(10.0 ** np.random.default_rng(2).uniform(-8, 8, len(x) // d), d)
    ref = host_product(colptr, rowidx, H, 0.0, x)
    y = ref[0].astype(np.float64)
    i = int(np.argmin(ref[1]))
    y[i] *= 1 + 1e-9
    assert np.abs(y - ref[0].astype(np.float64)).max() <= 1e-12 * np.abs(y).max()
    assert product_error(y, ref) > 1.0


# ---- the tile twin (CPU) ------------------------------------------------------------------------------------------
def test_tile_twin_reproduces_the_fixture_regimes(graph_of):
    """Tiles (TB = 112) and tiles per CTA at the default grid cap of the fixtures the GPU suite uses."""
    import sim3opt_b200 as s3
    from oracle import kitti_io
    from sim3opt_b200 import synth
    small = {"kitti_k1": kitti_io.build_kitti_sim3_graph(KITTI_DIR, use_one_constraint=True),
             "kitti_k118": graph_of("kitti_k118"),
             "sphere_small": synth.sphere(n_laps=12, poses_per_lap=40, seed=7),
             "manhattan_small": synth.manhattan3d(500, seed=5)}
    expect = {"kitti_k1": 14, "kitti_k118": 15, "sphere_small": 26, "manhattan_small": 23,
              "sphere_mid": 155, "s10k": 552, "s30k": 1628, "s100k": 5517}
    per_cta = {"sphere_mid": 1, "s10k": 2, "s30k": 6, "s100k": 19}
    for name, nt in expect.items():
        g = small[name] if name in small else graph_of(name)
        colptr, rowidx, _ = s3.host_structure(len(g["est"]), g["fixed"], g["v0"], g["v1"])
        plan = spmv_plan(row_blocks_of(colptr, rowidx), 7)
        assert plan["kernel"] == "v4" and plan["ntiles"] == nt, (name, plan["ntiles"])
        assert plan["per_cta"] == per_cta.get(name, 1), name


def test_tile_twin_chain_and_hub_regimes(graph_of):
    import sim3opt_b200 as s3
    rb = {}
    for name in ("chain21504", "chain21505", "hub111", "hub112"):
        g = graph_of(name)
        colptr, rowidx, _ = s3.host_structure(len(g["est"]), g["fixed"], g["v0"], g["v1"])
        rb[name] = row_blocks_of(colptr, rowidx)
    got = lambda name, **kw: tuple(spmv_plan(rb[name], 7, **kw)[k] for k in ("kernel", "ntiles", "grid", "per_cta"))
    assert got("chain21504", cfg=0, cap=1) == ("v4", 384, 1, 384)          # ntl == KMAX
    assert got("chain21504", cfg=2, cap=1) == ("v4", 768, 2, 384)          # two waves of KMAX
    assert got("chain21504", cfg=1, cap=1) == ("v4", 538, 2, 269)
    assert got("chain21505", cfg=0, cap=1) == ("v4", 385, 2, 193)
    assert rb["hub111"][0] == 112 and got("hub111", cfg=0)[0] == "v4"
    assert rb["hub112"][0] == 113 and got("hub112", cfg=0)[0] == "v2"


# ---- 2. the SpMV at every regime (GPU, s3o_hessian_multiply) -------------------------------------------------------
SIM3, ST, SC = 0, 1, 2      # s3.KIND_SIM3, KIND_SCALE_TRANS, KIND_SCALE
# id: (graph, kind, S3O_SPMV_VERSION, S3O_SPMV4_CFG, S3O_SPMV_GRID) -> (kernel, tiles, grid, tiles per CTA)
SPMV_CASES = {
    # one CTA walks every tile; ring wrap for every NS; tiles per CTA odd and even relative to NS
    "mid-tb112-cap1": (("sphere_mid", SIM3, None, 0, 1), ("v4", 155, 1, 155)),
    "mid-tb112-cap2": (("sphere_mid", SIM3, None, 0, 2), ("v4", 155, 2, 78)),
    "mid-tb112-cap3": (("sphere_mid", SIM3, None, 0, 3), ("v4", 155, 3, 52)),
    "mid-tb112-cap7": (("sphere_mid", SIM3, None, 0, 7), ("v4", 155, 7, 23)),
    "mid-tb80-cap1": (("sphere_mid", SIM3, None, 1, 1), ("v4", 215, 1, 215)),
    "mid-tb80-cap2": (("sphere_mid", SIM3, None, 1, 2), ("v4", 215, 2, 108)),
    "mid-tb80-cap3": (("sphere_mid", SIM3, None, 1, 3), ("v4", 215, 3, 72)),
    "mid-tb80-cap7": (("sphere_mid", SIM3, None, 1, 7), ("v4", 215, 7, 31)),
    "mid-tb56-cap1": (("sphere_mid", SIM3, None, 2, 1), ("v4", 311, 1, 311)),
    "mid-tb56-cap2": (("sphere_mid", SIM3, None, 2, 2), ("v4", 311, 2, 156)),
    "mid-tb56-cap3": (("sphere_mid", SIM3, None, 2, 3), ("v4", 311, 3, 104)),
    "mid-tb56-cap7": (("sphere_mid", SIM3, None, 2, 7), ("v4", 311, 7, 45)),
    # the default grid on the 30k-pose sphere
    "s30k-tb112": (("s30k", SIM3, None, 0, None), ("v4", 1628, 296, 6)),
    "s30k-tb80": (("s30k", SIM3, None, 1, None), ("v4", 2255, 296, 8)),
    "s30k-tb56": (("s30k", SIM3, None, 2, None), ("v4", 3258, 296, 12)),
    # KMAX descriptors per CTA, and grids that grow in waves
    "chain-tb112-kmax": (("chain21504", SIM3, None, 0, 1), ("v4", 384, 1, 384)),
    "chain-tb56-2waves": (("chain21504", SIM3, None, 2, 1), ("v4", 768, 2, 384)),
    "chain-tb80-cap1": (("chain21504", SIM3, None, 1, 1), ("v4", 538, 2, 269)),
    "chain+1-tb112-cap1": (("chain21505", SIM3, None, 0, 1), ("v4", 385, 2, 193)),
    "s10k-tb112-cap1": (("s10k", SIM3, None, 0, 1), ("v4", 552, 2, 276)),
    # a row of exactly tile_blocks blocks stays on v4; one more block takes the hub-row kernel (v2)
    "hub-tb112-fits": (("hub111", SIM3, None, 0, 2), ("v4", 28, 2, 14)),
    "hub-tb112-over": (("hub112", SIM3, None, 0, 2), ("v2", 28, 28, 1)),
    "hub-tb80-fits": (("hub79", SIM3, None, 1, 2), ("v4", 39, 2, 20)),
    "hub-tb80-over": (("hub80", SIM3, None, 1, 2), ("v2", 39, 39, 1)),
    "hub-tb56-fits": (("hub55", SIM3, None, 2, 2), ("v4", 55, 2, 28)),
    "hub-tb56-over": (("hub56", SIM3, None, 2, 2), ("v2", 55, 55, 1)),
    # d = 4 and d = 1: v3 with small grids, and a hub row longer than a tile (v2)
    "st-v3-cap1": (("kitti_k118", ST, None, None, 1), ("v3", 7, 1, 7)),
    "st-v3-cap3": (("kitti_k118", ST, None, None, 3), ("v3", 7, 3, 3)),
    "st-hub-v2": (("hub300", ST, None, None, None), ("v2", 13, 13, 1)),
    "scale-v3-cap1": (("kitti_k118", SC, None, None, 1), ("v3", 7, 1, 7)),
    "scale-v3-cap3": (("kitti_k118", SC, None, None, 3), ("v3", 7, 3, 3)),
    "scale-hub-v2": (("hub300", SC, None, None, None), ("v2", 13, 13, 1)),
    # the experiment kernels of d = 7, once each
    "mid-v1": (("sphere_mid", SIM3, 1, None, 1), ("v1", 134, None, None)),
    "mid-v3-cap1": (("sphere_mid", SIM3, 3, None, 1), ("v3", 155, 1, 155)),
}


def test_spmv_cases_are_distinct_regimes():
    """The item list of the sweep: at least one case has ntl == KMAX, one runs two or more waves, and every spmv4
    configuration has a case with more than NS tiles per CTA."""
    cases = list(SPMV_CASES.values())
    assert any(e[0] == "v4" and e[3] == KMAX for _, e in cases)
    assert any(e[0] == "v4" and a[4] and e[2] >= 2 * a[4] for a, e in cases)
    for cfg, ns in enumerate(SPMV4_NS):
        assert any(e[0] == "v4" and a[3] == cfg and e[3] >= ns + 1 for a, e in cases)


def probe_vectors(plan, n, d, seed):
    """A standard normal x, x with per-vertex magnitudes over 1e-8 .. 1e8, and unit vectors on the first and the last
    row of a few tiles (the last tile among them)."""
    rng = np.random.default_rng(seed)
    nf = n // d
    out = [("normal", rng.standard_normal(n)),
           ("spread", rng.standard_normal(n) * np.repeat(10.0 ** rng.uniform(-8, 8, nf), d))]
    tr = plan["tile_row"]
    nt = len(tr) - 1
    for t in sorted({0, 1, nt // 2, nt - 1} & set(range(nt))):
        for row, c in ((tr[t], 0), (tr[t + 1] - 1, d - 1)):
            e = np.zeros(n)
            e[row * d + c] = 1.0
            out.append((f"e[tile {t} row {row}]", e))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(SPMV_CASES))
def test_spmv_shapes_against_host_product(case, graph_of):
    (gname, kind, version, cfg, cap), expect = SPMV_CASES[case]
    g = as_kind(graph_of(gname), kind)
    gpu, colptr, rowidx, H, b = make_linearized(g, kind, version, cfg, cap)
    try:
        d = H.shape[-1]
        plan = spmv_plan(row_blocks_of(colptr, rowidx), d, 4 if version is None else version,
                         0 if cfg is None else cfg, DEFAULT_CAP if cap is None else cap)
        assert (plan["kernel"], plan["ntiles"], plan["grid"], plan["per_cta"]) == expect
        for lam in (0.0, 1e3 * gpu.max_diag()):
            for name, x in probe_vectors(plan, len(b), d, seed=len(case)):
                y = gpu.hessian_multiply(lam, x)
                err = product_error(y, host_product(colptr, rowidx, H, lam, x))
                assert err <= 1.0, (name, lam, err)
    finally:
        gpu.close()


# ---- 3. the PCG at those shapes (GPU, backward error with the host product) ----------------------------------------
# id: (graph, kind, S3O_SPMV4_CFG, S3O_SPMV_GRID, lambda / max_diag) -> grid the p.q reduction runs over
PCG_CASES = {
    "mid-tb112-cap1": (("sphere_mid", SIM3, 0, 1, 1e-5), 1),
    "mid-tb80-cap2": (("sphere_mid", SIM3, 1, 2, 1e-5), 2),
    "mid-tb56-cap3": (("sphere_mid", SIM3, 2, 3, 1e-5), 3),
    "mid-default": (("sphere_mid", SIM3, None, None, 1e-5), 155),
    "s30k-default": (("s30k", SIM3, None, None, 1e-4), 296),
    "s30k-tb56-default": (("s30k", SIM3, 2, None, 1e-4), 296),
    "s30k-tb112-cap1-waves": (("s30k", SIM3, 0, 1, 1e-4), 5),
    "chain-tb56-2waves": (("chain21504", SIM3, 2, 1, 1e-4), 2),
    "st-cap1": (("kitti_k118", ST, None, 1, 1e-5), 1),
    "st-cap3": (("kitti_k118", ST, None, 3, 1e-5), 3),
    "scale-cap1": (("kitti_k118", SC, None, 1, 1e-5), 1),
    "scale-cap3": (("kitti_k118", SC, None, 3, 1e-5), 3),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(PCG_CASES))
def test_pcg_shapes_backward_error(case, graph_of):
    import sim3opt_b200 as s3
    (gname, kind, cfg, cap, lam_rel), grid = PCG_CASES[case]
    g = as_kind(graph_of(gname), kind)
    gpu, colptr, rowidx, H, b = make_linearized(g, kind, None, cfg, cap)
    try:
        plan = spmv_plan(row_blocks_of(colptr, rowidx), H.shape[-1], 4, 0 if cfg is None else cfg,
                         DEFAULT_CAP if cap is None else cap)
        assert plan["grid"] == grid
        lam = lam_rel * gpu.max_diag()
        gpu.set_pcg(1e-11, 100000)
        for pre in (s3.PRECOND_BLOCK_JACOBI, s3.PRECOND_MULTILEVEL):
            gpu.set_preconditioner(pre)
            rc, x, it, rel = gpu.solve(lam)
            assert rc == 0 and rel <= 1e-11, (pre, rc, it, rel)
            assert backward_error(colptr, rowidx, H, lam, x, b) <= 1e-10, (pre, it)
        if len(b) <= 200000:                   # control: the exact solver on the same system (not through the SpMV)
            gpu.set_linear_solver(s3.LINSOLVER_DIRECT)
            rc, x, it, _ = gpu.solve(lam)
            assert rc == 0 and it == 0
            assert backward_error(colptr, rowidx, H, lam, x, b) <= 1e-12
    finally:
        gpu.close()


@pytest.mark.gpu
def test_pcg_ba_schur_one_cta():
    """d = 6: the Schur system of a bundle adjustment, one CTA walking every tile of the v3 SpMV."""
    import sim3opt_b200 as s3
    from sim3opt_b200 import synth
    g = synth.ba_loop(120, 6000, 8, seed=5)
    with spmv_env(cap=1):
        gpu = s3.BAProblem()
    try:
        gpu.set(g["cams"], g["points"], g["obs_cam"], g["obs_pt"], g["uv"], g["focal"], g["cx"], g["cy"])
        gpu.set_robust(s3.ROBUST_HUBER, 2.5)
        gpu.linearize()
        colptr, rowidx = gpu.build_structure()
        plan = spmv_plan(row_blocks_of(colptr, rowidx), 6, cap=1)
        assert plan["kernel"] == "v3" and plan["grid"] == 1 and plan["ntiles"] >= 4, plan["ntiles"]
        lam = 1e-5 * gpu.max_diag()
        S, bs = gpu.schur(lam)
        gpu.set_pcg(1e-12, 20000)
        rc, x, it, rel = gpu.solve(lam)
        assert rc == 0 and rel <= 1e-12
        assert backward_error(colptr, rowidx, S, 0.0, x[:6 * gpu.ncf], bs) <= 1e-10
    finally:
        gpu.close()


# ---- 4. the linearisation of the large graphs against the oracle, block by block ----------------------------------
def _dense_info(g, seed):
    g = dict(g)
    M = np.random.default_rng(seed).normal(0, 1, (len(g["v0"]), 7, 7))
    g["info"] = np.einsum("nij,nkj->nik", M, M) + 7 * np.eye(7)
    return g


@pytest.mark.gpu
@pytest.mark.parametrize("gname,dense", [("s30k", False), ("s30k", True), ("s100k", False)])
def test_linearize_per_block_against_oracle(gname, dense, graph_of):
    """Every Hessian block within 1e-10 of its own largest entry (a global scale lets a wrong small block through).

    Worst per-block ratio max|H_gpu - H_orc| / max|H_orc| measured on a B200 with analytic Jacobians: 5.7e-14 on the
    lock-step fixtures (kitti_k1 / kitti_k118; 5.2e-14 sphere_small, 1.2e-15 manhattan_small), 8.9e-14 on this 30k
    sphere, 1.0e-13 with dense information, 4.4e-12 on s100k."""
    from oracle import oracle as orc
    g = graph_of(gname)
    if dense:
        g = _dense_info(g, 12)
    gpu, cpu = make_gpu(g, jac=1), make_oracle(g, jac=orc.JAC_ANALYTIC)
    try:
        assert np.array_equal(gpu.build_structure()[1], cpu.build_structure()[1])
        Hg, _ = gpu.linearize()
        Hc, _ = cpu.linearize()
        scale = np.abs(Hc).max(axis=(1, 2))
        ratio = np.abs(Hg - Hc).max(axis=(1, 2)) / scale
        print(f"{gname} dense={dense}: worst per-block ratio {ratio.max():.3e}")
        assert (scale > 0).all() and ratio.max() <= 1e-10
    finally:
        gpu.close()


# ---- 5. the LinearSolver plug-in at block sizes 4 and 1 -------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind", [ST, SC])
def test_linsolver_block_sizes_4_and_1(kind, graph_of):
    """The oracle's scale+translation (d = 4) and scale (d = 1) systems of KITTI K118 through s3o_linsolver_solve:
    AUTO, forced PCG and forced DIRECT, row- and column-major blocks."""
    import sim3opt_b200 as s3
    from oracle import oracle as orc
    g = as_kind(graph_of("kitti_k118"), kind)
    cpu = make_oracle(g, kind=kind, jac=orc.JAC_ANALYTIC)
    colptr, rowidx = cpu.build_structure()
    H, b = cpu.linearize()
    d = H.shape[-1]
    assert d == (4 if kind == ST else 1)
    lam = 1e-5 * cpu.max_diag()
    rc, xc = cpu.solve(lam)
    assert rc == 0
    for mode in (s3.LINSOLVER_AUTO, s3.LINSOLVER_PCG, s3.LINSOLVER_DIRECT):
        ls = s3.LinearSolver(d)
        try:
            ls.set_pcg(1e-13, 200000)
            ls.set_linear_solver(mode)
            rc, x, method, its = ls.solve(colptr, rowidx, H, b, lam)
            assert rc == 0 and method == (s3.LINSOLVER_PCG if mode == s3.LINSOLVER_PCG else s3.LINSOLVER_DIRECT)
            assert backward_error(colptr, rowidx, H, lam, x, b) <= 1e-10, (mode, its)
            assert np.abs(x - xc).max() <= 1e-6 * np.abs(xc).max(), mode
            rc, x2, _, _ = ls.solve(colptr, rowidx, np.ascontiguousarray(H.transpose(0, 2, 1)), b, lam, column_major=True)
            assert rc == 0 and np.array_equal(x, x2), mode
        finally:
            ls.close()


# ---- 6. the SpMV switches are per problem ---------------------------------------------------------------------------
@pytest.mark.gpu
def test_spmv4_config_is_per_problem(graph_of):
    """Tiles are cut for the tile size of the problem's own configuration: a problem created later under another
    S3O_SPMV4_CFG does not change which kernel an earlier one runs."""
    g = graph_of("sphere_mid")
    a, cp_a, ri_a, H_a, _ = make_linearized(g, SIM3, cfg=0, cap=3)
    b, cp_b, ri_b, H_b, _ = make_linearized(g, SIM3, cfg=2, cap=3)
    try:
        rng = np.random.default_rng(9)
        for p, cp, ri, H in ((a, cp_a, ri_a, H_a), (b, cp_b, ri_b, H_b), (a, cp_a, ri_a, H_a)):
            x = rng.standard_normal(len(cp) * 7 - 7)
            assert product_error(p.hessian_multiply(0.5, x), host_product(cp, ri, H, 0.5, x)) <= 1.0
    finally:
        a.close()
        b.close()


@pytest.mark.gpu
def test_spmv_grid_cap_at_the_partials_limit(graph_of):
    """S3O_SPMV_GRID = kMaxPartials with the v3 kernel on s100k: a 4096-CTA grid, each CTA with its own p.q partial."""
    import sim3opt_b200 as s3
    gpu, colptr, rowidx, H, b = make_linearized(graph_of("s100k"), SIM3, version=3, cap=MAX_PARTIALS)
    try:
        plan = spmv_plan(row_blocks_of(colptr, rowidx), 7, version=3, cap=MAX_PARTIALS)
        assert (plan["kernel"], plan["ntiles"], plan["grid"]) == ("v3", 5517, MAX_PARTIALS)
        x = np.random.default_rng(10).standard_normal(len(b))
        assert product_error(gpu.hessian_multiply(0.0, x), host_product(colptr, rowidx, H, 0.0, x)) <= 1.0
        lam = 1e-3 * gpu.max_diag()
        gpu.set_preconditioner(s3.PRECOND_BLOCK_JACOBI)
        gpu.set_pcg(1e-11, 100000)
        rc, x, it, rel = gpu.solve(lam)
        assert rc == 0 and rel <= 1e-11
        assert backward_error(colptr, rowidx, H, lam, x, b) <= 1e-10
    finally:
        gpu.close()
