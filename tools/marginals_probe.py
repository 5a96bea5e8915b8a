"""Times s3o_compute_marginals (every diagonal block of H^-1) on K1, K118, sphere_small and the s10k sphere.

Each call is split by the library's CUDA events (S3O_MARGINALS_TRACE=1: linearise, factorisation, selected inverse,
gather) and timed end to end on the host; medians over --reps calls after --warmup calls.  Prints the plan's rounds,
blocks of L and block products, and for K1 / K118 the CPU oracle's dense inverse of the same H as a reference.
One JSON line per graph.

--ba: s3o_ba_compute_marginals (every camera and point diagonal block) on the graphs of tests/test_gpu_ba_marginals.py
(ba_small, ba_medium and the bench-size ba_loop(1000, 500000, 10); cameras 0 and 7 and the points seen by fewer than
two cameras fixed, Huber 2.5), split into linearise, Schur complement, factorisation, selected inverse, point phase and
gather.  Also prints sum_l |O(l)|^2, the 6x6-by-6x3 products of the point phase.

--pcg: the iterative route on the graphs beyond the sparse Cholesky's cap, s100k (synth.sphere(100, 1000)) and S1M
(synth.sphere(1000, 1000)).  The first call (one column vertex) includes the forced-cap plan analysis that finds the
factor too large; then one call each with 1, 2 and 8 column vertices (the diagonal block and one far row per column).
Per call: host time and CUDA-event time of the solves per column vertex, PCG iterations per right-hand side,
refinement rounds and the largest true residual.

    python tools/marginals_probe.py [--ba | --pcg] [--reps 50] [--warmup 5]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
os.environ["S3O_MARGINALS_TRACE"] = "1"


def graphs():
    from oracle import kitti_io
    from sim3opt_b200 import synth
    kd = os.path.join(ROOT, "tests", "golden", "kitti00")
    return {"K1": kitti_io.build_kitti_sim3_graph(kd, use_one_constraint=True),
            "K118": kitti_io.build_kitti_sim3_graph(kd, use_one_constraint=False),
            "sphere_small": synth.sphere(n_laps=12, poses_per_lap=40, seed=7),
            "s10k": synth.sphere(10, 1000, seed=42)}


class StderrCapture:
    """The library writes its trace lines to file descriptor 2: route it to a temporary file."""

    def __enter__(self):
        sys.stderr.flush()
        self.f = tempfile.TemporaryFile(mode="w+")
        self.saved = os.dup(2)
        os.dup2(self.f.fileno(), 2)
        return self

    def __exit__(self, *exc):
        os.dup2(self.saved, 2)
        os.close(self.saved)
        self.f.seek(0)
        self.text = self.f.read()
        self.f.close()


def ba_main(a, gpu_info):
    from sim3opt_b200 import synth
    from test_ba_marginals_host import ba_fixings, hessian_indices, point_observations
    from test_gpu_ba_marginals import make_ba
    graphs = {"ba_small": synth.ba_loop(24, 300, 5, seed=11), "ba_medium": synth.ba_loop(120, 6000, 8, seed=5),
              "ba_bench": synth.ba_loop(1000, 500000, 10, seed=42)}
    names = ["linearize", "schur", "factor", "selinv", "points", "gather"]
    for name, g in graphs.items():
        cf, pf = ba_fixings(g)
        ch, ph = hessian_indices(cf, pf)
        products = int(sum(len(k) ** 2 for k in point_observations(g, ch, ph)))
        p = make_ba(g, cf, pf)
        reps = a.reps if name != "ba_bench" else max(3, a.reps // 5)
        for _ in range(a.warmup):
            p.ba_marginals()
        wall = []
        with StderrCapture() as cap:
            for _ in range(reps):
                t0 = time.perf_counter()
                p.ba_marginals()
                wall.append(time.perf_counter() - t0)
        phases = np.array([[float(x) for x in line.split()[2:13:2]] for line in cap.text.splitlines()
                           if line.startswith("s3o_ba_compute_marginals:")])
        assert len(phases) == reps, cap.text[-2000:]
        med = np.median(phases, 0)
        st = p.stats()
        rec = {"graph": name, "free_cameras": p.ncf, "free_points": p.npf, "schur_blocks": p.nb,
               "factor_levels": st["direct_levels"], "factor_blocks": st["direct_blocks"], "point_products": products}
        rec.update({"ms_" + n: float(v) for n, v in zip(names, med)})
        rec.update(ms_call_wall=1e3 * float(np.median(wall)), reps=reps, gpu=gpu_info[:1])
        print(json.dumps(rec), flush=True)


def pcg_main(gpu_info):
    import re
    from conftest import make_gpu
    from sim3opt_b200 import synth
    col_re = re.compile(r"column (\d+) \(vertex \d+\): PCG iterations ([\d ]+), refinement rounds (\d+), true residual ([^,\s]+), backward error (\S+)")
    for name, laps in (("s100k", 100), ("S1M", 1000)):
        g = synth.sphere(laps, 1000, seed=42)
        p = make_gpu(g, jac=1)
        p.build_structure()
        nf = p.num_free

        def call(cols):
            pairs = np.array([(c, c) for c in cols] + [((c + nf // 2) % nf, c) for c in cols], np.int32)
            with StderrCapture() as cap:
                t0 = time.perf_counter()
                p.marginals(pairs)
                wall = time.perf_counter() - t0
            cols_out = [m.groups() for m in col_re.finditer(cap.text)]
            phase = [line for line in cap.text.splitlines() if line.startswith("s3o_compute_marginals: linearize")][-1]
            ms = [float(x) for x in phase.split()[2:9:2]]
            its = [int(x) for c in cols_out for x in c[1].split()]
            return {"columns": len(cols), "ms_call_wall": 1e3 * wall, "ms_wall_per_column": 1e3 * wall / len(cols),
                    "ms_linearize": ms[0], "ms_precond": ms[1], "ms_solves_per_column": ms[2] / len(cols),
                    "pcg_iters_per_rhs_mean": float(np.mean(its)), "pcg_iters_per_rhs_max": int(np.max(its)),
                    "refinement_rounds_max": max(int(c[2]) for c in cols_out),
                    "true_residual_max": max(float(c[3]) for c in cols_out),
                    "backward_error_max": max(float(c[4]) for c in cols_out)}

        rng = np.random.default_rng(1)
        rec = {"graph": name, "free": nf, "gpu": gpu_info[:1]}
        rec["first_call"] = call([nf - 1])          # includes the forced-cap plan analysis
        for k in (1, 2, 8):
            rec[f"cols_{k}"] = call(sorted(rng.choice(nf, k, replace=False).tolist()))
        print(json.dumps(rec), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--ba", action="store_true")
    ap.add_argument("--pcg", action="store_true")
    a = ap.parse_args()
    import sim3opt_b200 as s3
    from conftest import make_gpu, make_oracle
    from test_gpu_parity import dense_from_blocks
    gpu_info = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True).stdout.strip().splitlines()
    if a.ba:
        return ba_main(a, gpu_info)
    if a.pcg:
        return pcg_main(gpu_info)
    for name, g in graphs().items():
        plan = s3.host_direct_plan(len(g["est"]), g["fixed"], g["v0"], g["v1"], max_pairs=60000000)
        p = make_gpu(g, jac=1)
        for _ in range(a.warmup):
            p.marginals()
        wall = []
        with StderrCapture() as cap:
            for _ in range(a.reps):
                t0 = time.perf_counter()
                p.marginals()
                wall.append(time.perf_counter() - t0)
        phases = np.array([[float(x) for x in line.split()[2:9:2]] for line in cap.text.splitlines()
                           if line.startswith("s3o_compute_marginals:")])
        assert len(phases) == a.reps, cap.text[-2000:]
        med = np.median(phases, 0)
        rec = {"graph": name, "free": plan["n"], "rounds": plan["rounds"], "blocks_L": len(plan["brow"]),
               "factor_products": plan["n_pairs"], "selinv_products": 2 * plan["n_pairs"],
               "ms_linearize": med[0], "ms_factor": med[1], "ms_selinv": med[2], "ms_gather": med[3],
               "ms_call_wall": 1e3 * float(np.median(wall)), "reps": a.reps, "gpu": gpu_info[:1]}
        if name in ("K1", "K118"):          # reference, not a target: the oracle's H and a dense LAPACK inverse
            o = make_oracle(g, jac=1)
            cp, ri = o.build_structure()
            ts = []
            for _ in range(5):
                t0 = time.perf_counter()
                H, _ = o.linearize()
                np.linalg.inv(dense_from_blocks(cp, ri, H, 7))
                ts.append(time.perf_counter() - t0)
            rec["ms_cpu_oracle_dense_inverse"] = 1e3 * float(np.median(ts))
        print(json.dumps(rec), flush=True)


if __name__ == "__main__":
    main()
