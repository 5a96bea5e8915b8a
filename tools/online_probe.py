"""Cost of growing a built pose graph on the device (s3o_add_vertices / s3o_add_edges + merge) against a fresh set-up.

  python tools/online_probe.py            (a) KITTI-00 K118 replayed key frame by key frame, 100 per merge: per step,
                                              merge + optimize(5) against destroy + create + set + build + optimize(5)
                                              of the same graph; (b) 1000 poses with their edges appended to the s100k
                                              and S1M spheres: the merge, split by S3O_SETUP_TRACE stage, against a
                                              full set-up of the final graph in the same process

Prints the card name and power limit first; needs a GPU.
"""
import os
import re
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def kitti_replay(step=100, iters=5):
    import sim3opt_b200 as s3
    from oracle import kitti_io
    g = kitti_io.build_kitti_sim3_graph(os.path.join(ROOT, "tests", "golden", "kitti00"), use_one_constraint=False)
    n = len(g["est"])
    top = np.maximum(g["v0"], g["v1"])
    p, lo = None, 0
    print(f"(a) K118 replay, {step} key frames per merge, optimize({iters}) after each")
    print("  key frames  edges   merge+opt ms   rebuild+opt ms")
    for hi in list(range(step, n, step)) + [n]:
        eidx = np.nonzero((top >= lo) & (top < hi))[0]
        t0 = time.perf_counter()
        if p is None:
            p = s3.Problem(s3.KIND_SIM3)
            p.set_vertices(g["est"][:hi], g["fixed"][:hi])
            p.set_edges(g["v0"][eidx], g["v1"][eidx], g["meas"][eidx])
            p.build_structure()
        else:
            p.add_vertices(g["est"][lo:hi], g["fixed"][lo:hi])
            p.add_edges(g["v0"][eidx], g["v1"][eidx], g["meas"][eidx])
            p.build_structure()
        est = p.vertices()
        p.optimize(iters)
        t_inc = (time.perf_counter() - t0) * 1e3
        # the same graph from scratch, at the incremental problem's estimates before this step's optimisation (edge
        # order differs from the replay's; the cost does not depend on it)
        sel = np.nonzero(top < hi)[0]
        t0 = time.perf_counter()
        q = s3.Problem(s3.KIND_SIM3)
        q.set_vertices(est, g["fixed"][:hi])
        q.set_edges(g["v0"][sel], g["v1"][sel], g["meas"][sel])
        q.build_structure()
        q.optimize(iters)
        q.close()
        t_new = (time.perf_counter() - t0) * 1e3
        print(f"  {hi:10d} {len(sel):6d} {t_inc:14.2f} {t_new:16.2f}")
        lo = hi


def append_child(laps, add):
    """Runs in a child with S3O_SETUP_TRACE=1: base graph, then the timed merge and the timed full set-up."""
    import sim3opt_b200 as s3
    from sim3opt_b200 import synth
    g = synth.sphere(laps, 1000, seed=42)
    n = len(g["est"])
    top = np.maximum(g["v0"], g["v1"])
    old, new = np.nonzero(top < n - add)[0], np.nonzero(top >= n - add)[0]
    for warm in range(2):       # the first pass warms the kernels and the allocator; the second is reported
        q = s3.Problem(s3.KIND_SIM3)
        q.set_vertices(g["est"][:n - add], g["fixed"][:n - add])
        q.set_edges(g["v0"][old], g["v1"][old], g["meas"][old], g["info"][old])
        q.build_structure()
        print("@@ merge" if warm else "@@ warm", file=sys.stderr, flush=True)
        t0 = time.perf_counter()
        q.add_vertices(g["est"][n - add:], g["fixed"][n - add:])
        q.add_edges(g["v0"][new], g["v1"][new], g["meas"][new], g["info"][new])
        q.build_structure()
        t_merge = (time.perf_counter() - t0) * 1e3
        est = q.vertices()
        q.close()
        print("@@ full" if warm else "@@ warm", file=sys.stderr, flush=True)
        t0 = time.perf_counter()
        r = s3.Problem(s3.KIND_SIM3)
        r.set_vertices(est, g["fixed"])
        r.set_edges(g["v0"], g["v1"], g["meas"], g["info"])
        r.build_structure()
        t_full = (time.perf_counter() - t0) * 1e3
        r.close()
    print(f"RESULT {n} {len(top)} {t_merge:.2f} {t_full:.2f}")


def appends(add=1000):
    print(f"(b) {add} poses with their edges appended; merge (add calls + build) against a full set-up of the final graph")
    for name, laps in (("s100k", 100), ("S1M", 1000)):
        env = dict(os.environ, S3O_SETUP_TRACE="1")
        r = subprocess.run([sys.executable, __file__, "--child", str(laps), str(add)], capture_output=True, text=True, env=env)
        if r.returncode:
            print(r.stdout, r.stderr)
            raise SystemExit(r.returncode)
        n, ne, t_merge, t_full = r.stdout.split("RESULT")[1].split()
        print(f"  {name}: {n} vertices, {ne} edges: merge {t_merge} ms, full set-up {t_full} ms")
        part = r.stderr.split("@@ merge")[-1]
        merge_part, full_part = part.split("@@ full")
        for label, txt in (("merge stages", merge_part), ("full set-up stages", full_part)):
            print(f"    {label}:")
            for m in re.finditer(r"\[s3o setup\] (.*?)\s+([\d.]+) ms", txt):
                print(f"      {m.group(1):34s} {float(m.group(2)):9.1f} ms")


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "--child":
        append_child(int(sys.argv[2]), int(sys.argv[3]))
    else:
        print("card:", card())
        kitti_replay()
        appends()
