#!/usr/bin/env python
"""What greedy pose clustering on the device costs (csrc/cluster.cu).

1. run_pipeline against run_pipeline_clustered on the YCB frame (class mode) and run_pipeline_instance
   against run_pipeline_instance_clustered on `packed` (instance mode), 100 bases, <= 200 sets per base
   as the reference driver runs them; the two calls alternate, seed by seed, after a warm-up.
2. stocs_b200_cluster_poses on 10^4, 10^5 and 10^6 candidates, beside the host shim's greedy loop
   (host/test_clustering bin, which times clustering::greedy_clustering alone) on the same lists.

Host wall clock around calls that end in a device synchronise; the card's name and power limit are read
in the same run.   python profiles/cluster_latency.py [out.json]   (default profiles/r05_cluster_latency.json)"""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from model_matching_b200 import Context, synth  # noqa: E402

G = os.path.join(ROOT, "tests", "golden")
EXE = os.path.join(ROOT, "model_matching_b200", "host", "test_clustering")
PARAMS = dict(acceptable_fraction=0.5, maximum_pose_count=10, min_distance=0.03, min_angle=15.0, sym_info=(0, 0, 0))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def frame(name):
    with np.load(os.path.join(G, f"golden_{name}.npz")) as z:
        return {k: np.ascontiguousarray(z[k]) for k in ("mpos", "mnrm", "spos", "snrm", "scls", "spix")}


def pipeline_pair(ctx, g, instance, seeds=range(2, 22), reps=3):
    edge = None
    if instance:
        import cv2
        edge = cv2.imread(os.path.join(G, "examples", "packed", "probability_maps", "edge.png"), cv2.IMREAD_GRAYSCALE)
    ctx.upload_model(g["mpos"], g["mnrm"])

    def reset():   # instance sampling decays the prior: every timed run starts from the uploaded frame
        ctx.upload_scene(g["spos"], g["snrm"], g["scls"], g["spix"])
        if instance:
            ctx.upload_edge_map(edge)

    def plain(seed):
        return ctx.run_pipeline_instance(seed, 100, 200, 0.9) if instance else ctx.run_pipeline(seed, 100, 200)

    def clustered(seed):
        if instance:
            return ctx.run_pipeline_instance_clustered(seed, 100, 200, 0.9, **PARAMS)
        return ctx.run_pipeline_clustered(seed, 100, 200, **PARAMS)

    reset(); plain(1); reset(); clustered(1)      # warm-up: module loads, buffer growth
    tp, tc, npose, same = [], [], [], True
    for seed in seeds:
        bp = bc = 1e9
        for _ in range(reps):
            reset(); t0 = time.perf_counter(); r0 = plain(seed); bp = min(bp, time.perf_counter() - t0)
            reset(); t0 = time.perf_counter(); r1, poses = clustered(seed); bc = min(bc, time.perf_counter() - t0)
        tp.append(bp); tc.append(bc); npose.append(len(poses))
        same = same and (r0.best_index, r0.best_lcp) == (r1.best_index, r1.best_lcp)
    mp, mc = 1e3 * float(np.median(tp)), 1e3 * float(np.median(tc))
    return {"plain_ms_median": mp, "clustered_ms_median": mc, "clustering_adds_ms": mc - mp,
            "clustered_minus_plain_ms_per_seed": [round(1e3 * (c - p), 4) for p, c in zip(tp, tc)],
            "poses_per_seed": npose, "seeds": len(tp), "best_of_reps": reps, "same_best_pose": bool(same)}


def candidate_list(n, seed=11):
    """fitted-like hypotheses (40 % near the planted poses, LCP above the rest) and uniform clutter"""
    sc = synth.make_scene(n_points=20000, extent=(0.7, 0.5, 0.5), n_objects=5, seed=7)
    mpos, _ = synth.make_model(256)
    T, near = synth.make_hypotheses(n, sc["pos"], mpos, sc["gt_R"], sc["gt_t"], seed=seed, near_fraction=0.4,
                                    max_rot_deg=10.0, max_trans=0.02)
    rng = np.random.default_rng(seed)
    lcp = rng.uniform(0.0, 0.5, n).astype(np.float32)
    lcp[near] += np.float32(0.5)
    return np.ascontiguousarray(T, np.float32).reshape(-1, 16), lcp


def host_loop(T, lcp, best):
    p = PARAMS
    head = (np.array([len(lcp)], np.int64).tobytes() + np.array([p["acceptable_fraction"], best], np.float32).tobytes()
            + np.array([p["maximum_pose_count"]], np.int32).tobytes()
            + np.array([p["min_distance"], p["min_angle"], *p["sym_info"]], np.float32).tobytes())
    r = subprocess.run([EXE, "bin"], input=head + T.tobytes() + lcp.tobytes(), capture_output=True, check=True)
    ms = float(r.stderr.decode().split("greedy_clustering_ms")[1].split()[0])
    return np.array([int(x) for x in r.stdout.split()], np.int64), ms


def cluster_sizes(ctx, sizes=(10 ** 4, 10 ** 5, 10 ** 6), reps=20):
    out = []
    for n in sizes:
        T, lcp = candidate_list(n)
        best = float(lcp.max())
        args = (best, PARAMS["acceptable_fraction"], PARAMS["maximum_pose_count"], PARAMS["min_distance"],
                PARAMS["min_angle"], PARAMS["sym_info"])
        got = ctx.cluster_poses(T, lcp, *args)      # warm-up (scratch growth)
        want, host_ms = host_loop(T, lcp, best)
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter(); ctx.cluster_poses(T, lcp, *args); ts.append(time.perf_counter() - t0)
        out.append({"candidates": n, "above_threshold": int((lcp > np.float32(PARAMS["acceptable_fraction"]) * np.float32(best)).sum()),
                    "poses_kept": int(len(got)), "gpu_call_ms_median": 1e3 * float(np.median(ts)),
                    "gpu_call_ms_min": 1e3 * float(np.min(ts)), "gpu_call_includes": "upload of the poses and LCPs (pageable)",
                    "host_greedy_loop_ms": host_ms, "same_indices_as_host": bool(np.array_equal(got, want))})
    return out


def main():
    dst = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r05_cluster_latency.json")
    res = {"card": card(), "params": PARAMS,
           "method": "host wall clock around calls that end in a synchronise; warm-up first; plain and clustered "
                     "calls alternate per seed, best of 3 per seed, median over seeds"}
    ctx = Context(0)
    try:
        res["ycb_class_mode"] = pipeline_pair(ctx, frame("ycb"), False)
        res["packed_instance_mode"] = pipeline_pair(ctx, frame("packed"), True)
        res["cluster_poses"] = cluster_sizes(ctx)
    finally:
        ctx.close()
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(dst)), exist_ok=True)
    with open(dst, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
