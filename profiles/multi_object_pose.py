#!/usr/bin/env python
"""What giving K objects' scenes and pipelines to their contexts in one call saves (stocs_b200_upload_scenes +
stocs_b200_run_pipelines, one context per object) against the loop of single calls.

1. YCB frame, K = 1, 2, 4 and 8 objects (the clouds of profiles/multi_object_cloud.py's maps; models 024_bowl,
   obj_06 and dove round-robin), 100 bases, at most 200 sets: plain and clustered runs.
2. Packed frame, instance mode with the edge map, K = 1, 2 and 4.
For each case, K x (upload_scene + run_pipeline[_instance][_clustered]) on one set of contexts against
upload_scenes + run_pipelines on a second set, the two alternating; both must give the same results.
3. With --parent-lib <libstocs_b200.so of another build>: upload_scene, run_pipeline and run_pipeline_clustered
   on YCB of that build against this one, alternating, in the same process.

Host wall clock around calls that end in a device synchronise, after a warm-up; best of 3 per repetition,
median over 20 repetitions.  The card's name, power limit and maximum SM clock are read in the same run.
    python profiles/multi_object_pose.py [--parent-lib PATH] [--out out.json]
(default output: profiles/r07_multi_object_pose.json)"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))
import model_matching_b200._capi as capi  # noqa: E402
from multi_object_cloud import K_CAM, card, ycb_frame  # noqa: E402

G = os.path.join(ROOT, "tests", "golden")
PACKED = os.path.join(G, "examples", "packed")
PACKED_K = [615.957763671875, 308.1098937988281, 615.9578247070312, 246.33352661132812]
MODELS = ("ycb", "linemod", "packed")     # 024_bowl, obj_06, dove
N_BASES, MAX_SETS, VOXEL = 100, 200, 0.005
REPS, BEST_OF = 20, 3
CLUSTER = dict(acceptable_fraction=0.3, maximum_pose_count=10, min_distance=0.03, min_angle=15.0)
SYMS = ((0, 0, 0), (0, 0, 360), (180, 0, 90))


def model(k):
    g = np.load(os.path.join(G, f"golden_{MODELS[k % 3]}.npz"))
    return g["mpos"], g["mnrm"]


def timed(fn):
    best = 1e9
    for _ in range(BEST_OF):
        t0 = time.perf_counter()
        out = fn()
        best = min(best, time.perf_counter() - t0)
    return best, out


def ycb_clouds():
    depth, bgr, maps, thr = ycb_frame()
    c = capi.Context(0)
    try:
        return c.build_scene_clouds(depth, bgr, maps, None, K_CAM, 1 / 10000.0, VOXEL, thr), None
    finally:
        c.close()


def packed_clouds():
    import cv2
    depth = cv2.imread(os.path.join(PACKED, "depth.png"), cv2.IMREAD_UNCHANGED)
    bgr = cv2.imread(os.path.join(PACKED, "rgb.png"), cv2.IMREAD_COLOR)
    prob = cv2.imread(os.path.join(PACKED, "probability_maps", "dove.png"), cv2.IMREAD_UNCHANGED).astype(np.int64)
    edge = cv2.imread(os.path.join(PACKED, "probability_maps", "edge.png"), cv2.IMREAD_GRAYSCALE)
    maps = np.stack([prob, np.roll(prob, (9, -13), axis=(0, 1)), prob, np.roll(prob, (-20, 31), axis=(0, 1))]).astype(np.uint16)
    thr = np.array([0.10, 0.20, 0.50, 0.10], np.float32)
    c = capi.Context(0)
    try:
        return c.build_scene_clouds(depth, bgr, maps, edge, PACKED_K, 1 / 8000.0, VOXEL, thr), edge
    finally:
        c.close()


def contexts(k, edge):
    out = []
    for i in range(k):
        c = capi.Context(0)
        c.upload_model(*model(i))
        if edge is not None:
            c.upload_edge_map(edge)
        out.append(c)
    return out


def frame_serial(ctxs, clouds, seeds, instance, cluster):
    res = []
    for i, (c, cl) in enumerate(zip(ctxs, clouds)):
        c.upload_scene(cl["pos"], cl["nrm"], cl["cls"], cl["pix"])
        if cluster is None:
            r = c.run_pipeline_instance(seeds[i], N_BASES, MAX_SETS, 0.9) if instance else c.run_pipeline(seeds[i], N_BASES, MAX_SETS)
            res.append(bytes(r))
        else:
            fn = c.run_pipeline_instance_clustered if instance else c.run_pipeline_clustered
            r, p = fn(seeds[i], N_BASES, MAX_SETS, 0.9, **cluster[i]) if instance else fn(seeds[i], N_BASES, MAX_SETS, **cluster[i])
            res.append(bytes(r) + p.tobytes())
    return res


def frame_batched(ctxs, clouds, seeds, instance, cluster):
    capi.upload_scenes(ctxs, clouds)
    out = capi.run_pipelines(ctxs, seeds, N_BASES, MAX_SETS, instance=instance, cluster=cluster)
    return [bytes(r) if cluster is None else bytes(r[0]) + r[1].tobytes() for r in out]


def case(clouds, edge, k, instance, clustered):
    cl, seeds = clouds[:k], [1000 + 7 * i for i in range(k)]
    cluster = [dict(CLUSTER, sym_info=SYMS[i % 3]) for i in range(k)] if clustered else None
    a, b = contexts(k, edge), contexts(k, edge)
    try:
        frame_serial(a, cl, seeds, instance, cluster); frame_batched(b, cl, seeds, instance, cluster)   # warm-up
        ts, tb, ok = [], [], True
        for _ in range(REPS):
            x, rx = timed(lambda: frame_serial(a, cl, seeds, instance, cluster))
            y, ry = timed(lambda: frame_batched(b, cl, seeds, instance, cluster))
            ts.append(x); tb.append(y)
            ok = ok and rx == ry
    finally:
        for c in a + b:
            c.close()
    ms, mb = 1e3 * float(np.median(ts)), 1e3 * float(np.median(tb))
    return {"K": k, "instance": instance, "clustered": clustered, "points_per_object": [len(c["pos"]) for c in cl],
            "serial_loop_ms_median": ms, "batched_ms_median": mb, "saved_ms": ms - mb, "speedup": ms / mb,
            "serial_loop_ms_spread": [1e3 * float(np.min(ts)), 1e3 * float(np.max(ts))],
            "batched_ms_spread": [1e3 * float(np.min(tb)), 1e3 * float(np.max(tb))], "same_results": bool(ok)}


def other_build_context(path):
    """A Context whose calls go to the libstocs_b200.so at `path`."""
    L, cur = C.CDLL(os.path.abspath(path)), capi.lib()
    for name in ("stocs_b200_create", "stocs_b200_destroy", "stocs_b200_last_error", "stocs_b200_set_params",
                 "stocs_b200_upload_model", "stocs_b200_upload_scene", "stocs_b200_run_pipeline",
                 "stocs_b200_run_pipeline_clustered"):
        getattr(L, name).argtypes, getattr(L, name).restype = getattr(cur, name).argtypes, getattr(cur, name).restype
    c = capi.Context.__new__(capi.Context)
    c._L, c.h, c.M, c.S, c._last_H = L, C.c_void_p(), 0, 0, 0
    if L.stocs_b200_create(C.byref(c.h), 0) != 0:
        raise capi.StocsError("stocs_b200_create failed in " + path)
    return c


def single_ab(parent_lib, clouds):
    cl = clouds[0]
    this, parent = capi.Context(0), other_build_context(parent_lib)
    calls = {
        "upload_scene": lambda c: (c.upload_scene(cl["pos"], cl["nrm"], cl["cls"], cl["pix"]), b"")[1],
        "run_pipeline": lambda c: bytes(c.run_pipeline(1000, N_BASES, MAX_SETS)),
        "run_pipeline_clustered": lambda c: (lambda r: bytes(r[0]) + r[1].tobytes())(
            c.run_pipeline_clustered(1000, N_BASES, MAX_SETS, **CLUSTER)),
    }
    out = {}
    try:
        for c in (this, parent):
            c.upload_model(*model(0))
            c.upload_scene(cl["pos"], cl["nrm"], cl["cls"], cl["pix"])
        for name, fn in calls.items():
            fn(this); fn(parent)
            tt, tp, ok = [], [], True
            for _ in range(REPS):
                a, ra = timed(lambda: fn(this))
                b, rb = timed(lambda: fn(parent))
                tt.append(a); tp.append(b)
                ok = ok and ra == rb
            out[name] = {"this_build_ms_median": 1e3 * float(np.median(tt)), "parent_build_ms_median": 1e3 * float(np.median(tp)),
                         "this_build_ms_spread": [1e3 * float(np.min(tt)), 1e3 * float(np.max(tt))],
                         "parent_build_ms_spread": [1e3 * float(np.min(tp)), 1e3 * float(np.max(tp))],
                         "same_results": bool(ok)}
    finally:
        this.close(); parent.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", help="libstocs_b200.so of the build to compare the single calls with")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_multi_object_pose.json"))
    args = ap.parse_args()
    res = {"card": card(),
           "frames": "examples/ycb (640x480): the eight maps of profiles/multi_object_cloud.py, class mode; "
                     "examples/packed: the dove map, shifted and at other thresholds, instance mode with the edge map",
           "pipeline": {"n_bases": N_BASES, "max_sets": MAX_SETS, "cluster": CLUSTER, "models": "024_bowl, obj_06, dove round-robin"},
           "method": "host wall clock around upload + pipeline of every object (each call ends in a synchronise); warm-up "
                     "first; the serial loop and the batched calls alternate, best of %d per repetition, median over %d "
                     "repetitions" % (BEST_OF, REPS)}
    ycb, _ = ycb_clouds()
    packed, edge = packed_clouds()
    res["ycb"] = [case(ycb, None, k, False, c) for c in (False, True) for k in (1, 2, 4, 8)]
    res["packed_instance"] = [case(packed, edge, k, True, False) for k in (1, 2, 4)]
    if args.parent_lib:
        res["single_calls_vs_parent"] = single_ab(args.parent_lib, ycb)
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
