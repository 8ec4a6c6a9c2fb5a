#!/usr/bin/env python
"""What building K objects' scene clouds in one call saves (stocs_b200_build_scene_clouds, csrc/scene_cloud.cu).

1. On the YCB frame with K = 1, 2, 4 and 8 maps derived from the frame's own (the map, its complement, the
   map shifted, a constant map, the map at other thresholds, ...): K calls of build_scene_cloud against one
   call of build_scene_clouds, the two alternating; both must give the same arrays.
2. With --parent-lib <libstocs_b200.so of another build>: the single-object call of that build against this
   one, alternating, in the same process.

Host wall clock around calls that end in a device synchronise, after a warm-up; best of 3 per repetition,
median over 20 repetitions.  The card's name, power limit and maximum SM clock are read in the same run.
    python profiles/multi_object_cloud.py [--parent-lib PATH] [--out out.json]
(default output: profiles/r06_multi_object_cloud.json)"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import model_matching_b200._capi as capi  # noqa: E402

D = os.path.join(ROOT, "tests", "golden", "examples", "ycb")
K_CAM = [1066.778, 312.986, 1067.487, 241.310]
SCALE, VOXEL = 1 / 10000.0, 0.005
REPS, BEST_OF = 20, 3


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True)
    except OSError:
        return "unknown"
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def ycb_frame():
    import cv2
    depth = cv2.imread(os.path.join(D, "depth.png"), cv2.IMREAD_UNCHANGED)
    bgr = cv2.imread(os.path.join(D, "rgb.png"), cv2.IMREAD_COLOR)
    prob = cv2.imread(os.path.join(D, "probability_maps", "024_bowl.png"), cv2.IMREAD_UNCHANGED)
    p = prob.astype(np.int64)
    maps = np.stack([p, 10000 - np.clip(p, 0, 10000), np.roll(p, (9, -13), axis=(0, 1)), np.full_like(p, 1000),
                     p, np.roll(p, (-20, 31), axis=(0, 1)), 10000 - np.clip(p, 0, 10000), p]).astype(np.uint16)
    thr = np.array([0.10, 0.30, 0.20, 0.10, 0.50, 0.10, 0.60, 0.90], np.float32)
    return depth, bgr, maps, thr


def timed(fn):
    best = 1e9
    for _ in range(BEST_OF):
        t0 = time.perf_counter()
        out = fn()
        best = min(best, time.perf_counter() - t0)
    return best, out


def same(a, b):
    return len(a) == len(b) and all(all(np.array_equal(x[k], y[k]) for k in x) for x, y in zip(a, b))


def multi_vs_singles(ctx, depth, bgr, maps, thr):
    res = []
    for k in (1, 2, 4, 8):
        m, t = maps[:k], thr[:k]

        def singles():
            return [ctx.build_scene_cloud(depth, bgr, m[i], None, K_CAM, SCALE, VOXEL, float(t[i])) for i in range(k)]

        def multi():
            return ctx.build_scene_clouds(depth, bgr, m, None, K_CAM, SCALE, VOXEL, t)

        singles(); multi()                     # warm-up: module loads, buffer growth, read-back estimate
        ts, tm, ok = [], [], True
        for _ in range(REPS):
            a, ra = timed(singles)
            b, rb = timed(multi)
            ts.append(a); tm.append(b)
            ok = ok and same(ra, rb)
        ms, mm = 1e3 * float(np.median(ts)), 1e3 * float(np.median(tm))
        res.append({"K": k, "points_per_object": [len(c["pos"]) for c in rb], "k_single_calls_ms_median": ms,
                    "one_multi_call_ms_median": mm, "saved_ms": ms - mm, "speedup": ms / mm,
                    "k_single_calls_ms_spread": [1e3 * float(np.min(ts)), 1e3 * float(np.max(ts))],
                    "one_multi_call_ms_spread": [1e3 * float(np.min(tm)), 1e3 * float(np.max(tm))],
                    "same_arrays": bool(ok)})
    return res


def other_build_context(path):
    """A Context whose build_scene_cloud calls the libstocs_b200.so at `path` (which may predate other calls)."""
    L, cur = C.CDLL(os.path.abspath(path)), capi.lib()
    for name in ("stocs_b200_create", "stocs_b200_destroy", "stocs_b200_last_error", "stocs_b200_build_scene_cloud"):
        getattr(L, name).argtypes, getattr(L, name).restype = getattr(cur, name).argtypes, getattr(cur, name).restype
    c = capi.Context.__new__(capi.Context)
    c._L, c.h = L, C.c_void_p()
    if L.stocs_b200_create(C.byref(c.h), 0) != 0:
        raise capi.StocsError("stocs_b200_create failed in " + path)
    return c


def single_ab(ctx, parent_lib, depth, bgr, maps, thr):
    pctx = other_build_context(parent_lib)
    try:
        def run(c):
            return [c.build_scene_cloud(depth, bgr, maps[0], None, K_CAM, SCALE, VOXEL, float(thr[0]))]
        run(ctx); run(pctx)
        tt, tp, ok = [], [], True
        for _ in range(REPS):
            a, ra = timed(lambda: run(ctx))
            b, rb = timed(lambda: run(pctx))
            tt.append(a); tp.append(b)
            ok = ok and same(ra, rb)
    finally:
        pctx.close()
    return {"this_build_ms_median": 1e3 * float(np.median(tt)), "parent_build_ms_median": 1e3 * float(np.median(tp)),
            "this_build_ms_spread": [1e3 * float(np.min(tt)), 1e3 * float(np.max(tt))],
            "parent_build_ms_spread": [1e3 * float(np.min(tp)), 1e3 * float(np.max(tp))],
            "points": len(ra[0]["pos"]), "same_arrays": bool(ok)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", help="libstocs_b200.so of the build to compare the single-object call with")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_multi_object_cloud.json"))
    args = ap.parse_args()
    depth, bgr, maps, thr = ycb_frame()
    res = {"card": card(), "frame": "examples/ycb (640x480), 024_bowl map and maps derived from it, no edge map",
           "voxel_size": VOXEL, "thresholds": [float(v) for v in thr],
           "method": "host wall clock around calls that end in a synchronise; warm-up first; the two ways alternate, "
                     "best of %d per repetition, median over %d repetitions" % (BEST_OF, REPS)}
    ctx = capi.Context(0)
    try:
        res["multi_vs_singles"] = multi_vs_singles(ctx, depth, bgr, maps, thr)
        if args.parent_lib:
            res["single_object_call_vs_parent"] = single_ab(ctx, args.parent_lib, depth, bgr, maps, thr)
    finally:
        ctx.close()
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
