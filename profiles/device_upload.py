#!/usr/bin/env python
"""What planning a device upload on the device saves: stocs_b200_upload_scenes_device of this build (centroid, box,
class-weight bound and pixel range reduced on the device, one 64-byte read-back per context, the reference kd-tree
built on the device) against the parent build given with --parent-lib (every slice's positions, weights and pixels
copied to the host, host plan, kd-tree on a host thread), in the same process.

YCB frame, K = 1, 2, 4 and 8 objects (the maps of profiles/multi_object_cloud.py; models 024_bowl, obj_06 and dove
round-robin, one context per object), 100 bases, at most 200 sets:
  upload: upload_scenes_device alone, on device clouds built once (returns when every grid index is complete; the
          kd-tree of either build is still pending then, and joined by the first scoring launch);
  chain:  build_scene_clouds_device -> upload_scenes_device -> run_pipelines, the frame in CUDA tensors.
The two builds alternate, best of 3 per repetition, median over 20 repetitions (host wall clock around calls that end
in a device synchronise, after a warm-up); the results of the two builds must be identical.  A last pass profiles
this build's K = 1 upload with torch.profiler: device time by kernel and every device-to-host copy.  The card's name,
power limit and maximum SM clock are read in the same run.
    python profiles/device_upload.py --parent-lib PATH [--out out.json]
(default output: profiles/r10_device_upload.json)"""
import argparse
import contextlib
import ctypes as C
import json
import os
import sys
import tempfile
import time
from collections import defaultdict

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))
import model_matching_b200._capi as capi  # noqa: E402
from multi_object_cloud import K_CAM, SCALE, card, ycb_frame  # noqa: E402
from multi_object_pose import contexts  # noqa: E402

N_BASES, MAX_SETS, VOXEL = 100, 200, 0.005
REPS, BEST_OF = 20, 3


def other_build(path):
    """The libstocs_b200.so at `path`, with the argument types of this build's calls (those it exports)."""
    L, cur = C.CDLL(os.path.abspath(path)), capi.lib()
    for name in capi.SYMBOLS:
        if hasattr(L, name):
            getattr(L, name).argtypes, getattr(L, name).restype = getattr(cur, name).argtypes, getattr(cur, name).restype
    return L


@contextlib.contextmanager
def using(L):
    """capi's module-level calls and new Contexts go to L inside the block"""
    prev = capi._LIB
    capi._LIB = L
    try:
        yield
    finally:
        capi._LIB = prev


def timed(fn):
    best = 1e9
    for _ in range(BEST_OF):
        t0 = time.perf_counter()
        fn()
        best = min(best, time.perf_counter() - t0)
    return best


def alternate(fns):
    """{name: fn} warmed up, then alternated -> medians and spreads in ms"""
    for fn in fns.values():
        fn()
    t = {name: [] for name in fns}
    for _ in range(REPS):
        for name, fn in fns.items():
            t[name].append(timed(fn))
    out = {f"{name}_ms_median": 1e3 * float(np.median(v)) for name, v in t.items()}
    out.update({f"{name}_ms_spread": [1e3 * min(v), 1e3 * max(v)] for name, v in t.items()})
    out["this_minus_parent_ms"] = out["this_ms_median"] - out["parent_ms_median"]
    return out


def case(k, builds, dframe, thr):
    import torch
    seeds = [1000 + 7 * i for i in range(k)]
    dd, db, dm = dframe[0], dframe[1], dframe[2][:k]
    t = thr[:k]
    ctxs, fctx = {}, {}
    for name, L in builds.items():
        with using(L):
            ctxs[name], fctx[name] = contexts(k, None), capi.Context(0)
    clouds = fctx["this"].build_scene_clouds_device(dd, db, dm, None, K_CAM, SCALE, VOXEL, t)
    torch.cuda.synchronize()

    def upload(name):
        def fn():
            with using(builds[name]):
                capi.upload_scenes(ctxs[name], clouds)
        return fn

    def chain(name, out=None):
        def fn():
            with using(builds[name]):
                cl = fctx[name].build_scene_clouds_device(dd, db, dm, None, K_CAM, SCALE, VOXEL, t)
                capi.upload_scenes(ctxs[name], cl)
                res = [bytes(r) for r in capi.run_pipelines(ctxs[name], seeds, N_BASES, MAX_SETS)]
            if out is not None:
                out.append(res)
        return fn

    def state(name):
        with using(builds[name]):
            return [(c.counters()[[2, 3, 6]].tolist(), c.centroids()[0].tobytes(), c.centred()[0].tobytes()) if c.S else None
                    for c in ctxs[name]]

    try:
        res = {"K": k, "points_per_object": [len(c["pos"]) for c in clouds]}
        res["upload_scenes_device"] = alternate({"this": upload("this"), "parent": upload("parent")})
        res["upload_scenes_device"]["same_results"] = state("this") == state("parent")
        got = {"this": [], "parent": []}
        res["chain"] = alternate({name: chain(name, got[name]) for name in builds})
        res["chain"]["same_results"] = got["this"] == got["parent"] and state("this") == state("parent")
        torch.cuda.synchronize()
    finally:
        for name, L in builds.items():
            with using(L):
                for c in ctxs[name] + [fctx[name]]:
                    c.close()
    return res


def profile_k1(dframe, thr, n=10):
    """device time by kernel and the device-to-host copies of n K = 1 uploads of this build"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    ctxs, f = contexts(1, None), capi.Context(0)
    try:
        clouds = f.build_scene_clouds_device(dframe[0], dframe[1], dframe[2][:1], None, K_CAM, SCALE, VOXEL, thr[:1])
        capi.upload_scenes(ctxs, clouds)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            for _ in range(n):
                capi.upload_scenes(ctxs, clouds)
            torch.cuda.synchronize()
        with tempfile.TemporaryDirectory() as d:
            path = os.path.join(d, "trace.json")
            prof.export_chrome_trace(path)
            with open(path) as fh:
                events = json.load(fh)["traceEvents"]
    finally:
        for c in ctxs + [f]:
            c.close()
    kern = defaultdict(float)
    for e in events:
        if e.get("cat") == "kernel":
            name = e["name"].replace("void ", "").replace("(anonymous namespace)::", "")
            kern[name.split("(")[0].split("<")[0]] += e["dur"] / n
    d2h = [e["args"]["bytes"] for e in events if e.get("cat") == "gpu_memcpy" and "DtoH" in e.get("name", "")]
    return {"uploads": n, "kernel_us_per_upload": dict(sorted(kern.items(), key=lambda kv: -kv[1])),
            "device_to_host_copies_per_upload": len(d2h) / n, "device_to_host_bytes_max": max(d2h) if d2h else 0}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", required=True, help="libstocs_b200.so of the parent build")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_device_upload.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("device_upload.py measures on the GPU; none is visible")
    builds = {"this": capi.lib(), "parent": other_build(args.parent_lib)}
    depth, bgr, maps, thr = ycb_frame()
    dframe = (torch.from_numpy(depth).cuda(), torch.from_numpy(bgr).cuda(), torch.from_numpy(maps).cuda())
    res = {"card": card(),
           "frame": "examples/ycb (640x480): the eight maps of profiles/multi_object_cloud.py, no edge map",
           "pipeline": {"n_bases": N_BASES, "max_sets": MAX_SETS, "models": "024_bowl, obj_06, dove round-robin"},
           "method": "host wall clock around calls that end in a synchronise; warm-up first; this build and the parent "
                     "alternate, best of %d per repetition, median over %d repetitions" % (BEST_OF, REPS)}
    res["cases"] = [case(k, builds, dframe, thr) for k in (1, 2, 4, 8)]
    res["profile_k1_this_build"] = profile_k1(dframe, thr)
    res["card_after"] = card()
    bad = [c["K"] for c in res["cases"] for key in ("upload_scenes_device", "chain") if not c[key]["same_results"]]
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))
    assert not bad, f"results differ: {bad}"


if __name__ == "__main__":
    main()
