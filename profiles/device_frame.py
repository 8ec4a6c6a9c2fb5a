#!/usr/bin/env python
"""What building and uploading a frame's scene clouds from GPU memory saves (stocs_b200_build_scene_clouds_device +
stocs_b200_upload_scenes_device) against the host chain, for a caller whose frame is already on the GPU.

1. YCB frame, K = 1, 2, 4 and 8 objects (the maps of profiles/multi_object_cloud.py; models 024_bowl, obj_06 and dove
   round-robin, one context per object), 100 bases, at most 200 sets:
   host chain:   numpy depth, BGR and uint16 maps -> build_scene_clouds -> upload_scenes -> run_pipelines;
   device chain: the same frame already in CUDA tensors -> build_scene_clouds_device -> upload_scenes (device
                 clouds) -> run_pipelines.
   Each call is also timed on its own.  Both chains must give the same clouds and the same pipeline results.
2. With --parent-lib <libstocs_b200.so of another build>: build_scene_clouds and upload_scenes (K = 1 and 8) of that
   build against this one, alternating, in the same process: the host calls must be unchanged.

Host wall clock around calls that end in a device synchronise, after a warm-up; the two ways alternate, best of 3 per
repetition, median over 20 repetitions.  The card's name, power limit and maximum SM clock are read in the same run.
    python profiles/device_frame.py [--parent-lib PATH] [--out out.json]
(default output: profiles/r08_device_frame.json)"""
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
from multi_object_cloud import K_CAM, SCALE, card, ycb_frame  # noqa: E402
from multi_object_pose import contexts  # noqa: E402

N_BASES, MAX_SETS, VOXEL = 100, 200, 0.005
REPS, BEST_OF = 20, 3


def timed(fn):
    best, out = 1e9, None
    for _ in range(BEST_OF):
        t0 = time.perf_counter()
        out = fn()
        best = min(best, time.perf_counter() - t0)
    return best, out


def alternate(a, b, same):
    """a and b warmed up, then alternated: -> (medians, spreads, every pair of results equal)"""
    ra, rb = a(), b()
    ok = same(ra, rb)
    ta, tb = [], []
    for _ in range(REPS):
        x, ra = timed(a)
        y, rb = timed(b)
        ta.append(x); tb.append(y)
        ok = ok and same(ra, rb)
    ms = lambda t: 1e3 * float(np.median(t))   # noqa: E731
    return {"host_ms_median": ms(ta), "device_ms_median": ms(tb), "saved_ms": ms(ta) - ms(tb),
            "host_ms_spread": [1e3 * min(ta), 1e3 * max(ta)], "device_ms_spread": [1e3 * min(tb), 1e3 * max(tb)],
            "same_results": bool(ok)}


def same_clouds(host, dev):
    return len(host) == len(dev) and all(h[k].tobytes() == d[k].cpu().numpy().tobytes() for h, d in zip(host, dev) for k in h)


def case(k, depth, bgr, maps, thr, dframe):
    import torch
    m, t = maps[:k], thr[:k]
    seeds = [1000 + 7 * i for i in range(k)]
    dd, db, dm = dframe[0], dframe[1], dframe[2][:k]
    hc, dc = contexts(k, None), contexts(k, None)
    bh, bd = capi.Context(0), capi.Context(0)   # the frame-side contexts of the two ways

    def build_host():
        return bh.build_scene_clouds(depth, bgr, m, None, K_CAM, SCALE, VOXEL, t)

    def build_dev():
        return bd.build_scene_clouds_device(dd, db, dm, None, K_CAM, SCALE, VOXEL, t)

    def chain(build, ctxs):
        clouds = build()
        capi.upload_scenes(ctxs, clouds)
        return clouds, [bytes(r) for r in capi.run_pipelines(ctxs, seeds, N_BASES, MAX_SETS)]

    try:
        res = {"K": k}
        res["chain"] = alternate(lambda: chain(build_host, hc), lambda: chain(build_dev, dc),
                                 lambda a, b: same_clouds(a[0], b[0]) and a[1] == b[1])
        res["points_per_object"] = [len(c["pos"]) for c in build_host()]
        res["build_scene_clouds"] = alternate(build_host, build_dev, same_clouds)
        hcl, dcl = build_host(), build_dev()
        res["upload_scenes"] = alternate(lambda: capi.upload_scenes(hc, hcl), lambda: capi.upload_scenes(dc, dcl),
                                         lambda a, b: [c.centred()[0].tobytes() for c in hc] == [c.centred()[0].tobytes() for c in dc])
        res["run_pipelines"] = alternate(lambda: [bytes(r) for r in capi.run_pipelines(hc, seeds, N_BASES, MAX_SETS)],
                                         lambda: [bytes(r) for r in capi.run_pipelines(dc, seeds, N_BASES, MAX_SETS)],
                                         lambda a, b: a == b)
        torch.cuda.synchronize()
    finally:
        for c in hc + dc + [bh, bd]:
            c.close()
    return res


def other_build(path):
    """The libstocs_b200.so at `path`, with the argument types of this build's calls."""
    L, cur = C.CDLL(os.path.abspath(path)), capi.lib()
    for name in ("stocs_b200_create", "stocs_b200_destroy", "stocs_b200_last_error", "stocs_b200_build_scene_clouds",
                 "stocs_b200_upload_scenes", "stocs_b200_get_centred"):
        getattr(L, name).argtypes, getattr(L, name).restype = getattr(cur, name).argtypes, getattr(cur, name).restype
    return L


def parent_ab(parent_lib, depth, bgr, maps, thr):
    """build_scene_clouds and upload_scenes straight through the C ABI of either build"""
    builds = {"this": capi.lib(), "parent": other_build(parent_lib)}
    H, W = depth.shape
    out = {}
    for k in (1, 8):
        m, t = np.ascontiguousarray(maps[:k]), np.ascontiguousarray(thr[:k])
        cap = k * H * W
        ctxs = {}
        for name, L in builds.items():
            hs = []
            for _ in range(k + 1):
                h = C.c_void_p()
                assert L.stocs_b200_create(C.byref(h), 0) == 0
                hs.append(h)
            ctxs[name] = hs

        def build(name):
            L, h = builds[name], ctxs[name][0]
            a = dict(pos=np.empty((cap, 3), np.float32), nrm=np.empty((cap, 3), np.float32), rgb=np.empty((cap, 3), np.float32),
                     pix=np.empty((cap, 2), np.int32), cls=np.empty(cap, np.float32), edge=np.empty(cap, np.float32))
            offs = np.zeros(k + 1, np.int64)
            p = capi._ptr
            assert L.stocs_b200_build_scene_clouds(h, p(depth), p(bgr), p(m), p(t), k, None, W, H, *K_CAM, SCALE, VOXEL,
                                                   p(a["pos"]), p(a["nrm"]), p(a["rgb"]), p(a["pix"]), p(a["cls"]), p(a["edge"]),
                                                   cap, p(offs)) == 0
            n = int(offs[-1])
            return {key: v[:n].tobytes() for key, v in a.items()}, offs

        built, offs = build("this")
        arrays = {key: np.frombuffer(v, np.int32 if key == "pix" else np.float32).copy() for key, v in built.items()}

        def upload(name):
            L, hs = builds[name], ctxs[name][1:]
            p = capi._ptr
            handles = (C.c_void_p * k)(*[h.value for h in hs])
            assert L.stocs_b200_upload_scenes(handles, k, p(arrays["pos"]), p(arrays["nrm"]), p(arrays["cls"]), p(arrays["pix"]),
                                              p(offs)) == 0
            res = []
            for i, h in enumerate(hs):
                c = np.empty((int(offs[i + 1] - offs[i]), 3), np.float32)
                if len(c):
                    assert L.stocs_b200_get_centred(h, p(c), None) == 0
                res.append(c.tobytes())
            return res

        try:
            out[f"K{k}"] = {"build_scene_clouds": alternate(lambda: build("this")[0], lambda: build("parent")[0], lambda a, b: a == b),
                            "upload_scenes": alternate(lambda: upload("this"), lambda: upload("parent"), lambda a, b: a == b)}
        finally:
            for name, hs in ctxs.items():
                for h in hs:
                    builds[name].stocs_b200_destroy(h)
        for call in out[f"K{k}"].values():   # here "host" is this build and "device" the parent build
            call["this_build_ms_median"] = call.pop("host_ms_median")
            call["parent_build_ms_median"] = call.pop("device_ms_median")
            call["this_build_ms_spread"] = call.pop("host_ms_spread")
            call["parent_build_ms_spread"] = call.pop("device_ms_spread")
            call["this_minus_parent_ms"] = -call.pop("saved_ms")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", help="libstocs_b200.so of the build to compare the host calls with")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_device_frame.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("device_frame.py measures on the GPU; none is visible")
    depth, bgr, maps, thr = ycb_frame()
    dframe = (torch.from_numpy(depth).cuda(), torch.from_numpy(bgr).cuda(), torch.from_numpy(maps).cuda())
    res = {"card": card(),
           "frame": "examples/ycb (640x480): the eight maps of profiles/multi_object_cloud.py, no edge map",
           "pipeline": {"n_bases": N_BASES, "max_sets": MAX_SETS, "models": "024_bowl, obj_06, dove round-robin"},
           "method": "host wall clock around calls that end in a synchronise; warm-up first; the host and the device way "
                     "alternate, best of %d per repetition, median over %d repetitions; the device way's frame is in CUDA "
                     "tensors before timing, its clouds stay CUDA tensors" % (BEST_OF, REPS)}
    res["cases"] = [case(k, depth, bgr, maps, thr, dframe) for k in (1, 2, 4, 8)]
    if args.parent_lib:
        res["host_calls_vs_parent"] = parent_ab(args.parent_lib, depth, bgr, maps, thr)
    res["card_after"] = card()
    bad = [c["K"] for c in res["cases"] for key in ("chain", "build_scene_clouds", "upload_scenes", "run_pipelines")
           if not c[key]["same_results"]]
    bad += [k for k, v in res.get("host_calls_vs_parent", {}).items() for c in v.values() if not c["same_results"]]
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))
    assert not bad, f"results differ: {bad}"


if __name__ == "__main__":
    main()
