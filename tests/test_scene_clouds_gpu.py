"""stocs_b200_build_scene_clouds: the scene clouds of several objects of one frame from one pass over it.
Every object's slice must equal stocs_b200_build_scene_cloud with that object's map and threshold, bit
for bit and in the same order, and at least one object per frame must also equal the CPU oracle."""
import os

import numpy as np
import pytest

import oracle
from model_matching_b200 import Context, StocsError
from model_matching_b200._capi import _ptr

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "examples")
MAX_OBJECTS = 32          # STOCS_B200_MAX_CLOUD_OBJECTS
E_ARG, E_CAPACITY = -1, -5
KEYS = ("pos", "nrm", "rgb", "pix", "cls", "edge")

CASES = {
    "ycb": ("024_bowl", [1066.778, 312.986, 1067.487, 241.310], 1 / 10000.0, False),
    "linemod": ("obj_06", [572.4114, 325.2611, 573.57043, 242.04899], 1 / 1000.0, False),
    "packed": ("dove", [615.957763671875, 308.1098937988281, 615.9578247070312, 246.33352661132812], 1 / 8000.0, True),
}


def _read(scene):
    import cv2
    obj, K, scale, with_edge = CASES[scene]
    d = os.path.join(G, scene)
    depth = cv2.imread(os.path.join(d, "depth.png"), cv2.IMREAD_UNCHANGED)
    bgr = cv2.imread(os.path.join(d, "rgb.png"), cv2.IMREAD_COLOR)
    prob = cv2.imread(os.path.join(d, "probability_maps", obj + ".png"), cv2.IMREAD_UNCHANGED)
    edge = cv2.imread(os.path.join(d, "probability_maps", "edge.png"), cv2.IMREAD_GRAYSCALE) if with_edge else None
    return depth, bgr, prob, edge, K, scale


def _derived(prob):
    """Eight maps from one, with per-object thresholds: the map, its complement (a large cloud), the map
    shifted, an all-zero map (an empty slice between non-empty ones), a constant 1000 at 0.10 (p equal to
    the threshold passes), a constant 999 at 0.10 (drops everything) and one map twice."""
    p = prob.astype(np.int64)
    maps = [p, 10000 - np.clip(p, 0, 10000), np.roll(p, (9, -13), axis=(0, 1)), np.zeros_like(p),
            np.full_like(p, 1000), np.full_like(p, 999), p, p]
    thr = [0.10, 0.30, 0.20, 0.05, 0.10, 0.10, 0.15, 0.15]
    return np.stack(maps).astype(np.uint16), np.array(thr, np.float32)


def _same(a, b):
    assert a["pos"].shape == b["pos"].shape
    for k in KEYS:
        assert np.array_equal(a[k], b[k]), k


def _singles(ctx, depth, bgr, maps, edge, K, scale, voxel, thr):
    return [ctx.build_scene_cloud(depth, bgr, m, edge, K, scale, voxel, float(t)) for m, t in zip(maps, thr)]


def _raw(ctx, depth, bgr, maps, thr, edge, K, scale, voxel, cap, n_obj=None, outputs=True, rgb_edge=True, offs=True):
    """The C call with explicit capacity and pointers -> (status, offsets, output arrays)."""
    H, W = maps.shape[1:] if depth is None else depth.shape
    n_obj = len(maps) if n_obj is None else n_obj
    c = max(cap, 1)
    out = dict(pos=np.zeros((c, 3), np.float32), nrm=np.zeros((c, 3), np.float32), rgb=np.zeros((c, 3), np.float32),
               pix=np.zeros((c, 2), np.int32), cls=np.zeros(c, np.float32), edge=np.zeros(c, np.float32))
    off = np.full(n_obj + 1 if n_obj > 0 else 1, -7, np.int64)
    ptr = {k: (_ptr(v) if outputs and (rgb_edge or k not in ("rgb", "edge")) else None) for k, v in out.items()}
    rc = ctx._L.stocs_b200_build_scene_clouds(ctx.h, _ptr(depth), _ptr(bgr), _ptr(maps), _ptr(thr), n_obj, _ptr(edge),
                                              W, H, K[0], K[1], K[2], K[3], scale, voxel, ptr["pos"], ptr["nrm"],
                                              ptr["rgb"], ptr["pix"], ptr["cls"], ptr["edge"], cap,
                                              _ptr(off) if offs else None)
    return rc, off, out


def _prepare(depth, bgr, maps, edge):
    return (np.ascontiguousarray(depth, np.uint16), None if bgr is None else np.ascontiguousarray(bgr, np.uint8),
            np.ascontiguousarray(maps, np.uint16), None if edge is None else np.ascontiguousarray(edge, np.uint8))


@pytest.fixture(scope="module")
def ycb():
    depth, bgr, prob, edge, K, scale = _read("ycb")
    maps, thr = _derived(prob)
    return depth, bgr, maps, edge, K, scale, thr


@pytest.mark.parametrize("scene", sorted(CASES))
def test_example_frames_match_the_single_call_and_the_oracle(gpu_ctx, scene):
    depth, bgr, prob, edge, K, scale = _read(scene)
    maps, thr = _derived(prob)
    got = gpu_ctx.build_scene_clouds(depth, bgr, maps, edge, K, scale, 0.005, thr)
    want = _singles(gpu_ctx, depth, bgr, maps, edge, K, scale, 0.005, thr)
    assert len(got) == len(maps)
    for g, w in zip(got, want):
        _same(g, w)
    _same(got[0], oracle.build_scene_cloud(depth, bgr, prob, edge, K, scale, 0.005, 0.10))
    n = [len(g["pos"]) for g in got]
    assert n[0] > 1000 and n[1] > n[0] and n[2] > 0 and n[4] > 0
    assert n[3] == 0 and n[5] == 0            # empty slices between non-empty ones
    assert n[4] >= max(n)                      # p == threshold passes: every centroid that survives the geometry
    _same(got[6], got[7])


def test_one_object_and_the_object_limit(gpu_ctx, ycb):
    depth, bgr, maps, edge, K, scale, thr = ycb
    one = gpu_ctx.build_scene_clouds(depth, bgr, maps[:1], edge, K, scale, 0.005, 0.10)
    assert len(one) == 1
    _same(one[0], gpu_ctx.build_scene_cloud(depth, bgr, maps[0], edge, K, scale, 0.005, 0.10))
    # the linemod frame: its 32 clouds hold more points than one object's bound (H * W)
    ldepth, lbgr, lprob, _, lK, lscale = _read("linemod")
    lmaps, lthr = _derived(lprob)
    idx = np.arange(MAX_OBJECTS) % len(lmaps)
    many = gpu_ctx.build_scene_clouds(ldepth, lbgr, lmaps[idx], None, lK, lscale, 0.005, lthr[idx])
    want = _singles(gpu_ctx, ldepth, lbgr, lmaps, None, lK, lscale, 0.005, lthr)
    assert len(many) == MAX_OBJECTS
    assert sum(len(g["pos"]) for g in many) > ldepth.size
    for g, i in zip(many, idx):
        _same(g, want[i])
    d, b, m, _ = _prepare(depth, bgr, maps[np.arange(MAX_OBJECTS + 1) % len(maps)], None)
    t = np.full(MAX_OBJECTS + 1, 0.1, np.float32)
    for n_obj in (0, -1, MAX_OBJECTS + 1):
        rc, _, _ = _raw(gpu_ctx, d, b, m, t, None, K, scale, 0.005, depth.size, n_obj=n_obj)
        assert rc == E_ARG, n_obj
    with pytest.raises(StocsError):
        gpu_ctx.build_scene_clouds(depth, bgr, m, None, K, scale, 0.005, 0.1)


def _synthetic():
    rng = np.random.default_rng(1234)
    H, W = 480, 640
    yy, xx = np.mgrid[0:H, 0:W]
    depth = (1000 + 0.2 * xx + 0.1 * yy + rng.normal(0, 1.0, (H, W))).astype(np.uint16)
    depth[100:200, 100:300] -= 150
    depth[rng.uniform(size=depth.shape) < 0.05] = 0
    depth[:, :40] = 0
    bgr = rng.integers(0, 256, (H, W, 3)).astype(np.uint8)
    maps = rng.integers(0, 10001, (8, H, W)).astype(np.uint16)
    edge = rng.integers(0, 256, (H, W)).astype(np.uint8)
    return depth, bgr, maps, edge, [572.4114, 325.2611, 573.57043, 242.04899]


def test_synthetic_frame_and_empty_frame(gpu_ctx):
    depth, bgr, maps, edge, K = _synthetic()
    thr = np.linspace(0.05, 0.9, len(maps)).astype(np.float32)
    for voxel in (0.005, 0.01):
        got = gpu_ctx.build_scene_clouds(depth, bgr, maps, edge, K, 1 / 1000.0, voxel, thr)
        want = _singles(gpu_ctx, depth, bgr, maps, edge, K, 1 / 1000.0, voxel, thr)
        for g, w in zip(got, want):
            _same(g, w)
        _same(got[0], oracle.build_scene_cloud(depth, bgr, maps[0], edge, K, 1 / 1000.0, voxel, float(thr[0])))
        assert len(got[0]["pos"]) > 500 and len(got[-1]["pos"]) > 0
    z = np.zeros_like(depth)
    d, b, m, e = _prepare(z, bgr, maps, edge)
    rc, off, _ = _raw(gpu_ctx, d, b, m, thr, e, K, 1 / 1000.0, 0.005, depth.size)
    assert rc == 0 and np.array_equal(off, np.zeros(len(maps) + 1))
    rc, off, _ = _raw(gpu_ctx, d, b, m, thr, e, K, 1 / 1000.0, 0.005, 0)          # cap 0 on an empty frame
    assert rc == 0 and np.array_equal(off, np.zeros(len(maps) + 1))
    rc, off, _ = _raw(gpu_ctx, d, b, m, thr, e, K, 1 / 1000.0, 0.005, 0, outputs=False)   # nothing to write
    assert rc == 0 and np.array_equal(off, np.zeros(len(maps) + 1))


def test_capacity(gpu_ctx, ycb):
    depth, bgr, maps, edge, K, scale, thr = ycb
    want = _singles(gpu_ctx, depth, bgr, maps, edge, K, scale, 0.005, thr)
    ends = np.concatenate([[0], np.cumsum([len(w["pos"]) for w in want])])
    total = int(ends[-1])
    d, b, m, e = _prepare(depth, bgr, maps, edge)
    rc, off, _ = _raw(gpu_ctx, d, b, m, thr, e, K, scale, 0.005, total - 1)
    assert rc == E_CAPACITY and np.array_equal(off, ends)
    for rgb_edge in (True, False):   # rgb3 and edge_p may be NULL
        rc, off, out = _raw(gpu_ctx, d, b, m, thr, e, K, scale, 0.005, total, rgb_edge=rgb_edge)
        assert rc == 0 and np.array_equal(off, ends)
        for k, w in enumerate(want):
            for key in KEYS:
                if rgb_edge or key not in ("rgb", "edge"):
                    assert np.array_equal(out[key][ends[k]:ends[k + 1]], w[key]), (k, key)


def test_read_back_estimate():
    depth, bgr, prob, edge, K, scale = _read("ycb")
    maps, thr = _derived(prob)
    ctx = Context(0)
    try:
        small = np.zeros((48, 64), np.uint16)
        small[8:40, 8:56] = 600
        ctx.build_scene_cloud(small, None, np.full((48, 64), 9000, np.uint16), None, [50.0, 32.0, 50.0, 24.0], 0.001, 0.005, 0.1)
        first = ctx.build_scene_clouds(depth, bgr, maps, edge, K, scale, 0.005, thr)    # estimate too small
        again = ctx.build_scene_clouds(depth, bgr, maps, edge, K, scale, 0.005, thr)    # estimate covers it
    finally:
        ctx.close()
    for a, b in zip(first, again):
        _same(a, b)
    assert sum(len(a["pos"]) for a in first) > 4 * len(first[0]["pos"])


def test_interleaving_matches_fresh_contexts(ycb):
    depth, bgr, maps, edge, K, scale, thr = ycb
    synth = _synthetic()

    def fresh(fn):
        c = Context(0)
        try:
            return fn(c)
        finally:
            c.close()

    def single(c):
        return c.build_scene_cloud(synth[0], synth[1], synth[2][3], synth[3], synth[4], 1 / 1000.0, 0.005, 0.3)

    def multi(c):
        return c.build_scene_clouds(depth, bgr, maps, edge, K, scale, 0.005, thr)

    c = Context(0)
    try:
        s1, m, s2 = single(c), multi(c), single(c)
    finally:
        c.close()
    want_s, want_m = fresh(single), fresh(multi)
    _same(s1, want_s)
    _same(s2, want_s)
    for a, b in zip(m, want_m):
        _same(a, b)


def test_bad_arguments(gpu_ctx, ycb):
    depth, bgr, maps, edge, K, scale, thr = ycb
    d, b, m, e = _prepare(depth, bgr, maps, edge)
    cap = 8 * depth.size
    assert _raw(gpu_ctx, d, b, None, thr, e, K, scale, 0.005, cap, n_obj=len(maps))[0] == E_ARG
    assert _raw(gpu_ctx, d, b, m, None, e, K, scale, 0.005, cap, n_obj=len(maps))[0] == E_ARG
    assert _raw(gpu_ctx, d, b, m, thr, e, K, scale, 0.005, cap, offs=False)[0] == E_ARG
    assert _raw(gpu_ctx, None, b, m, thr, e, K, scale, 0.005, cap)[0] == E_ARG
    assert _raw(gpu_ctx, d, b, m, thr, e, K, scale, 0.0, cap)[0] == E_ARG
    assert _raw(gpu_ctx, d, b, m, thr, e, K, scale, 0.005, -1)[0] == E_ARG
    rc, off, _ = _raw(gpu_ctx, d, b, m, thr, e, K, scale, 0.005, cap, outputs=False)   # points, nowhere to put them
    assert rc == E_ARG and off[-1] > 0
    assert b"output pointer is NULL" in gpu_ctx._L.stocs_b200_last_error(gpu_ctx.h)
    # the context is still usable
    got = gpu_ctx.build_scene_clouds(depth, bgr, maps[:2], edge, K, scale, 0.005, thr[:2])
    _same(got[1], gpu_ctx.build_scene_cloud(depth, bgr, maps[1], edge, K, scale, 0.005, float(thr[1])))
