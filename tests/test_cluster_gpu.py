"""Greedy pose clustering on the device (csrc/cluster.cu; clustering::greedy_clustering, reference
src/pose_clustering.cpp:79-122) against the host shim's loop (model_matching_b200/host, run through
`test_clustering bin`).  Both evaluate the pose distance with csrc/stocs_pose_math.h, so every case
compares the kept index lists for exact equality."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from model_matching_b200 import Context, StocsError, synth
from model_matching_b200._capi import ClusterParams, POSE, PipelineResult
from scenes import object_scene

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "model_matching_b200", "host", "test_clustering")
G = os.path.join(ROOT, "tests", "golden")
SEED = 20181018
E_ARG, E_STATE = -1, -3
SYMS = [(0, 0, 0), (0, 0, 360), (180, 0, 0), (90, 90, 90), (90, 180, 360)]


def shim(T, lcp, best, frac, max_count, min_d, min_a, sym=(0, 0, 0)):
    """the host loop: T (H, 16) column-major world poses"""
    T, lcp = np.ascontiguousarray(T, np.float32).reshape(-1, 16), np.ascontiguousarray(lcp, np.float32)
    head = (np.array([len(lcp)], np.int64).tobytes() + np.array([frac, best], np.float32).tobytes()
            + np.array([max_count], np.int32).tobytes() + np.array([min_d, min_a, *sym], np.float32).tobytes())
    out = subprocess.run([EXE, "bin"], input=head + T.tobytes() + lcp.tobytes(), capture_output=True, check=True).stdout
    return np.array([int(x) for x in out.split()], np.int64)


def pose_diff(Tt, Tb, sym=(0, 0, 0)):
    """the host get_pose_diff of one pair -> (rot, trans) float32"""
    head = np.array([1], np.int64).tobytes() + np.array(sym, np.float32).tobytes()
    out = subprocess.run([EXE, "diff"], input=head + np.float32(Tt).tobytes() + np.float32(Tb).tobytes(),
                         capture_output=True, check=True).stdout
    r, t = np.frombuffer(out, np.float32)
    return r, t


def both(ctx, T, lcp, best, frac, max_count, min_d, min_a, sym=(0, 0, 0)):
    want = shim(T, lcp, best, frac, max_count, min_d, min_a, sym)
    got = ctx.cluster_poses(np.asarray(T, np.float32).reshape(-1, 16), lcp, best, frac, max_count, min_d, min_a, sym)
    assert got.dtype == np.int64
    assert np.array_equal(got, want), (got[:20], want[:20])
    return got


def clustered_list(rng, n_centres=6, per=12, spread_deg=6.0, spread_t=0.004):
    """poses scattered around a few centres, as test_clustering.py builds them (column-major)"""
    centres = synth.random_rotations(rng, n_centres)
    T, lcp = [], []
    for c in range(n_centres):
        t0 = rng.uniform(-0.3, 0.3, 3)
        for _ in range(per):
            dR = synth.axis_angle(rng.normal(size=3), np.deg2rad(rng.uniform(0, spread_deg)))
            M = np.eye(4)
            M[:3, :3] = dR @ centres[c]
            M[:3, 3] = t0 + rng.normal(0, spread_t, 3)
            T.append(M.T.reshape(16))
            lcp.append(rng.uniform(0.05, 0.6))
    return np.array(T, np.float32), np.array(lcp, np.float32)


@pytest.mark.parametrize("sym", SYMS)
def test_random_lists(gpu_ctx, sym):
    rng = np.random.Generator(np.random.Philox(5 + int(sum(sym))))
    for trial in range(4):
        T, lcp = clustered_list(rng, n_centres=4 + 2 * trial, per=8 + 4 * trial)
        got = both(gpu_ctx, T, lcp, float(lcp.max()), 0.5, 10, 0.03, 15.0, sym)
        assert len(got) >= 1 and got[0] == int(np.argmax(lcp))
        both(gpu_ctx, T, lcp, float(lcp.max()), 0.2, 1023, 0.01, 4.0, sym)


def test_large_list_with_fitted_hypotheses(gpu_ctx):
    """2 x 10^5 poses: fitted-like hypotheses around planted poses (most of them near one another, as
    in S1-fit where every hypothesis lands the model on scene surface) and uniform clutter"""
    rng = np.random.Generator(np.random.Philox(17))
    sc = synth.make_scene(n_points=20000, extent=(0.7, 0.5, 0.5), n_objects=5, seed=7)
    mpos, _ = synth.make_model(256)
    T, near = synth.make_hypotheses(200000, sc["pos"], mpos, sc["gt_R"], sc["gt_t"], seed=11, near_fraction=0.4,
                                    max_rot_deg=10.0, max_trans=0.02)
    T = np.ascontiguousarray(T, np.float32).reshape(-1, 16)
    lcp = rng.uniform(0.0, 0.5, len(T)).astype(np.float32)
    lcp[near] += np.float32(0.5)
    lcp = np.round(lcp * 512) / 512      # many equal LCPs: the index order decides among them
    lcp = lcp.astype(np.float32)
    got = both(gpu_ctx, T, lcp, float(lcp.max()), 0.5, 40, 0.02, 10.0)
    assert len(got) > 1
    both(gpu_ctx, T, lcp, float(lcp.max()), 0.95, 1023, 0.005, 3.0, (0, 0, 360))


def test_thresholds_on_the_boundary(gpu_ctx):
    """min_distance / min_angle equal to the exact float distance of a pair, and one ulp either side"""
    rng = np.random.Generator(np.random.Philox(23))
    T, lcp = clustered_list(rng, n_centres=3, per=6)
    order = np.argsort(-lcp, kind="stable")
    a, b = order[0], order[1]                # b is tested against a, the first kept pose
    rot, trans = pose_diff(T[b], T[a])
    assert rot > 0 and trans > 0
    seen = set()
    for d_min in (np.nextafter(trans, np.float32(0)), trans, np.nextafter(trans, np.float32(1))):
        for a_min in (np.nextafter(rot, np.float32(0)), rot, np.nextafter(rot, np.float32(1e9))):
            got = both(gpu_ctx, T, lcp, float(lcp.max()), 0.0, 1023, float(d_min), float(a_min))
            seen.add(int(b) in got.tolist())
            assert (int(b) in got.tolist()) == (not (rot < a_min and trans < d_min))
    assert seen == {True, False}


def test_lcp_edge_cases(gpu_ctx):
    rng = np.random.Generator(np.random.Philox(29))
    T, lcp = clustered_list(rng, n_centres=5, per=10)
    # equal LCPs everywhere: the order is the index order
    eq = np.full_like(lcp, 0.25)
    got = both(gpu_ctx, T, eq, 0.25, 0.5, 20, 0.03, 15.0)
    assert got[0] == 0
    # +0.0 / -0.0 / negative / NaN LCPs under a negative threshold (frac -1, best 1: lcp > -1)
    mixed = lcp.copy()
    mixed[::7] = 0.0
    mixed[3::7] = -0.0
    mixed[5::11] = -0.5
    mixed[2::13] = np.nan
    got = both(gpu_ctx, T, mixed, 1.0, -1.0, 1023, 0.03, 15.0)
    assert not np.isnan(mixed[got]).any()
    got = both(gpu_ctx, T, mixed, 1.0, -1.0, 1023, 1e-9, 1e-9)     # nothing close: every candidate is kept
    cand = np.flatnonzero(mixed > np.float32(-1.0))
    assert sorted(got.tolist()) == cand.tolist()
    zeros = np.flatnonzero(mixed == 0)
    assert [i for i in got if mixed[i] == 0] == sorted(zeros.tolist())   # -0.0 and +0.0 tie: index order
    # NaN transforms among the candidates
    Tn = T.copy()
    Tn[4::9] = np.nan
    Tn[6, 12] = np.nan
    both(gpu_ctx, Tn, lcp, float(lcp.max()), 0.3, 1023, 0.03, 15.0)
    both(gpu_ctx, Tn, lcp, float(lcp.max()), 0.3, 1023, 0.03, 15.0, (90, 180, 360))


def test_parameter_edge_cases(gpu_ctx):
    rng = np.random.Generator(np.random.Philox(31))
    T, lcp = clustered_list(rng, n_centres=8, per=10)
    best = float(lcp.max())
    assert len(both(gpu_ctx, T, lcp, best, 0.0, 1023, 0.03, 15.0)) > 1
    assert len(both(gpu_ctx, T, lcp, best, 1.0, 1023, 0.03, 15.0)) == 0          # lcp > best: nothing
    assert len(both(gpu_ctx, T, lcp, 0.0, 0.5, 1023, 0.03, 15.0)) > 1            # best 0: every lcp > 0
    assert len(both(gpu_ctx, T, -lcp, -1.0, 0.5, 1023, 0.03, 15.0)) > 0          # negative threshold
    assert len(both(gpu_ctx, T, lcp, best, 0.0, 0, 0.03, 15.0)) == 1             # maximum_pose_count 0: one pose
    for m in (1, 2, 3):                                                           # the max + 1 rule
        assert len(both(gpu_ctx, T, lcp, best, 0.0, m, 0.03, 15.0)) == m + 1
    assert len(gpu_ctx.cluster_poses(T[:0], lcp[:0], best, 0.5, 10, 0.03, 15.0)) == 0   # H = 0
    # a tile boundary: many poses kept, more than one tile of candidates
    T2, l2 = clustered_list(rng, n_centres=40, per=30)
    assert len(both(gpu_ctx, T2, l2, float(l2.max()), 0.0, 1023, 1e-4, 1.0)) > 256


def _raw_cluster(ctx, H, p, cap):
    T, lcp = np.zeros((max(H, 1), 16), np.float32), np.ones(max(H, 1), np.float32)
    out, n = np.zeros(max(cap, 1), np.int64), C.c_int64(0)
    return ctx._L.stocs_b200_cluster_poses(ctx.h, T.ctypes.data, lcp.ctypes.data, H, 1.0, p, out.ctypes.data, cap,
                                           C.byref(n))


def test_error_codes(gpu_ctx):
    ctx = gpu_ctx
    p = ClusterParams(0.5, 10, 0.03, 15.0, (C.c_float * 3)(0, 0, 0))
    assert _raw_cluster(ctx, 4, C.byref(p), 11) == 0
    assert _raw_cluster(ctx, 4, C.byref(p), 10) == E_ARG                 # cap < maximum_pose_count + 1
    assert _raw_cluster(ctx, 4, None, 11) == E_ARG                       # NULL params
    assert _raw_cluster(ctx, -1, C.byref(p), 11) == E_ARG
    for m in (-1, 1024):
        q = ClusterParams(0.5, m, 0.03, 15.0, (C.c_float * 3)(0, 0, 0))
        assert _raw_cluster(ctx, 4, C.byref(q), 2000) == E_ARG
    q = ClusterParams(0.5, 1023, 0.03, 15.0, (C.c_float * 3)(0, 0, 0))
    assert _raw_cluster(ctx, 4, C.byref(q), 1024) == 0
    with pytest.raises(StocsError):
        ctx.cluster_poses(np.zeros((2, 16)), np.ones(2), 1.0, 0.5, 1024, 0.03, 15.0)
    fresh = Context(0)
    try:
        r, poses, n = PipelineResult(), np.zeros(11, POSE), C.c_int32(0)
        args = (fresh.h, 1, 10, 10, C.byref(p), C.byref(r), poses.ctypes.data, 11, C.byref(n))
        assert fresh._L.stocs_b200_run_pipeline_clustered(*args) == E_STATE      # nothing uploaded
        assert fresh._L.stocs_b200_run_pipeline_instance_clustered(fresh.h, 1, 10, 10, 0.9, C.byref(p), C.byref(r),
                                                                     poses.ctypes.data, 11, C.byref(n)) == E_STATE
        assert fresh._L.stocs_b200_run_pipeline_clustered(fresh.h, 1, 10, 10, C.byref(p), C.byref(r), poses.ctypes.data,
                                                          10, C.byref(n)) == E_ARG   # cap too small
        assert fresh._L.stocs_b200_run_pipeline_clustered(fresh.h, 1, 10, 10, None, C.byref(r), poses.ctypes.data,
                                                          11, C.byref(n)) == E_ARG   # NULL params
    finally:
        fresh.close()


# ---- the clustered pipeline

PARAMS = dict(acceptable_fraction=0.3, maximum_pose_count=10, min_distance=0.03, min_angle=15.0, sym_info=(0, 0, 0))
N_BASES, MAX_SETS = 100, 200


def _golden(name):
    g = np.load(os.path.join(G, f"golden_{name}.npz"))
    return g["spos"], g["snrm"], g["scls"], g["mpos"], g["mnrm"], (g["spix"] if "spix" in g else None)


def _edge():
    import cv2
    return cv2.imread(os.path.join(G, "examples", "packed", "probability_maps", "edge.png"), cv2.IMREAD_GRAYSCALE)


def _world(name):
    if name == "object_scene":
        sc, mpos, mnrm = object_scene()
        return sc["pos"], sc["nrm"], sc["cls"], mpos, mnrm, None
    return _golden(name)


def _setup(ctx, world, instance):
    spos, snrm, scls, mpos, mnrm, spix = world
    ctx.upload_model(mpos, mnrm)
    ctx.upload_scene(spos, snrm, scls, spix)
    if instance:
        ctx.upload_edge_map(_edge())


def _rebuild(world, instance, seed, n_bases, max_sets):
    """the run's transform list through the per-call ABI: bases, congruent sets, the even spread of at
    most max_sets quads per base, fits (the failed ones are never pushed), scores"""
    ctx = Context(0)
    try:
        _setup(ctx, world, instance)
        if instance:
            bases = []
            for b in range(n_bases):
                ok, ids, inv, _ = ctx.sample_instance_base(seed, b + 1, 0.9, want_mask=False)
                if ok:
                    bases.append((ids.copy(), inv.copy()))
            ids = np.array([b[0] for b in bases], np.int32).reshape(-1, 4)
            inv = np.array([b[1] for b in bases], np.float32).reshape(-1, 2)
        else:
            ids, inv, ok = ctx.sample_bases(seed, 0, n_bases)
            ids, inv = ids[ok], inv[ok]
        quads, offs = ctx.find_congruent(ids, inv)
        ib, iq, base_of = [], [], []
        for b in range(len(ids)):
            cnt = int(offs[b + 1] - offs[b])
            for k in (range(cnt) if cnt < max_sets else [(j * cnt) // max_sets for j in range(max_sets)]):
                ib.append(ids[b]); iq.append(quads[offs[b] + k]); base_of.append(b)
        Tc, Tw, fok = ctx.fit_transforms(np.array(ib, np.int32).reshape(-1, 4), np.array(iq, np.int32).reshape(-1, 4))
        Tc, Tw, base_of = Tc[fok], Tw[fok], np.array(base_of, np.int32)[fok]
        lcp, _ = ctx.score_lcp(Tc)
        return Tc, Tw, base_of, lcp
    finally:
        ctx.close()


def _check_clustered(name, instance, params=PARAMS, seed=SEED):
    world = _world(name)
    ctx = Context(0)
    plain = Context(0)
    try:
        _setup(ctx, world, instance)
        _setup(plain, world, instance)
        if instance:
            r, poses = ctx.run_pipeline_instance_clustered(seed, N_BASES, MAX_SETS, 0.9, **params)
            r0 = plain.run_pipeline_instance(seed, N_BASES, MAX_SETS, 0.9)
        else:
            r, poses = ctx.run_pipeline_clustered(seed, N_BASES, MAX_SETS, **params)
            r0 = plain.run_pipeline(seed, N_BASES, MAX_SETS)
    finally:
        ctx.close()
        plain.close()
    for f in ("n_valid_bases", "n_congruent_sets", "n_transforms", "best_index", "best_lcp", "best_base"):
        assert getattr(r, f) == getattr(r0, f), f
    assert list(r.best_T_centred) == list(r0.best_T_centred) and list(r.best_T_world) == list(r0.best_T_world)
    Tc, Tw, base_of, lcp = _rebuild(world, instance, seed, N_BASES, MAX_SETS)
    assert len(lcp) == r.n_transforms
    want = shim(Tw, lcp, r.best_lcp, params["acceptable_fraction"], params["maximum_pose_count"], params["min_distance"],
                params["min_angle"], params["sym_info"])
    assert np.array_equal(poses["index"], want)
    assert np.array_equal(poses["lcp"].view(np.uint32), lcp[want].view(np.uint32))
    assert np.array_equal(poses["base"], base_of[want])
    assert np.array_equal(poses["T_centred"].view(np.uint32), Tc[want].view(np.uint32))
    assert np.array_equal(poses["T_world"].view(np.uint32), Tw[want].view(np.uint32))
    if r.best_index >= 0:
        p0 = poses[0]
        assert p0["index"] == r.best_index and p0["lcp"] == r.best_lcp and p0["base"] == r.best_base
        assert list(p0["T_world"]) == list(r.best_T_world)
    return r, poses


_MULTI = []


@pytest.mark.parametrize("name", ["ycb", "linemod", "object_scene"])
def test_clustered_pipeline_class_mode(name):
    r, poses = _check_clustered(name, instance=False)
    assert r.best_index >= 0
    _MULTI.append(len(poses))


def test_clustered_pipeline_instance_mode_packed():
    r, poses = _check_clustered("packed", instance=True)
    assert r.best_index >= 0
    _MULTI.append(len(poses))
    assert max(_MULTI) > 1, _MULTI          # some frame holds more than one distinct pose


def test_clustered_pipeline_retry_paths(monkeypatch):
    """with the congruent-set capacities shrunk the run is enqueued again after growing them; the
    clustering enqueued behind it must come back unchanged"""
    world = _world("object_scene")
    ctx0 = Context(0)
    try:
        _setup(ctx0, world, False)
        r0, p0 = ctx0.run_pipeline_clustered(SEED, 48, 40, **PARAMS)
    finally:
        ctx0.close()
    monkeypatch.setenv("STOCS_CONG_CAP_CODES", "64")
    monkeypatch.setenv("STOCS_CONG_CAP_QUADS", "16")
    ctx = Context(0)
    try:
        _setup(ctx, world, False)
        r, p = ctx.run_pipeline_clustered(SEED, 48, 40, **PARAMS)
    finally:
        ctx.close()
    assert (r.n_transforms, r.best_index, r.best_lcp) == (r0.n_transforms, r0.best_index, r0.best_lcp)
    assert len(p0) >= 1 and p.tobytes() == p0.tobytes()
