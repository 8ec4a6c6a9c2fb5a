"""stocs_b200_upload_scenes / stocs_b200_run_pipelines: several objects of one frame, one context per object,
given their work together.  Every object's outcome must be bit-identical to the single calls on a second
set of contexts fed the same inputs, and every context must end in the same state."""
import ctypes as C
import os

import numpy as np
import pytest

from model_matching_b200 import Context, StocsError, run_pipelines, upload_scenes
from model_matching_b200._capi import POSE, ClusterParams, PipelineResult, _cluster_params, _ptr
from test_scene_clouds_gpu import _derived, _read

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
E_ARG, E_STATE = -1, -3
N_BASES, MAX_SETS = 100, 200
MODELS = ("ycb", "linemod", "packed")          # 024_bowl, obj_06, dove
SYMS = ((0, 0, 0), (0, 0, 360), (180, 0, 90))
VOXEL = 0.005


def _model(name):
    g = np.load(os.path.join(G, f"golden_{name}.npz"))
    return g["mpos"], g["mnrm"]


def _params(k, max_count=10):
    return dict(acceptable_fraction=0.3, maximum_pose_count=max_count, min_distance=0.03, min_angle=15.0,
                sym_info=SYMS[k % len(SYMS)])


@pytest.fixture
def contexts():
    """make(n, edge=None, device=0, first=0) -> n contexts, the k-th holding model (first + k) mod 3 (and the edge map)."""
    made = []

    def make(n, edge=None, device=0, first=0):
        out = []
        for k in range(first, first + n):
            c = Context(device)
            made.append(c)
            c.upload_model(*_model(MODELS[k % len(MODELS)]))
            if edge is not None:
                c.upload_edge_map(edge)
            out.append(c)
        return out

    yield make
    for c in made:
        c.close()


def _frame(scene, n=None):
    depth, bgr, prob, edge, K, scale = _read(scene)
    maps, thr = _derived(prob)
    if n is not None:
        maps, thr = maps[:n], thr[:n]
    probe = Context(0)
    try:
        clouds = probe.build_scene_clouds(depth, bgr, maps, edge, K, scale, VOXEL, thr)
    finally:
        probe.close()
    return clouds, edge


def _upload_singly(ctxs, clouds):
    for c, cl in zip(ctxs, clouds):
        if len(cl["pos"]):
            c.upload_scene(cl["pos"], cl["nrm"], cl["cls"], cl["pix"])


def _run_singly(ctxs, seeds, instance=False, cluster=None):
    out = []
    for k, (c, s) in enumerate(zip(ctxs, seeds)):
        if c.S == 0:
            r = PipelineResult()
            r.best_index = r.best_base = -1
            out.append(r if cluster is None else (r, np.zeros(0, POSE)))
        elif cluster is None:
            out.append(c.run_pipeline_instance(s, N_BASES, MAX_SETS, 0.9) if instance else c.run_pipeline(s, N_BASES, MAX_SETS))
        elif instance:
            out.append(c.run_pipeline_instance_clustered(s, N_BASES, MAX_SETS, 0.9, **cluster[k]))
        else:
            out.append(c.run_pipeline_clustered(s, N_BASES, MAX_SETS, **cluster[k]))
    return out


def _same_results(got, want):
    assert len(got) == len(want)
    for k, (g, w) in enumerate(zip(got, want)):
        if isinstance(w, tuple):
            assert bytes(g[0]) == bytes(w[0]), k
            assert g[1].tobytes() == w[1].tobytes(), k
        else:
            assert bytes(g) == bytes(w), k


def _same_scenes(a, b, clouds):
    for k, (x, y) in enumerate(zip(a, b)):
        assert x.S == y.S == len(clouds[k]["pos"]), k
        cx, cy = x.counters(), y.counters()
        assert [cx[2], cx[3], cx[6]] == [cy[2], cy[3], cy[6]], k
        if x.S:
            assert x.centroids()[0].tobytes() == y.centroids()[0].tobytes(), k
            assert x.centred()[0].tobytes() == y.centred()[0].tobytes(), k


def _no_pose(r):
    return r.best_index == -1 and r.best_base == -1 and r.n_transforms == 0 and r.best_lcp == 0.0


def test_ycb_class_mode_frames_and_interleaving(contexts):
    """eight objects (two of them empty slices between non-empty ones), plain and clustered, two frames, and
    single calls interleaved with batched ones on the same contexts"""
    clouds, _ = _frame("ycb")
    sizes = [len(c["pos"]) for c in clouds]
    assert sizes[3] == 0 and sizes[5] == 0 and min(sizes[:3]) > 0
    bat, ref = contexts(8), contexts(8)
    seeds = [1000 + 7 * k for k in range(8)]
    cl = [_params(k) for k in range(8)]

    upload_scenes(bat, clouds)
    _upload_singly(ref, clouds)
    _same_scenes(bat, ref, clouds)
    got = run_pipelines(bat, seeds)
    _same_results(got, _run_singly(ref, seeds))
    assert all(_no_pose(got[k]) for k in (3, 5)) and got[0].best_index >= 0
    got = run_pipelines(bat, seeds, cluster=cl)
    _same_results(got, _run_singly(ref, seeds, cluster=cl))
    assert len(got[3][1]) == 0 and max(len(p) for _, p in got) > 1

    # second frame on the same contexts: other objects visible (objects 2 and 4 vanish), other seeds
    clouds2 = clouds[::-1]
    upload_scenes(bat, clouds2)
    ref2 = contexts(8)
    _upload_singly(ref2, clouds2)
    seeds2 = [77 + k for k in range(8)]
    _same_scenes(bat, ref2, clouds2)
    _same_results(run_pipelines(bat, seeds2, cluster=cl), _run_singly(ref2, seeds2, cluster=cl))

    # single calls on batched contexts, then a batch again
    bat[0].upload_scene(clouds[1]["pos"], clouds[1]["nrm"], clouds[1]["cls"], clouds[1]["pix"])
    ref2[0].upload_scene(clouds[1]["pos"], clouds[1]["nrm"], clouds[1]["cls"], clouds[1]["pix"])
    assert bytes(bat[0].run_pipeline(5, N_BASES, MAX_SETS)) == bytes(ref2[0].run_pipeline(5, N_BASES, MAX_SETS))
    _same_results(run_pipelines(bat, seeds), _run_singly(ref2, seeds))


def test_packed_instance_mode_state_carries_over(contexts):
    clouds, edge = _frame("packed", 4)
    assert len(clouds[3]["pos"]) == 0 and min(len(c["pos"]) for c in clouds[:3]) > 0
    bat, ref = contexts(4, edge), contexts(4, edge)
    upload_scenes(bat, clouds)
    _upload_singly(ref, clouds)
    _same_scenes(bat, ref, clouds)
    for frame, cl in ((0, None), (1, [_params(k) for k in range(4)])):   # the second batch sees the first's decay
        seeds = [31 + 10 * frame + k for k in range(4)]
        got = run_pipelines(bat, seeds, instance=True, cluster=cl)
        _same_results(got, _run_singly(ref, seeds, instance=True, cluster=cl))
        for a, b in zip(bat[:3], ref[:3]):
            assert a.class_probability().tobytes() == b.class_probability().tobytes()
    assert not np.array_equal(bat[0].class_probability(), clouds[0]["cls"])   # the prior did decay


def test_one_object(contexts):
    clouds, _ = _frame("ycb", 1)
    (bat,), (ref,) = contexts(1), contexts(1)
    upload_scenes([bat], clouds)
    _upload_singly([ref], clouds)
    _same_scenes([bat], [ref], clouds)
    _same_results(run_pipelines([bat], [9]), _run_singly([ref], [9]))
    _same_results(run_pipelines([bat], [9], cluster=[_params(0)]), _run_singly([ref], [9], cluster=[_params(0)]))


def test_retry_paths(contexts, monkeypatch):
    """objects 0 and 2 start from tiny congruent-set capacities and retry alone; a one-record candidate
    capacity makes every index build retry"""
    clouds, _ = _frame("ycb", 4)
    seeds = [3, 4, 5, 6]
    cl = [_params(k) for k in range(4)]
    ref = contexts(4)
    _upload_singly(ref, clouds)
    want_plain, want_cl = _run_singly(ref, seeds), _run_singly(ref, seeds, cluster=cl)
    bat = []
    for k in range(4):
        if k % 2 == 0:
            monkeypatch.setenv("STOCS_CONG_CAP_CODES", "64")
            monkeypatch.setenv("STOCS_CONG_CAP_QUADS", "16")
        else:
            monkeypatch.delenv("STOCS_CONG_CAP_CODES", raising=False)
            monkeypatch.delenv("STOCS_CONG_CAP_QUADS", raising=False)
        bat += contexts(1, first=k)
    monkeypatch.setenv("STOCS_CAND_CAP", "1")
    upload_scenes(bat, clouds)
    monkeypatch.delenv("STOCS_CAND_CAP")
    _same_scenes(bat, ref, clouds)
    assert len(clouds[3]["pos"]) == 0
    for want, kw in ((want_plain, {}), (want_cl, dict(cluster=cl))):
        before = [c.counters()[0] for c in bat]          # scoring launches: one per attempt of a run
        _same_results(run_pipelines(bat, seeds, **kw), want)
        launches = [c.counters()[0] - b for c, b in zip(bat, before)]
        if not kw:   # the first run: objects 0 and 2 overflow and are enqueued again, alone
            assert launches[0] >= 2 and launches[2] >= 2 and launches[1] == 1 and launches[3] == 0, launches
        else:        # their capacities have grown: one attempt each
            assert launches == [1, 1, 1, 0], launches


def _raw_upload(ctxs, n, pos, nrm, cls, pix, offs):
    arr = (C.c_void_p * max(len(ctxs), 1))(*[None if c is None else c.h for c in ctxs])
    return ctxs[0]._L.stocs_b200_upload_scenes(arr, n, _ptr(pos), _ptr(nrm), _ptr(cls), _ptr(pix), _ptr(offs))


def _raw_run(ctxs, n, seeds, n_bases=N_BASES, max_sets=MAX_SETS, mode=0, cluster=None, results=True, poses=True, cap=None):
    arr = (C.c_void_p * max(len(ctxs), 1))(*[None if c is None else c.h for c in ctxs])
    res = (PipelineResult * max(n, 1))() if results else None
    params = (ClusterParams * len(cluster))(*[_cluster_params(**p) for p in cluster]) if cluster else None
    cap = 11 if cap is None else cap
    ps = np.zeros((max(n, 1), max(cap, 1)), POSE) if poses else None
    npo = np.zeros(max(n, 1), np.int32)
    return ctxs[0]._L.stocs_b200_run_pipelines(arr, n, _ptr(seeds), n_bases, max_sets, mode, 0.9, params, res, _ptr(ps), cap,
                                               _ptr(npo))


def _err(c):
    return c._L.stocs_b200_last_error(c.h).decode()


def test_rejected_calls_change_nothing(contexts):
    clouds, _ = _frame("ycb", 3)
    ctxs = contexts(3)
    upload_scenes(ctxs, clouds)
    seeds = np.array([11, 12, 13], np.uint64)
    before = run_pipelines(ctxs, seeds)
    centred = [c.centred()[0].tobytes() for c in ctxs]
    pos = np.ascontiguousarray(np.concatenate([c["pos"] for c in clouds]), np.float32)
    nrm = np.ascontiguousarray(np.concatenate([c["nrm"] for c in clouds]), np.float32)
    cls = np.ascontiguousarray(np.concatenate([c["cls"] for c in clouds]), np.float32)
    n = [len(c["pos"]) for c in clouds]
    offs = np.array([0, n[0], n[0] + n[1], sum(n)], np.int64)
    a, b, c = ctxs
    # upload_scenes
    assert _raw_upload(ctxs, 0, pos, nrm, cls, None, offs) == E_ARG
    assert _raw_upload([a, None, c], 3, pos, nrm, cls, None, offs) == E_ARG and "object 1" in _err(a)
    assert _raw_upload([a, b, a], 3, pos, nrm, cls, None, offs) == E_ARG and "object 2" in _err(a)
    assert _raw_upload(ctxs, 3, None, nrm, cls, None, offs) == E_ARG
    assert _raw_upload(ctxs, 3, pos, nrm, cls, None, None) == E_ARG
    assert _raw_upload(ctxs, 3, pos, nrm, cls, None, offs + 1) == E_ARG
    assert _raw_upload(ctxs, 3, pos, nrm, cls, None, np.array([0, 5, 3, 9], np.int64)) == E_ARG and "object 1" in _err(a)
    assert _raw_upload(ctxs, 3, pos, nrm, cls, None, np.array([0, 1, 2 + (1 << 27), 3 + (1 << 27)], np.int64)) == E_ARG
    assert "object 1" in _err(a) and "object 1" in _err(b)
    # run_pipelines
    no_model = Context(0)
    no_scene = contexts(1)[0]
    try:
        assert _raw_run(ctxs, 0, seeds) == E_ARG
        assert _raw_run([a, None, c], 3, seeds) == E_ARG
        assert _raw_run([a, b, b], 3, seeds) == E_ARG and "object 2" in _err(a)
        assert _raw_run(ctxs, 3, None) == E_ARG
        assert _raw_run(ctxs, 3, seeds, results=False) == E_ARG
        assert _raw_run(ctxs, 3, seeds, n_bases=0) == E_ARG
        assert _raw_run(ctxs, 3, seeds, max_sets=0) == E_ARG
        assert _raw_run(ctxs, 3, seeds, mode=2) == E_ARG
        assert _raw_run([a, b, no_model], 3, seeds) == E_STATE and "object 2" in _err(no_model) and "object 2" in _err(a)
        assert _raw_run([a, no_scene, c], 3, seeds) == E_STATE and "object 1" in _err(a)
        assert _raw_run(ctxs, 3, seeds, mode=1) == E_STATE                        # no edge map
        assert _raw_run(ctxs, 3, seeds, n_bases=256, mode=1) == E_ARG
        cl = [_params(k) for k in range(3)]
        assert _raw_run(ctxs, 3, seeds, cluster=cl, cap=10) == E_ARG               # cap < maximum_pose_count + 1
        assert _raw_run(ctxs, 3, seeds, cluster=cl, poses=False) == E_ARG
        assert _raw_run(ctxs, 3, seeds, cluster=cl[:2] + [_params(2, 5000)], cap=5001) == E_ARG and "object 2" in _err(a)
    finally:
        no_model.close()
    assert [x.centred()[0].tobytes() for x in ctxs] == centred
    _same_results(run_pipelines(ctxs, seeds), before)
    for x in ctxs:
        x.upload_edge_map(np.full((480, 640), 255, np.uint8))
    upload_scenes(ctxs, [dict(o, pix=None) for o in clouds])                     # no pixel coordinates
    assert _raw_run(ctxs, 3, seeds, mode=1) == E_STATE and "object 0" in _err(a) and "pixel" in _err(a)


def test_failure_after_validation(contexts):
    """non-finite coordinates are found while centring: the first failing object's error comes back, the
    others complete, and the failing context is left without a scene as upload_scene leaves it"""
    clouds, _ = _frame("ycb", 3)
    bad = [dict(c) for c in clouds]
    bad[1]["pos"] = bad[1]["pos"].copy()
    bad[1]["pos"][5, 0] = np.nan
    bat, ref = contexts(3), contexts(3)
    with pytest.raises(StocsError, match="object 1.*non-finite"):
        upload_scenes(bat, bad)
    with pytest.raises(StocsError, match="non-finite"):
        ref[1].upload_scene(bad[1]["pos"], bad[1]["nrm"], bad[1]["cls"], bad[1]["pix"])
    _upload_singly([ref[0], ref[2]], [clouds[0], clouds[2]])
    assert [c.S for c in bat] == [len(clouds[0]["pos"]), 0, len(clouds[2]["pos"])]
    for k in (0, 2):
        assert bat[k].centred()[0].tobytes() == ref[k].centred()[0].tobytes()
    with pytest.raises(StocsError, match="object 1.*upload_scene first"):
        run_pipelines(bat, [1, 2, 3])
    _same_results(run_pipelines([bat[0], bat[2]], [1, 3]), _run_singly([ref[0], ref[2]], [1, 3]))


def test_two_devices(contexts):
    try:
        probe = Context(1)
        probe.close()
    except StocsError:
        pytest.skip("one device")
    clouds, _ = _frame("ycb", 2)
    bat = contexts(1) + contexts(1, device=1, first=1)
    ref = contexts(2)
    upload_scenes(bat, clouds)
    _upload_singly(ref, clouds)
    _same_scenes(bat, ref, clouds)
    _same_results(run_pipelines(bat, [8, 9]), _run_singly(ref, [8, 9]))
