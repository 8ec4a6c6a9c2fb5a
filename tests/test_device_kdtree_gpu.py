"""A scene uploaded from device memory is planned on the device: the reference centroid, box, class-weight bound and
pixel range come back as one small record, and the reference kd-tree of the scoring kernel's tie rule is built on
the device.  The device tree must equal the host build node for node, and every context must end exactly as the
host upload leaves it."""
import json

import numpy as np
import pytest

from model_matching_b200 import Context, _capi, synth, upload_scenes
from test_device_frames_gpu import _device, _err, _frame, _gpu, _host, _pipelines_match, _raw_upload
from test_multi_object_gpu import _params, _same_scenes, _upload_singly, contexts  # noqa: F401

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def frames():
    return {name: _frame(name) for name in ("ycb", "linemod", "packed")}


@pytest.fixture(scope="module")
def clouds(frames):
    """host clouds of the three example frames (eight objects each)"""
    ctx = Context(0)
    try:
        return {name: _host(ctx, f) for name, f in frames.items()}
    finally:
        ctx.close()


def _same_tree(ctx, pos):
    pos = np.ascontiguousarray(pos, np.float32)
    d_order, d_n, d_nodes = ctx.debug_kdtree(pos, True)
    h_order, h_n, h_nodes = ctx.debug_kdtree(pos, False)
    ref_order, ref_n = _capi.host_kdtree_order(pos)
    assert d_n == h_n == ref_n
    assert np.array_equal(h_order, ref_order)
    assert np.array_equal(d_nodes, h_nodes)
    assert np.array_equal(d_order, h_order)
    assert np.array_equal(np.sort(d_order), np.arange(len(pos)))
    return d_n, d_nodes


def _lattice(seed, n=5000):
    rng = np.random.default_rng(seed)
    pos = (rng.integers(0, 12, (n, 3)) * 0.0625).astype(np.float32)
    pos[: n // 5] = pos[0]
    return pos


@pytest.mark.parametrize("name", ["ycb", "linemod", "packed"])
def test_tree_of_frame_clouds(gpu_ctx, clouds, name):
    objs = [c["pos"] for c in clouds[name] if len(c["pos"])]
    for pos in objs[:3]:
        _same_tree(gpu_ctx, pos - pos.mean(0, dtype=np.float32))
    _same_tree(gpu_ctx, np.concatenate(objs))


def test_tree_of_s1_scene(gpu_ctx):
    sc = synth.make_scene(n_points=1 << 20, seed=1234)
    n, nodes = _same_tree(gpu_ctx, sc["pos"])
    assert n >= 2 * (1 << 20) // 64 - 1 and nodes[:, 0].sum() == (n + 1) // 2


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_tree_of_repeated_coordinates(gpu_ctx, seed):
    _same_tree(gpu_ctx, _lattice(seed))


def test_tree_depth_cap(gpu_ctx):
    """200 copies of one point: every split leaves the left child empty until the level-32 leaf rule"""
    n, nodes = _same_tree(gpu_ctx, np.tile(np.array([[0.25, -0.5, 1.0]], np.float32), (200, 1)))
    assert n == 1 + 2 * 32 and nodes[-1, 0] == 1 and nodes[-1, 2] == 200


@pytest.mark.parametrize("n", [1, 64, 65, 129])
def test_tree_small_sizes(gpu_ctx, n):
    rng = np.random.default_rng(n)
    got_n, nodes = _same_tree(gpu_ctx, rng.normal(0, 0.1, (n, 3)).astype(np.float32))
    assert nodes[0, 0] == 0 and got_n >= 3     # the root is always split


def test_tree_points_on_split_values(gpu_ctx):
    """x in {0, 0.5, 1} (0.5 is the root's split value exactly), then more points on each later split"""
    rng = np.random.default_rng(11)
    x = rng.choice(np.array([0, 0.25, 0.5, 0.75, 1.0], np.float32), 3000)
    pos = np.stack([x, rng.integers(0, 3, 3000) * np.float32(0.125), np.zeros(3000, np.float32)], -1).astype(np.float32)
    _same_tree(gpu_ctx, pos)


def _same_ties(a, b):
    assert a.counters()[1] > 0 and a.counters()[1] == b.counters()[1]


def test_uploads_ycb_class_mode(contexts, frames):
    f = frames["ycb"]
    probe = Context(0)
    try:
        host = _host(probe, f)
        dev = _device(probe, f, _gpu(f["maps"]))
    finally:
        probe.close()
    bat, ref = contexts(8), contexts(8)
    upload_scenes(bat, dev)
    upload_scenes(ref, host)
    _same_scenes(bat, ref, host)
    assert any(len(h["pos"]) == 0 for h in host)                 # empty slices among the eight
    _pipelines_match(bat, ref, [500 + k for k in range(8)])
    _pipelines_match(bat, ref, [600 + k for k in range(8)], cluster=[_params(k) for k in range(8)])


def test_uploads_packed_instance_mode(contexts, frames):
    f = frames["packed"]
    probe = Context(0)
    try:
        host = _host(probe, f, f["maps"][:4], f["thr"][:4])
        dev = _device(probe, f, _gpu(f["maps"][:4]), f["thr"][:4])
    finally:
        probe.close()
    bat, ref = contexts(4, f["edge"]), contexts(4, f["edge"])
    upload_scenes(bat, dev)
    _upload_singly(ref, host)
    _same_scenes(bat, ref, host)
    _pipelines_match(bat, ref, [71, 72, 73, 74], instance=True, cluster=[_params(k) for k in range(4)])


def _lattice_scene():
    g = np.arange(-8, 9, dtype=np.float32) * np.float32(0.0078125)
    X, Y = np.meshgrid(g, g, indexing="ij")
    pos = np.stack([X.ravel(), Y.ravel(), np.zeros(X.size, np.float32)], -1)
    rng = np.random.default_rng(3)
    nrm = rng.normal(size=pos.shape).astype(np.float32)
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    cls = rng.integers(1000, 10001, size=len(pos)).astype(np.float32) / np.float32(10000)
    h = np.float32(0.00390625)
    mp = np.array([[h, 0, 0], [-h, 0, 0], [h, h, 0], [0, h, 0], [3 * h, h, 0], [h, -3 * h, 0]], np.float32)
    mp = np.concatenate([mp, -mp])
    mn = np.tile(np.array([[0, 0, 1]], np.float32), (len(mp), 1))
    T = []
    for i in range(-4, 5):
        for j in range(-4, 5):
            M4 = np.eye(4, dtype=np.float32)
            M4[0, 3], M4[1, 3] = i * 2 * h, j * 2 * h
            T.append(M4.T.reshape(16))
    return pos, nrm, cls, mp, mn, np.array(T, np.float32)


def test_lattice_scene_takes_the_tie_path(monkeypatch):
    """exact distance ties: the device tree decides them as the host tree does, through the device upload and
    through a host upload planned on the device (STOCS_DEVICE_CENTROID)"""
    pos, nrm, cls, mp, mn, T = _lattice_scene()
    ctxs = [Context(0, distance_threshold=0.008) for _ in range(3)]
    try:
        for c in ctxs:
            c.upload_model(mp, mn)
        ctxs[0].upload_scene(pos, nrm, cls)
        upload_scenes([ctxs[1]], [dict(pos=_gpu(pos), nrm=_gpu(nrm), cls=_gpu(cls))])
        monkeypatch.setenv("STOCS_DEVICE_CENTROID", "1")
        ctxs[2].upload_scene(pos, nrm, cls)
        monkeypatch.delenv("STOCS_DEVICE_CENTROID")
        want = ctxs[0].score_lcp(T)
        for c in ctxs[1:]:
            got = c.score_lcp(T)
            assert np.array_equal(got[1], want[1]) and got[0].tobytes() == want[0].tobytes()
            assert c.centred()[0].tobytes() == ctxs[0].centred()[0].tobytes()
            _same_ties(c, ctxs[0])
    finally:
        for c in ctxs:
            c.close()


def test_nothing_scene_sized_crosses_to_the_host(contexts, frames, tmp_path):
    f = frames["ycb"]
    probe = Context(0)
    try:
        dev = _device(probe, f, _gpu(f["maps"]))
    finally:
        probe.close()
    ctxs = contexts(8)
    n = [len(d["pos"]) for d in dev]
    offs = np.concatenate([[0], np.cumsum(n)]).astype(np.int64)
    pos, nrm = torch.cat([d["pos"] for d in dev]), torch.cat([d["nrm"] for d in dev])
    cls, pix = torch.cat([d["cls"] for d in dev]), torch.cat([d["pix"] for d in dev])
    assert _raw_upload(ctxs, pos, nrm, cls, pix, offs) == 0        # warm: buffers grown, modules loaded
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        assert _raw_upload(ctxs, pos, nrm, cls, pix, offs) == 0
        torch.cuda.synchronize()
    trace = str(tmp_path / "upload.json")
    prof.export_chrome_trace(trace)
    with open(trace) as fh:
        events = json.load(fh)["traceEvents"]
    d2h = [e for e in events if e.get("cat") == "gpu_memcpy" and "DtoH" in e.get("name", "")]
    assert d2h, "the plan record and the index lengths come back"
    assert max(e["args"]["bytes"] for e in d2h) <= 256
    assert sum(e["args"]["bytes"] for e in d2h) <= 256 * sum(1 for k in n if k)
    assert sum(1 for e in events if e.get("cat") == "kernel" and "kd_level_kernel" in e.get("name", "")) > 0
    assert [c.counters()[3] > 0 for c in ctxs] == [k > 0 for k in n]


def test_non_finite_coordinate_in_a_device_slice(contexts, frames):
    f = frames["ycb"]
    probe = Context(0)
    try:
        host = _host(probe, f, f["maps"][:3], f["thr"][:3])
        dev = _device(probe, f, _gpu(f["maps"][:3]), f["thr"][:3])
    finally:
        probe.close()
    ctxs, ref = contexts(3), contexts(3)
    bad = [dict(d) for d in dev]
    bad[1]["pos"] = bad[1]["pos"].clone()
    bad[1]["pos"][len(bad[1]["pos"]) // 2, 1] = float("inf")
    with pytest.raises(Exception):
        upload_scenes(ctxs, bad)
    assert "object 1" in _err(ctxs[0]) and "non-finite" in _err(ctxs[0])
    assert [c.S for c in ctxs] == [len(host[0]["pos"]), 0, len(host[2]["pos"])]
    upload_scenes(ref, host)
    _same_scenes([ctxs[0], ctxs[2]], [ref[0], ref[2]], [host[0], host[2]])
    _pipelines_match([ctxs[0], ctxs[2]], [ref[0], ref[2]], [5, 6])
    upload_scenes(ctxs, dev)                                   # the failed context takes the next frame
    _same_scenes(ctxs, ref, host)
    _pipelines_match(ctxs, ref, [7, 8, 9])


def test_second_device(contexts, frames):
    if torch.cuda.device_count() < 2:
        pytest.skip("one device")
    f = frames["ycb"]
    probe = Context(0)
    try:
        host = _host(probe, f, f["maps"][:3], f["thr"][:3])
        dev = _device(probe, f, _gpu(f["maps"][:3]), f["thr"][:3])
    finally:
        probe.close()
    bat, ref = contexts(1) + contexts(2, device=1, first=1), contexts(3)
    upload_scenes(bat, dev)
    _upload_singly(ref, host)
    _same_scenes(bat, ref, host)
    _pipelines_match(bat, ref, [21, 22, 23])
    other = Context(1)
    try:
        pos = _lattice(1)
        assert np.array_equal(other.debug_kdtree(pos, True)[2], other.debug_kdtree(pos, False)[2])
    finally:
        other.close()
