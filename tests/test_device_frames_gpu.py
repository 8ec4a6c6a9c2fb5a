"""stocs_b200_build_scene_clouds_device / stocs_b200_upload_scenes_device: a frame whose images and class maps are
already in GPU memory becomes every object's scene cloud and indexed scene.  Every array must equal the host calls
byte for byte, and every context must end in the state the host calls leave."""
import ctypes as C

import numpy as np
import pytest

from model_matching_b200 import Context, run_pipelines, upload_scenes
from model_matching_b200._capi import _ptr
from test_multi_object_gpu import (MAX_SETS, N_BASES, _params, _run_singly, _same_results, _same_scenes,  # noqa: F401
                                   _upload_singly, contexts)
from test_scene_clouds_gpu import CASES, KEYS, _derived, _read

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu
VOXEL = 0.005
E_ARG, E_CAPACITY = -1, -5


def _exact_f32(maps):
    """float maps holding exactly what the library makes of uint16 maps: (float)((double)(float)v * (1.0/10000))"""
    return (maps.astype(np.float32).astype(np.float64) * (1.0 / 10000)).astype(np.float32)


def _gpu(a, device=0):
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(f"cuda:{device}")


def _frame(scene):
    depth, bgr, prob, edge, K, scale = _read(scene)
    maps, thr = _derived(prob)
    return dict(depth=depth, bgr=bgr, edge=edge, K=K, scale=scale, maps=maps, thr=thr, prob=prob)


def _host(ctx, f, maps=None, thr=None):
    maps = f["maps"] if maps is None else maps
    return ctx.build_scene_clouds(f["depth"], f["bgr"], maps, f["edge"], f["K"], f["scale"], VOXEL,
                                  f["thr"] if thr is None else thr)


def _device(ctx, f, maps, thr=None, **kw):
    return ctx.build_scene_clouds_device(_gpu(f["depth"]), _gpu(f["bgr"]), maps, _gpu(f["edge"]), f["K"], f["scale"], VOXEL,
                                         f["thr"] if thr is None else thr, **kw)


def _same_clouds(dev, host):
    assert len(dev) == len(host)
    for k, (d, h) in enumerate(zip(dev, host)):
        for key in KEYS:
            got = d[key].cpu().numpy()
            assert got.shape == h[key].shape and got.tobytes() == h[key].tobytes(), (k, key)


@pytest.fixture(scope="module")
def ycb():
    return _frame("ycb")


@pytest.mark.parametrize("map_type", ["u16", "f32"])
@pytest.mark.parametrize("scene", sorted(CASES))
def test_clouds_match_the_host_call(gpu_ctx, scene, map_type):
    """eight objects: empty slices between non-empty ones, a constant at the threshold and a repeated map"""
    f = _frame(scene)
    want = _host(gpu_ctx, f)
    maps = _gpu(f["maps"]) if map_type == "u16" else _gpu(_exact_f32(f["maps"]))
    got = _device(gpu_ctx, f, maps)
    _same_clouds(got, want)
    n = [len(w["pos"]) for w in want]
    assert n[0] > 1000 and n[3] == 0 and n[5] == 0 and n[4] >= max(n)


def test_shuffled_channels_of_one_network_output(gpu_ctx, ycb):
    rng = np.random.default_rng(5)
    out = _gpu(_exact_f32(ycb["maps"]))                     # [C, H, W], as a network writes it
    order = np.concatenate([rng.permutation(len(ycb["maps"])), [2, 2]])
    thr = rng.uniform(0.05, 0.5, len(order)).astype(np.float32)
    got = _device(gpu_ctx, ycb, [out[i] for i in order], thr)
    _same_clouds(got, _host(gpu_ctx, ycb, ycb["maps"][order], thr))


def test_float_boundaries(gpu_ctx, ycb):
    H, W = ycb["depth"].shape
    t = np.float32(0.1)
    assert _exact_f32(np.array([1000], np.uint16))[0] == t
    at = _device(gpu_ctx, ycb, [_gpu(np.full((H, W), t, np.float32))], [t])
    _same_clouds(at, _host(gpu_ctx, ycb, np.full((1, H, W), 1000, np.uint16), [t]))   # p == threshold passes
    assert len(at[0]["pos"]) > 1000
    below = _device(gpu_ctx, ycb, [_gpu(np.full((H, W), np.nextafter(t, np.float32(0)), np.float32))], [t])
    assert len(below[0]["pos"]) == 0
    # NaN never passes: the same as a zero where the NaNs are
    rng = np.random.default_rng(9)
    nan = rng.uniform(size=(H, W)) < 0.3
    u16 = np.clip(ycb["prob"], 0, 10000).astype(np.uint16)[None].repeat(2, 0)
    f = _exact_f32(u16)
    f[0][nan] = np.nan
    f[1][nan] = -np.nan
    u16[:, nan] = 0
    thr = np.array([0.1, 0.02], np.float32)
    got = _device(gpu_ctx, ycb, _gpu(f), thr)
    _same_clouds(got, _host(gpu_ctx, ycb, u16, thr))
    assert not torch.isnan(got[0]["cls"]).any() and len(got[0]["pos"]) > 100


def test_caller_stream_orders_the_call(gpu_ctx, ycb):
    want = _host(gpu_ctx, ycb)
    exact = _gpu(_exact_f32(ycb["maps"]))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        maps = torch.zeros_like(exact)
        torch.cuda._sleep(20_000_000)        # the maps are written well after the call is made
        maps.copy_(exact)
    got = _device(gpu_ctx, ycb, maps, stream=side)
    _same_clouds(got, want)
    torch.cuda.synchronize()


def test_capacity_retry_and_error(gpu_ctx, ycb):
    want = _host(gpu_ctx, ycb)
    _same_clouds(_device(gpu_ctx, ycb, _gpu(ycb["maps"]), cap=10), want)   # the wrapper retries at the reported size
    ends = np.concatenate([[0], np.cumsum([len(w["pos"]) for w in want])])
    rc, offs, _ = _raw_build(gpu_ctx, ycb, cap=int(ends[-1]) - 1)
    assert rc == E_CAPACITY and np.array_equal(offs, ends)


def _raw_build(ctx, f, cap, table=None, map_type=0, n_obj=None, host_depth=False, host_out=False, thr=None, device=0):
    """The C call with explicit pointers (maps on device 0, depth and outputs on `device`) -> (status, offsets, outputs)"""
    H, W = f["depth"].shape
    depth = f["depth"] if host_depth else _gpu(f["depth"], device)
    maps = _gpu(f["maps"])
    n_obj = len(f["maps"]) if n_obj is None else n_obj
    table = (C.c_void_p * max(n_obj, 1))(*[maps[k % len(maps)].data_ptr() for k in range(max(n_obj, 1))]) if table is None else table
    thr = np.resize(f["thr"], max(n_obj, 1)).astype(np.float32) if thr is None else thr
    c = max(cap, 1)
    d = f"cuda:{device}"
    out = [torch.zeros((c, 3), device=d) for _ in range(3)] + [torch.zeros((c, 2), dtype=torch.int32, device=d),
                                                               torch.zeros(c, device=d), torch.zeros(c, device=d)]
    host_pos = np.zeros((c, 3), np.float32)
    ptrs = [o.data_ptr() for o in out]
    if host_out:
        ptrs[0] = _ptr(host_pos)
    offs = np.full(max(n_obj, 1) + 1, -7, np.int64)
    K = f["K"]
    rc = ctx._L.stocs_b200_build_scene_clouds_device(
        ctx.h, _ptr(depth) if host_depth else depth.data_ptr(), None, table, map_type, _ptr(thr), n_obj, None, W, H,
        K[0], K[1], K[2], K[3], f["scale"], VOXEL, *ptrs, cap, _ptr(offs), None)
    return rc, offs, out


def _err(ctx):
    return ctx._L.stocs_b200_last_error(ctx.h).decode()


def test_rejected_builds_change_nothing(ycb):
    ctx = Context(0)
    try:
        want = _host(ctx, ycb)
        before = ctx.counters()
        cap = 8 * ycb["depth"].size
        rc, offs, _ = _raw_build(ctx, ycb, cap, host_depth=True)
        assert rc == E_ARG and "d_depth" in _err(ctx)
        rc, _, _ = _raw_build(ctx, ycb, cap, host_out=True)
        assert rc == E_ARG and "d_pos3" in _err(ctx)
        assert _raw_build(ctx, ycb, cap, map_type=2)[0] == E_ARG and "map_type" in _err(ctx)
        maps = _gpu(ycb["maps"])
        table = (C.c_void_p * 8)(*[maps[k].data_ptr() for k in range(8)])
        table[1] = None
        assert _raw_build(ctx, ycb, cap, table=table)[0] == E_ARG and "d_class_maps[1] is NULL" in _err(ctx)
        host_map = np.zeros(ycb["depth"].shape, np.uint16)
        table[1] = _ptr(host_map)
        assert _raw_build(ctx, ycb, cap, table=table)[0] == E_ARG and "d_class_maps[1]" in _err(ctx)
        for n_obj in (0, -1, 33):
            assert _raw_build(ctx, ycb, cap, n_obj=n_obj)[0] == E_ARG, n_obj
        assert np.array_equal(ctx.counters(), before)
        _same_clouds(_device(ctx, ycb, _gpu(ycb["maps"])), want)
    finally:
        ctx.close()


def _pipelines_match(bat, ref, seeds, instance=False, cluster=None):
    _same_results(run_pipelines(bat, seeds, instance=instance, cluster=cluster),
                  _run_singly(ref, seeds, instance=instance, cluster=cluster))


def test_uploads_and_pipelines_ycb(contexts, ycb):
    """device clouds -> upload_scenes_device must leave every context as upload_scenes leaves it from host copies"""
    probe = Context(0)
    try:
        host = _host(probe, ycb)
        dev = _device(probe, ycb, _gpu(ycb["maps"]))
    finally:
        probe.close()
    bat, ref = contexts(8), contexts(8)
    seeds = [1000 + 7 * k for k in range(8)]
    cl = [_params(k) for k in range(8)]
    upload_scenes(bat, dev)
    upload_scenes(ref, host)
    _same_scenes(bat, ref, host)
    _pipelines_match(bat, ref, seeds)
    _pipelines_match(bat, ref, seeds, cluster=cl)
    assert bytes(bat[0].run_pipeline(5, N_BASES, MAX_SETS)) == bytes(ref[0].run_pipeline(5, N_BASES, MAX_SETS))

    # a second frame on the same contexts: slices in another order (concatenated, not views of one buffer)
    upload_scenes(bat, dev[::-1])
    ref2 = contexts(8)
    _upload_singly(ref2, host[::-1])
    _same_scenes(bat, ref2, host[::-1])
    _pipelines_match(bat, ref2, [77 + k for k in range(8)], cluster=cl)

    # interleaved with host uploads on the same contexts
    bat[0].upload_scene(host[1]["pos"], host[1]["nrm"], host[1]["cls"], host[1]["pix"])
    upload_scenes(bat[1:4], dev[:3])
    upload_scenes(ref2[1:4], host[:3])
    ref2[0].upload_scene(host[1]["pos"], host[1]["nrm"], host[1]["cls"], host[1]["pix"])
    _same_scenes(bat[:4], ref2[:4], [host[1]] + host[:3])
    _pipelines_match(bat[:4], ref2[:4], [3, 4, 5, 6])


def test_uploads_and_pipelines_packed_instance(contexts):
    f = _frame("packed")
    probe = Context(0)
    try:
        host = _host(probe, f, f["maps"][:4], f["thr"][:4])
        dev = _device(probe, f, _gpu(_exact_f32(f["maps"][:4])), f["thr"][:4])
    finally:
        probe.close()
    assert len(host[3]["pos"]) == 0 and min(len(h["pos"]) for h in host[:3]) > 0
    bat, ref = contexts(4, f["edge"]), contexts(4, f["edge"])
    upload_scenes(bat, dev)
    _upload_singly(ref, host)
    _same_scenes(bat, ref, host)
    _pipelines_match(bat, ref, [31, 32, 33, 34], instance=True)
    _pipelines_match(bat, ref, [41, 42, 43, 44], instance=True, cluster=[_params(k) for k in range(4)])


def _raw_upload(ctxs, pos, nrm, cls, pix, offs):
    arr = (C.c_void_p * len(ctxs))(*[c.h for c in ctxs])
    p = [None if t is None else (t.data_ptr() if isinstance(t, torch.Tensor) else _ptr(t)) for t in (pos, nrm, cls, pix)]
    return ctxs[0]._L.stocs_b200_upload_scenes_device(arr, len(ctxs), *p, _ptr(offs), None)


def test_rejected_uploads_change_nothing(contexts, ycb):
    probe = Context(0)
    try:
        dev = _device(probe, ycb, _gpu(ycb["maps"][:3]), ycb["thr"][:3])
    finally:
        probe.close()
    ctxs = contexts(3)
    upload_scenes(ctxs, dev)
    seeds = [11, 12, 13]
    before = run_pipelines(ctxs, seeds)
    centred = [c.centred()[0].tobytes() for c in ctxs]
    n = [len(d["pos"]) for d in dev]
    pos = torch.cat([d["pos"] for d in dev]); nrm = torch.cat([d["nrm"] for d in dev])
    cls = torch.cat([d["cls"] for d in dev]); pix = torch.cat([d["pix"] for d in dev])
    offs = np.array([0, n[0], n[0] + n[1], sum(n)], np.int64)
    a = ctxs[0]
    assert _raw_upload(ctxs, pos, nrm, cls, pix, np.array([0, 5, 3, 9], np.int64)) == E_ARG and "object 1" in _err(a)
    assert _raw_upload(ctxs, pos.cpu().numpy(), nrm, cls, pix, offs) == E_ARG and "d_pos3" in _err(a)
    assert _raw_upload(ctxs, pos, nrm, cls.cpu().numpy(), pix, offs) == E_ARG and "d_class_probability" in _err(a)
    assert _raw_upload(ctxs, None, nrm, cls, pix, offs) == E_ARG
    assert [c.centred()[0].tobytes() for c in ctxs] == centred
    _same_results(run_pipelines(ctxs, seeds), before)
    assert _raw_upload(ctxs, pos, nrm, cls, pix, offs) == 0             # the concatenation, raw
    _same_results(run_pipelines(ctxs, seeds), before)


def test_second_device(contexts, ycb):
    if torch.cuda.device_count() < 2:
        pytest.skip("one device")
    probe = Context(0)
    try:
        host = _host(probe, ycb, ycb["maps"][:3], ycb["thr"][:3])
        dev = _device(probe, ycb, _gpu(ycb["maps"][:3]), ycb["thr"][:3])
    finally:
        probe.close()
    bat = contexts(1) + contexts(2, device=1, first=1)      # clouds on device 0, two contexts on device 1
    ref = contexts(3)
    upload_scenes(bat, dev)
    _upload_singly(ref, host)
    _same_scenes(bat, ref, host)
    _pipelines_match(bat, ref, [8, 9, 10])
    # a map on another device than the context's
    other = Context(1)
    try:
        rc = _raw_build(other, ycb, 8 * ycb["depth"].size, device=1)[0]
        assert rc == E_ARG and "d_class_maps[0] is not device memory on device 1" in _err(other)
    finally:
        other.close()
