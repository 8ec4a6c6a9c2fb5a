"""Brick-bit refinement of the top-K path (csrc/score.cu, kPrune, loop 1b): after the coarse test, the
survivors whose brick is empty are dropped and the bound is applied again.  Records of
score_sharded_device must stay equal, bit for bit, to records built from the unpruned per-hypothesis
results of the same context (score_lcp_device)."""
import numpy as np
import pytest

from model_matching_b200 import sharding, synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def scene():
    return synth.make_scene(n_points=200000, extent=(0.7, 0.5, 0.5), n_objects=5, seed=1234)


@pytest.fixture(scope="module")
def s1_case(scene):
    from model_matching_b200 import Context
    mpos, mnrm = synth.make_model(512)
    ctx = Context(0)
    ctx.upload_model(mpos, mnrm)
    ctx.upload_scene(scene["pos"], scene["nrm"], scene["cls"])
    T, near = synth.make_hypotheses(200000, scene["pos"], mpos, scene["gt_R"], scene["gt_t"], seed=41, near_fraction=0.01)
    yield ctx, mpos, T, near
    ctx.close()


def _full(ctx, T):
    import torch
    dT = torch.from_numpy(np.ascontiguousarray(T, np.float32)).cuda()
    lcp = torch.empty(max(len(T), 1), dtype=torch.float32, device="cuda")
    inl = torch.empty(max(len(T), 1), dtype=torch.int32, device="cuda")
    ctx.score_lcp_device(dT.data_ptr(), len(T), lcp.data_ptr(), inl.data_ptr())
    torch.cuda.synchronize()
    return lcp.cpu().numpy()[:len(T)], inl.cpu().numpy()[:len(T)]


def _check(ctx, T, K):
    """pruned records == unpruned records; -> change of the rejection counters [4], [5], [8]"""
    import torch
    lcp, inl = _full(ctx, T)
    want = sharding.local_records(lcp, inl, T, 0, K)
    c0 = ctx.counters()
    dT = torch.from_numpy(np.ascontiguousarray(T, np.float32).reshape(-1)).cuda()
    drec = torch.zeros(K * 64, dtype=torch.uint8, device="cuda")
    ctx.score_sharded_device(dT.data_ptr(), len(T), 0, K, drec.data_ptr())
    torch.cuda.synchronize()
    got = drec.cpu().numpy().view(sharding.RECORD)
    assert got.tobytes() == want.tobytes()
    d = ctx.counters() - c0
    return int(d[4]), int(d[5]), int(d[8])


@pytest.mark.parametrize("K", [1, 32])
def test_s1_style_list_rejects_after_refinement(s1_case, K):
    ctx, mpos, T, near = s1_case
    r = _check(ctx, T, K)
    assert r[2] > 0, "the S1-style list must exercise the rejection after the brick-bit refinement"


def test_fitted_list(s1_case, scene):
    # every pose near the truth: most hypotheses have many coarse survivors and skip the refinement
    ctx, mpos, T, near = s1_case
    Tf, _ = synth.make_hypotheses(50000, scene["pos"], mpos, scene["gt_R"], scene["gt_t"], seed=42, near_fraction=1.0)
    _check(ctx, Tf, 32)


def test_nan_transforms(s1_case):
    ctx, mpos, T, near = s1_case
    T2 = T[:100000].copy()
    T2[::5] = np.nan
    T2[1::11, 3] = np.nan    # NaN in the translation only
    _check(ctx, T2, 32)


def test_fewer_hypotheses_than_k(s1_case):
    ctx, mpos, T, near = s1_case
    assert _check(ctx, np.concatenate([T[near[:6]], T[:10]]), 32) == (0, 0, 0)


def test_list_the_refinement_cannot_reject(s1_case):
    # copies of one random pose: every hypothesis reaches theta, so no bound can reject any of them
    ctx, mpos, T, near = s1_case
    mask = np.ones(len(T), bool)
    mask[near] = False
    pose = T[np.flatnonzero(mask)[0]]
    assert _check(ctx, np.repeat(pose[None], 40000, axis=0), 32) == (0, 0, 0)


@pytest.mark.parametrize("n_model", [250, 1024, 1100])
@pytest.mark.parametrize("K", [1, 32])
def test_model_sizes(scene, n_model, K):
    from model_matching_b200 import Context
    mpos, mnrm = synth.make_model(n_model)
    T, _ = synth.make_hypotheses(100000, scene["pos"], mpos, scene["gt_R"], scene["gt_t"], seed=43 + n_model, near_fraction=0.01)
    ctx = Context(0)
    try:
        ctx.upload_model(mpos, mnrm)
        ctx.upload_scene(scene["pos"], scene["nrm"], scene["cls"])
        _check(ctx, T, K)
    finally:
        ctx.close()
