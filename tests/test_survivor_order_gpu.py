"""Survivor order of the device top-K path (csrc/score.cu, survivor_count_kernel / rank_scatter_kernel):
a top-K launch of more than 300 000 hypotheses (above the heavy-first range) counts every hypothesis's
coarse survivors first, claims in descending count and stops at the first claim the bound rejects.  The counts must be loop 1's, and the
records must equal, bit for bit, those built from the unpruned per-hypothesis results."""
import numpy as np
import pytest

from model_matching_b200 import sharding, synth

pytestmark = pytest.mark.gpu

RANKED_MIN = 300001   # smallest launch that takes the survivor order (above lpt_max in score.cu)
N = 320000


@pytest.fixture(scope="module")
def order_case(small_scene):
    from model_matching_b200 import Context
    sc, mpos, mnrm = small_scene
    ctx = Context(0)
    ctx.upload_model(mpos, mnrm)
    ctx.upload_scene(sc["pos"], sc["nrm"], sc["cls"])
    T, near = synth.make_hypotheses(N, sc["pos"], mpos, sc["gt_R"], sc["gt_t"], seed=41, near_fraction=0.01)
    yield ctx, sc, mpos, mnrm, T, near
    ctx.close()


def _dev(T):
    import torch
    return torch.from_numpy(np.ascontiguousarray(T, np.float32).reshape(-1)).cuda()


def _counts(ctx, T):
    dT = _dev(T)
    return ctx.debug_survivor_counts(dT.data_ptr(), len(T))


def _full(ctx, T):
    import torch
    dT = _dev(T)
    lcp = torch.empty(len(T), dtype=torch.float32, device="cuda")
    inl = torch.empty(len(T), dtype=torch.int32, device="cuda")
    ctx.score_lcp_device(dT.data_ptr(), len(T), lcp.data_ptr(), inl.data_ptr())
    torch.cuda.synchronize()
    return lcp.cpu().numpy(), inl.cpu().numpy()


def _pruned(ctx, T, K):
    import torch
    dT = _dev(T)
    drec = torch.zeros(K * 64, dtype=torch.uint8, device="cuda")
    ctx.score_sharded_device(dT.data_ptr(), len(T), 0, K, drec.data_ptr())
    torch.cuda.synchronize()
    return drec.cpu().numpy().view(sharding.RECORD).copy()


def _check(ctx, T, K=32):
    lcp, inl = _full(ctx, T)
    want = sharding.local_records(lcp, inl, T, 0, K)
    got = _pruned(ctx, T, K)
    assert got.tobytes() == want.tobytes()
    return lcp


def test_counts_equal_loop1_per_hypothesis(order_case):
    ctx, sc, mpos, mnrm, T, near = order_case
    idx = np.concatenate([near[:200], np.arange(1800)])
    T2 = T[idx]
    ns = _counts(ctx, T2)
    dT = _dev(T2)
    for h in range(len(T2)):
        c = ctx.score_counters(dT[16 * h:16 * (h + 1)].data_ptr(), 1)
        assert ns[h] == c["coarse_survivors"], h
    assert ns[:200].mean() > ns[200:].mean()   # near-truth poses keep more of the model


def test_count_sum_equals_coarse_survivors(order_case):
    ctx, sc, mpos, mnrm, T, near = order_case
    T = T[:200000]
    ns = _counts(ctx, T)
    dT = _dev(T)
    assert int(ns.astype(np.int64).sum()) == ctx.score_counters(dT.data_ptr(), len(T))["coarse_survivors"]


def test_non_finite_transforms_count_every_point(order_case):
    ctx, sc, mpos, mnrm, T, near = order_case
    T2 = T[:1000].copy()
    T2[::7] = np.nan
    T2[3, 12] = np.inf
    T2[5, 0] = 1e38                      # finite, but the grid map of it overflows
    ns = _counts(ctx, T2)
    bad = np.zeros(len(T2), bool)
    bad[::7] = bad[3] = bad[5] = True
    assert (ns[bad] == len(mpos)).all()
    assert (ns[~bad] == _counts(ctx, T2[~bad])).all()


@pytest.mark.parametrize("direction", ["ascending", "descending"])
def test_lists_sorted_by_count(order_case, direction):
    ctx, sc, mpos, mnrm, T, near = order_case
    ns = _counts(ctx, T)
    order = np.argsort(ns, kind="stable")
    if direction == "descending":
        order = order[::-1]
    _check(ctx, T[order])


def test_one_count_bin(order_case):
    ctx, sc, mpos, mnrm, T, near = order_case
    T2 = np.repeat(T[near[:1]], N, axis=0)
    assert len(np.unique(_counts(ctx, T2))) == 1
    _check(ctx, T2)
    _check(ctx, T2, K=1)


def test_all_nan_and_every_7th_row_nan(order_case):
    ctx, sc, mpos, mnrm, T, near = order_case
    _check(ctx, np.full((N, 16), np.nan, np.float32))
    T2 = T.copy()
    T2[::7] = np.nan
    _check(ctx, T2)


@pytest.mark.parametrize("H", [RANKED_MIN - 1, RANKED_MIN, 1000000])
@pytest.mark.parametrize("K", [1, 32])
def test_list_sizes_around_the_threshold(order_case, H, K):
    ctx, sc, mpos, mnrm, T, near = order_case
    _check(ctx, np.resize(T, (H, 16)), K)


def test_fewer_scored_poses_than_k(order_case):
    """K larger than the number of hypotheses with a nonzero LCP: theta never rises, nothing is cut"""
    ctx, sc, mpos, mnrm, T, near = order_case
    far = np.setdiff1d(np.arange(len(T)), near)
    lcp, _ = _full(ctx, T[far])
    T2 = np.concatenate([np.resize(T[far][lcp == 0], (N - 5, 16)), T[near[:5]]])
    _check(ctx, T2)
    _check(ctx, T[near[:20]])           # H < K


@pytest.mark.parametrize("n_model", [250, 1024, 1100])
def test_model_sizes(small_scene, n_model):
    from model_matching_b200 import Context
    sc, _, _ = small_scene
    mpos, mnrm = synth.make_model(n_model)
    T, _ = synth.make_hypotheses(N, sc["pos"], mpos, sc["gt_R"], sc["gt_t"], seed=42, near_fraction=0.01)
    ctx = Context(0)
    try:
        ctx.upload_model(mpos, mnrm)
        ctx.upload_scene(sc["pos"], sc["nrm"], sc["cls"])
        before = ctx.counters()[4]
        _check(ctx, T)
        assert ctx.counters()[4] > before
    finally:
        ctx.close()


def test_cut_counter_moves_only_on_the_top_k_path(order_case):
    ctx, sc, mpos, mnrm, T, near = order_case
    c0 = ctx.counters()
    _pruned(ctx, T, 32)
    c1 = ctx.counters()
    assert 0 < c1[4] - c0[4]
    assert (c1[4] - c0[4]) + (c1[5] - c0[5]) + (c1[8] - c0[8]) <= len(T)
    _full(ctx, T)
    dT = _dev(T)
    ctx.score_counters(dT.data_ptr(), len(T))
    _counts(ctx, T)
    assert (ctx.counters()[[4, 5, 8]] == c1[[4, 5, 8]]).all()
