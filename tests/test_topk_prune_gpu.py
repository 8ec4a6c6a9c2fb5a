"""Top-K pruning of the device top-K path (csrc/score.cu, kPrune): score_sharded_device may leave
hypotheses that provably cannot enter the top K unscored, so its records must equal, bit for bit, the
records built from the unpruned per-hypothesis results of the same context (score_lcp_device)."""
import numpy as np
import pytest

from model_matching_b200 import sharding, synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def prune_case(small_scene):
    from model_matching_b200 import Context
    sc, mpos, mnrm = small_scene
    ctx = Context(0)
    ctx.upload_model(mpos, mnrm)
    ctx.upload_scene(sc["pos"], sc["nrm"], sc["cls"])
    # S1-style: 1 % near-truth poses; H inside the heavy-first range (32 768 .. 300 000)
    T, near = synth.make_hypotheses(200000, sc["pos"], mpos, sc["gt_R"], sc["gt_t"], seed=31, near_fraction=0.01)
    yield ctx, sc, mpos, mnrm, T, near
    ctx.close()


def _full(ctx, T):
    """unpruned per-hypothesis results of the same context"""
    import torch
    dT = torch.from_numpy(np.ascontiguousarray(T, np.float32)).cuda()
    lcp = torch.empty(max(len(T), 1), dtype=torch.float32, device="cuda")
    inl = torch.empty(max(len(T), 1), dtype=torch.int32, device="cuda")
    ctx.score_lcp_device(dT.data_ptr(), len(T), lcp.data_ptr(), inl.data_ptr())
    torch.cuda.synchronize()
    return lcp.cpu().numpy()[:len(T)], inl.cpu().numpy()[:len(T)]


def _pruned(ctx, T, K, off=0):
    import torch
    dT = torch.from_numpy(np.ascontiguousarray(T, np.float32).reshape(-1)).cuda()
    drec = torch.zeros(K * 64, dtype=torch.uint8, device="cuda")
    ctx.score_sharded_device(dT.data_ptr(), len(T), off, K, drec.data_ptr())
    torch.cuda.synchronize()
    return drec.cpu().numpy().view(sharding.RECORD).copy()


def _check(ctx, T, K, off=0):
    lcp, inl = _full(ctx, T)
    want = sharding.local_records(lcp, inl, T, off, K)
    got = _pruned(ctx, T, K, off)
    assert got.tobytes() == want.tobytes()
    return lcp, got


def _rejected(ctx):
    c = ctx.counters()
    return int(c[4]), int(c[5])


@pytest.mark.parametrize("K", [1, 8, 32])
def test_s1_style_records_equal_unpruned(prune_case, K):
    ctx, sc, mpos, mnrm, T, near = prune_case
    r0 = _rejected(ctx)
    _check(ctx, T, K, off=1000)
    r1 = _rejected(ctx)
    assert (r1[0] - r0[0]) + (r1[1] - r0[1]) > 0, "the S1-style list must exercise the rejection"


@pytest.mark.parametrize("where", ["end", "front"])
def test_near_truth_poses_at_one_end(prune_case, where):
    ctx, sc, mpos, mnrm, T, near = prune_case
    mask = np.zeros(len(T), bool)
    mask[near] = True
    order = np.concatenate([np.flatnonzero(~mask), np.flatnonzero(mask)])
    if where == "front":
        order = order[::-1]
    _check(ctx, T[order], 32)


@pytest.mark.parametrize("H", [20000, 40000, 299999])
def test_list_sizes_around_the_heavy_first_range(prune_case, H):
    ctx, sc, mpos, mnrm, T, near = prune_case
    _check(ctx, np.concatenate([T, T])[:H], 32)


def test_duplicates_and_ties_at_the_kth_place(prune_case):
    ctx, sc, mpos, mnrm, T, near = prune_case
    K = 8
    T2 = T[:60000].copy()
    lcp, _ = _full(ctx, T2)
    order = np.lexsort((np.arange(lcp.size), -lcp.astype(np.float64)))
    best, kth = T2[order[0]].copy(), T2[order[K - 1]].copy()
    for i in (0, len(T2) - 1, 777, 31337, 45000):     # strongest hypothesis at the first, last and scattered indices
        T2[i] = best
    for i in (5, 12345, 40000, 59990):                 # copies of the one at the K-th place: index breaks the tie
        T2[i] = kth
    lcp2, got = _check(ctx, T2, K)
    assert (lcp2 == lcp2[5]).sum() >= 4
    _check(ctx, T2, 32)


def test_rejected_fits_mixed_in(prune_case):
    ctx, sc, mpos, mnrm, T, near = prune_case
    T2 = T[:100000].copy()
    T2[::7] = np.nan
    _check(ctx, T2, 32)


def test_short_and_empty_lists(prune_case):
    ctx, sc, mpos, mnrm, T, near = prune_case
    _check(ctx, T[near[:5]], 32)         # H < K
    _check(ctx, T[:20], 32)
    got = _pruned(ctx, T[:0], 16)        # H = 0
    assert (got["index"] == -1).all() and (got["lcp"] == 0).all()


def test_scene_with_all_weights_zero(small_scene):
    from model_matching_b200 import Context
    sc, mpos, mnrm = small_scene
    T, _ = synth.make_hypotheses(50000, sc["pos"], mpos, sc["gt_R"], sc["gt_t"], seed=32, near_fraction=0.01)
    ctx = Context(0)
    try:
        ctx.upload_model(mpos, mnrm)
        ctx.upload_scene(sc["pos"], sc["nrm"], np.zeros_like(sc["cls"]))
        _, got = _check(ctx, T, 32)
        assert (got["index"] == -1).all()
    finally:
        ctx.close()


def test_scene_with_a_negative_weight_is_not_pruned(small_scene):
    from model_matching_b200 import Context
    sc, mpos, mnrm = small_scene
    T, _ = synth.make_hypotheses(100000, sc["pos"], mpos, sc["gt_R"], sc["gt_t"], seed=33, near_fraction=0.01)
    cls = sc["cls"].copy()
    cls[123] = -0.25
    ctx = Context(0)
    try:
        ctx.upload_model(mpos, mnrm)
        ctx.upload_scene(sc["pos"], sc["nrm"], cls)
        _check(ctx, T, 32)
        assert _rejected(ctx) == (0, 0)
    finally:
        ctx.close()


def test_rejection_counters_only_move_on_the_top_k_path(prune_case):
    import torch
    ctx, sc, mpos, mnrm, T, near = prune_case
    _pruned(ctx, T, 32)
    before = _rejected(ctx)
    assert sum(before) > 0
    _full(ctx, T)
    dT = torch.from_numpy(T).cuda()
    ctx.score_counters(dT.data_ptr(), len(T))
    assert _rejected(ctx) == before


def test_group_without_per_hypothesis_outputs(small_scene):
    import torch
    from model_matching_b200 import Group
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    sc, mpos, mnrm = small_scene
    T, _ = synth.make_hypotheses(200000, sc["pos"], mpos, sc["gt_R"], sc["gt_t"], seed=34, near_fraction=0.01)
    g = Group([0, 1])
    try:
        g.upload_model(mpos, mnrm)
        g.upload_scene(sc["pos"], sc["nrm"], sc["cls"])
        rec_all, lcp, inl = g.score_best(T, K=32, want_all=True)
        rec = g.score_best(T, K=32)
        assert rec.tobytes() == rec_all.tobytes() == sharding.local_records(lcp, inl, T, 0, 32).tobytes()
    finally:
        g.close()


@pytest.mark.parametrize("n_model", [250, 1024, 1100])
def test_model_sizes(small_scene, n_model):
    """a partly padded last mask word (250), one full 32-word window (1024), two windows (1100)"""
    from model_matching_b200 import Context
    sc, _, _ = small_scene
    mpos, mnrm = synth.make_model(n_model)
    T, _ = synth.make_hypotheses(60000, sc["pos"], mpos, sc["gt_R"], sc["gt_t"], seed=35, near_fraction=0.01)
    ctx = Context(0)
    try:
        ctx.upload_model(mpos, mnrm)
        ctx.upload_scene(sc["pos"], sc["nrm"], sc["cls"])
        _check(ctx, T, 32)
        assert sum(_rejected(ctx)) > 0
    finally:
        ctx.close()


def test_weights_replaced_after_upload(small_scene):
    """the bound follows set_class_probability: uploaded with half the weights, scored with the real ones"""
    from model_matching_b200 import Context
    sc, mpos, mnrm = small_scene
    T, _ = synth.make_hypotheses(100000, sc["pos"], mpos, sc["gt_R"], sc["gt_t"], seed=36, near_fraction=0.01)
    ctx = Context(0)
    try:
        ctx.upload_model(mpos, mnrm)
        ctx.upload_scene(sc["pos"], sc["nrm"], sc["cls"] * np.float32(0.5))
        ctx.set_class_probability(sc["cls"])
        _check(ctx, T, 32)
        assert sum(_rejected(ctx)) > 0
        cls = sc["cls"].copy()
        cls[7] = -1.0                    # a negative weight set after the upload turns pruning off
        ctx.set_class_probability(cls)
        before = _rejected(ctx)
        _check(ctx, T, 32)
        assert _rejected(ctx) == before
    finally:
        ctx.close()


def test_instance_prior_growth_turns_pruning_off(small_scene):
    """instance sampling rewrites weights in place as dispersion * w: a dispersion above 1 can lift them
    over the uploaded maximum, so the scene is no longer pruned"""
    from model_matching_b200 import Context
    sc, mpos, mnrm = small_scene
    n = len(sc["pos"])
    pix = np.stack([np.arange(n) % 480, np.arange(n) % 640], -1).astype(np.int32)
    edge = np.full((480, 640), 255, np.uint8)
    edge[::30] = 0
    T, _ = synth.make_hypotheses(100000, sc["pos"], mpos, sc["gt_R"], sc["gt_t"], seed=37, near_fraction=0.01)
    ctx = Context(0)
    try:
        ctx.upload_model(mpos, mnrm)
        ctx.upload_scene(sc["pos"], sc["nrm"], sc["cls"], pix)
        ctx.upload_edge_map(edge)
        for b in range(1, 4):
            ctx.sample_instance_base(3, b, dispersion=3.0)
        before = _rejected(ctx)
        _check(ctx, T, 32)
        assert _rejected(ctx) == before
    finally:
        ctx.close()
