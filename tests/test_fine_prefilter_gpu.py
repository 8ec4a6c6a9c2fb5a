"""Fine prefilter of the device top-K path (csrc/score.cu, survivor_count_kernel on the scene's fine
occupancy map): a top-K launch of more than 300 000 hypotheses orders and stops its claims by each
hypothesis's count of model points whose fine block (2^fine_shift cells per axis) is occupied.  That count
must never exceed loop 1's coarse count, never fall below the inliers the unpruned scorer finds, and the
K records must equal, bit for bit, those built from the unpruned per-hypothesis results."""
import os

import numpy as np
import pytest

from model_matching_b200 import sharding, synth

pytestmark = pytest.mark.gpu

N = 320000   # above the 300 000 hypotheses from which a top-K launch takes the survivor order


def _dev(T):
    import torch
    return torch.from_numpy(np.ascontiguousarray(T, np.float32).reshape(-1)).cuda()


def _counts(ctx, T):
    dT = _dev(T)
    coarse = ctx.debug_survivor_counts(dT.data_ptr(), len(T))
    fine, shifts = ctx.debug_survivor_counts(dT.data_ptr(), len(T), fine=True)
    return coarse, fine, shifts


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
    """bounds per hypothesis, then records bit-identical to the unpruned path; returns the shifts"""
    lcp, inl = _full(ctx, T)
    coarse, fine, shifts = _counts(ctx, T)
    assert (fine <= coarse).all()
    assert (fine >= inl).all()
    if shifts[0] == shifts[1]:
        assert (fine == coarse).all()
    want = sharding.local_records(lcp, inl, T, 0, K)
    got = _pruned(ctx, T, K)
    assert got.tobytes() == want.tobytes()
    return shifts


def _context(sc, mpos, mnrm, fine_bits=None):
    from model_matching_b200 import Context
    ctx = Context(0)
    ctx.upload_model(mpos, mnrm)
    old = os.environ.get("STOCS_FINE_BITS")
    if fine_bits is not None:
        os.environ["STOCS_FINE_BITS"] = str(fine_bits)
    try:
        ctx.upload_scene(sc["pos"], sc["nrm"], sc["cls"])
    finally:
        if fine_bits is not None:
            if old is None:
                del os.environ["STOCS_FINE_BITS"]
            else:
                os.environ["STOCS_FINE_BITS"] = old
    return ctx


@pytest.fixture(scope="module")
def small_case(small_scene):
    sc, mpos, mnrm = small_scene
    ctx = _context(sc, mpos, mnrm)
    T, near = synth.make_hypotheses(N, sc["pos"], mpos, sc["gt_R"], sc["gt_t"], seed=51, near_fraction=0.01)
    yield ctx, sc, mpos, T, near
    ctx.close()


def test_small_scene_has_a_finer_map(small_case):
    ctx, sc, mpos, T, near = small_case
    coarse, fine, (fs, cs) = _counts(ctx, T)
    assert 2 <= fs < cs
    assert fine.sum() < coarse.sum()
    assert fine[near].mean() > fine.mean()        # near-truth poses keep more of the model


def test_small_scene_records(small_case):
    ctx, sc, mpos, T, near = small_case
    _check(ctx, T)
    _check(ctx, T, K=1)


def test_non_finite_and_huge_transforms_count_every_point(small_case):
    ctx, sc, mpos, T, near = small_case
    T2 = T[:1000].copy()
    T2[::7] = np.nan
    T2[3, 12] = np.inf
    T2[5, 0] = 1e38
    _, fine, _ = _counts(ctx, T2)
    bad = np.zeros(len(T2), bool)
    bad[::7] = bad[3] = bad[5] = True
    assert (fine[bad] == len(mpos)).all()
    assert (fine[~bad] == _counts(ctx, T2[~bad])[1]).all()


def test_model_across_apron_and_border(small_case):
    """translations on the faces, edges and corners of the scene's box, a few eps in and out of it, and
    far outside the grid on either side"""
    ctx, sc, mpos, T, near = small_case
    rng = np.random.default_rng(52)
    lo, hi = sc["pos"].min(0), sc["pos"].max(0)
    T2 = T.copy()
    pick = rng.integers(0, 2, size=(N, 3))
    edge = np.where(pick == 1, hi, lo)
    # one axis free inside the box for a third of the rows (faces and edges), all on the box otherwise
    free = rng.integers(0, 3, size=N)
    inside = lo + rng.random((N, 3)) * (hi - lo)
    rows = np.arange(N) % 3 == 0
    edge[rows, free[rows]] = inside[rows, free[rows]]
    t = edge + rng.uniform(-0.12, 0.12, size=(N, 3))
    far = np.arange(N) % 50 == 1
    t[far] += rng.choice([-1.0, 1.0], size=(far.sum(), 3)) * 10.0
    T2[:, 12:15] = t.astype(np.float32)
    T2 = np.concatenate([T2[: N - 4000], T[near[:4000]]])
    _check(ctx, T2)


def test_tiny_and_subnormal_model_coordinates(small_scene):
    sc, mpos, mnrm = small_scene
    m = mpos.copy()
    m[:64] *= np.float32(1e-39)      # subnormal in binary32
    m[64:96] = 0.0
    m[96:128] *= np.float32(1e-20)
    m[128:136] = np.float32(1.4e-45)  # the smallest subnormal
    ctx = _context(sc, m, mnrm)
    try:
        T, _ = synth.make_hypotheses(N, sc["pos"], mpos, sc["gt_R"], sc["gt_t"], seed=53, near_fraction=0.01)
        fs, cs = _check(ctx, T)
        assert fs < cs
    finally:
        ctx.close()


def test_scene_at_brick_scale_has_one_map():
    """a scene small enough that the coarse map is already at brick scale: d = 0, the count is loop 1's"""
    sc = synth.make_scene(n_points=20000, extent=(0.25, 0.2, 0.2), n_objects=3, seed=54)
    mpos, mnrm = synth.make_model(256)
    ctx = _context(sc, mpos, mnrm)
    try:
        T, _ = synth.make_hypotheses(N, sc["pos"], mpos, sc["gt_R"], sc["gt_t"], seed=55, near_fraction=0.01)
        assert _check(ctx, T) == (2, 2)
    finally:
        ctx.close()


def test_finer_map_over_budget_falls_back_to_the_coarse_one(small_scene):
    sc, mpos, mnrm = small_scene
    ctx = _context(sc, mpos, mnrm, fine_bits=1024)
    try:
        T, _ = synth.make_hypotheses(N, sc["pos"], mpos, sc["gt_R"], sc["gt_t"], seed=56, near_fraction=0.01)
        fs, cs = _check(ctx, T)
        assert fs == cs > 2
    finally:
        ctx.close()


def test_s1_workload():
    """S1 (bench.py): 2^20 scene points, 512 model points, 10^6 hypotheses"""
    import bench
    from model_matching_b200 import Context
    sc, mpos, mnrm, T = bench.workload(0, 1000000)
    ctx = Context(0)
    try:
        ctx.upload_model(mpos, mnrm)
        ctx.upload_scene(sc["pos"], sc["nrm"], sc["cls"])
        fs, cs = _check(ctx, T)
        assert fs < cs
        c0 = ctx.counters()
        _pruned(ctx, T, 32)
        c1 = ctx.counters()
        assert (c1[4] - c0[4]) + (c1[5] - c0[5]) + (c1[8] - c0[8]) <= len(T)
    finally:
        ctx.close()
