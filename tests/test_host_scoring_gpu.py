"""Host-buffer scoring calls (csrc/capi.cu, stocs_score_host): stocs_b200_score_sharded from pageable
transforms, from page-locked ones read in place and from page-locked ones staged through HBM must
agree with stocs_b200_score_lcp bit for bit, and every call leaves the resident lcp array that
stocs_b200_reduce_best(NULL) answers from."""
import ctypes as C

import numpy as np
import pytest

from model_matching_b200 import sharding, synth

pytestmark = pytest.mark.gpu
H = 150_000            # above the 2^16 threshold of the chunked (staged) path
K = 32
OFF = 987_654_321      # global index of the first local hypothesis


@pytest.fixture(scope="module")
def case(gpu_ctx, small_scene):
    sc, mpos, mnrm = small_scene
    T, _ = synth.make_hypotheses(H, sc["pos"], mpos, sc["gt_R"], sc["gt_t"], seed=5, near_fraction=0.03)
    gpu_ctx.upload_model(mpos, mnrm)
    gpu_ctx.upload_scene(sc["pos"], sc["nrm"], sc["cls"])
    lcp, inl = gpu_ctx.score_lcp(T)
    want = sharding.local_records(lcp, inl, T, OFF, K)
    assert (want["index"] >= OFF).all()          # K real winners, not empty records
    return T, lcp, inl, want


def _pinned(T):
    import torch
    return torch.from_numpy(T).pin_memory()


def _sharded_ptr(ctx, hT, want_local):
    out = np.zeros(K, sharding.RECORD)
    lcp = np.empty(H, np.float32) if want_local else None
    inl = np.empty(H, np.int32) if want_local else None
    ctx.score_sharded_ptr(hT.data_ptr(), H, OFF, K, out, None if lcp is None else lcp.ctypes.data,
                          None if inl is None else inl.ctypes.data)
    return out, lcp, inl


def _resident_best(ctx, n, k):
    """stocs_b200_reduce_best(NULL): the K best of the resident array of n results (the Python wrapper
    would pass the size of its last score_lcp call)"""
    bi, bl = C.c_int64(0), C.c_float(0)
    ti, tl = np.empty(k, np.int64), np.empty(k, np.float32)
    rc = ctx._L.stocs_b200_reduce_best(ctx.h, None, n, k, C.byref(bi), C.byref(bl), ti.ctypes.data, tl.ctypes.data)
    assert rc == 0, ctx._L.stocs_b200_last_error(ctx.h)
    return bi.value, bl.value, ti, tl


def _same_best(got, want, k):
    assert got[0] == want[0] and got[1] == want[1]
    assert np.array_equal(got[2], want[2][:k]) and np.array_equal(got[3], want[3][:k])


def test_sharded_input_paths_agree_with_score_lcp(gpu_ctx, case, monkeypatch):
    T, lcp, inl, want = case
    hT = _pinned(T)
    runs = [gpu_ctx.score_sharded(T, OFF, K, want_local=True),     # pageable: staged
            _sharded_ptr(gpu_ctx, hT, True)]                        # page-locked: read in place
    monkeypatch.setenv("STOCS_NO_ZERO_COPY", "1")
    runs.append(_sharded_ptr(gpu_ctx, hT, True))                    # page-locked, staged
    for rec, l, i in runs:
        assert rec.tobytes() == want.tobytes()
        assert np.array_equal(l.view(np.uint32), lcp.view(np.uint32)) and np.array_equal(i, inl)


def test_sharded_records_only_leave_the_resident_array(gpu_ctx, case, monkeypatch):
    T, lcp, inl, want = case
    best = gpu_ctx.reduce_best(lcp, K=32)
    hT = _pinned(T)
    for staged in (False, True):
        if staged:
            monkeypatch.setenv("STOCS_NO_ZERO_COPY", "1")
        gpu_ctx.reduce_best(np.zeros(H, np.float32))   # a resident array of the same size, to be replaced
        rec, _, _ = _sharded_ptr(gpu_ctx, hT, False)
        assert rec.tobytes() == want.tobytes()
        for k in (1, 7, 32):
            _same_best(_resident_best(gpu_ctx, H, k), best, k)
    # the pageable path without per-hypothesis outputs
    gpu_ctx.reduce_best(np.zeros(H, np.float32))
    assert gpu_ctx.score_sharded(T, OFF, K).tobytes() == want.tobytes()
    _same_best(_resident_best(gpu_ctx, H, 32), best, 32)
    # an empty block scores nothing: K empty records, and the resident array stays the last call's
    rec = gpu_ctx.score_sharded(T[:0], OFF, K)
    assert rec.tobytes() == sharding.empty_records(K).tobytes()
    for k in (1, 7, 32):
        _same_best(_resident_best(gpu_ctx, H, k), best, k)


def test_reduce_best_explicit_then_resident(gpu_ctx, case):
    _, lcp, _, _ = case
    for n in (H, 70_000, 5, 0):
        want = gpu_ctx.reduce_best(lcp[:n], K=32)
        wi, wv = sharding.merge_topk(np.arange(n), lcp[:n], 32)
        assert np.array_equal(want[2], wi) and np.array_equal(want[3].view(np.uint32), wv.view(np.uint32))
        assert (want[0], want[1]) == (int(wi[0]), float(wv[0]))
        for k in (1, 7, 32):
            _same_best(_resident_best(gpu_ctx, n, k), want, k)
            _same_best(gpu_ctx.reduce_best(lcp[:n], K=k), want, k)
