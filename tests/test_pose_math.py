"""The pinned pose distance (csrc/stocs_pose_math.h, which clustering::get_pose_diff and the clustering
kernels share) against the same arithmetic with libm's atan2 / asin, evaluated with numpy (CPU only).

The only thing the pinned statement changes on the host is atan2 / asin: libm -> the binary64 series of
stocs_math.h.  The numpy model below repeats every binary32 step of reference src/pose_clustering.cpp:5-72
in the same order and calls numpy's (libm's) arctan2 / arcsin, so the two may differ only by the last
bits of those functions, which the binary32 rounding hides almost always."""
import os
import subprocess

import numpy as np
import pytest

from model_matching_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "model_matching_b200", "host", "test_clustering")
F = np.float32


def _pinned(Tt, Tb, sym):
    """get_pose_diff of the host shim (column-major 16-float poses) -> (rot, trans) float32"""
    n = len(Tt)
    head = np.array([n], np.int64).tobytes() + np.array(sym, np.float32).tobytes()
    out = subprocess.run([EXE, "diff"], input=head + np.ascontiguousarray(Tt, np.float32).tobytes()
                         + np.ascontiguousarray(Tb, np.float32).tobytes(), capture_output=True, check=True).stdout
    r = np.frombuffer(out, np.float32)
    return r[:n], r[n:]


def _libm(Tt, Tb, sym):
    """the same statement in numpy: binary32 steps in the host order, libm atan2 / asin in binary64"""
    a = lambda T, i, j: T[:, j * 4 + i]          # (row i, col j) of column-major poses
    m = [[a(Tt, i, j) for j in range(3)] for i in range(3)]
    c00 = m[1][1] * m[2][2] - m[1][2] * m[2][1]
    c01 = m[1][2] * m[2][0] - m[1][0] * m[2][2]
    c02 = m[1][0] * m[2][1] - m[1][1] * m[2][0]
    det = (m[0][0] * c00 + m[0][1] * c01) + m[0][2] * c02
    idet = F(1) / det
    ti = [[c00 * idet, (m[0][2] * m[2][1] - m[0][1] * m[2][2]) * idet, (m[0][1] * m[1][2] - m[0][2] * m[1][1]) * idet],
          [c01 * idet, (m[0][0] * m[2][2] - m[0][2] * m[2][0]) * idet, (m[0][2] * m[1][0] - m[0][0] * m[1][2]) * idet],
          [c02 * idet, (m[0][1] * m[2][0] - m[0][0] * m[2][1]) * idet, (m[0][0] * m[1][1] - m[0][1] * m[1][0]) * idet]]
    rd = [[ti[i][0] * a(Tb, 0, j) + (ti[i][1] * a(Tb, 1, j) + ti[i][2] * a(Tb, 2, j)) for j in range(3)] for i in range(3)]
    # Shoemake, all four branches, selected per pair
    tr = (rd[0][0] + rd[1][1]) + rd[2][2]
    with np.errstate(invalid="ignore", divide="ignore"):
        t = np.sqrt(tr + F(1)); h = F(0.5) / t
        q = {"w": F(0.5) * t, "x": (rd[2][1] - rd[1][2]) * h, "y": (rd[0][2] - rd[2][0]) * h, "z": (rd[1][0] - rd[0][1]) * h}
        i_sel = np.where(rd[1][1] > rd[0][0], 1, 0)
        i_sel = np.where(rd[2][2] > np.choose(i_sel, [rd[0][0], rd[1][1]]), 2, i_sel)
        for i in range(3):
            j, k = (i + 1) % 3, (i + 2) % 3
            tt = np.sqrt(((rd[i][i] - rd[j][j]) - rd[k][k]) + F(1)); hh = F(0.5) / tt
            qq = [None] * 3
            qq[i] = F(0.5) * tt
            qq[j] = (rd[j][i] + rd[i][j]) * hh
            qq[k] = (rd[k][i] + rd[i][k]) * hh
            sel = ~(tr > 0) & (i_sel == i)
            q["w"] = np.where(sel, (rd[k][j] - rd[j][k]) * hh, q["w"])
            for name, v in zip("xyz", qq):
                q[name] = np.where(sel, v, q[name])
    qw, qx, qy, qz = (q[c].astype(F) for c in "wxyz")
    d = lambda v: v.astype(np.float64)
    e0 = np.arctan2(2.0 * d(qw * qx + qy * qz), 1.0 - 2.0 * d(qx * qx + qy * qy)).astype(F)
    sinp = 2.0 * d(qw * qy - qz * qx)
    with np.errstate(invalid="ignore"):
        e1 = np.where(np.abs(sinp) >= 1, np.copysign(np.pi / 2, sinp), np.arcsin(np.clip(sinp, -1, 1))).astype(F)
    e2 = np.arctan2(2.0 * d(qw * qz + qx * qy), 1.0 - 2.0 * d(qy * qy + qz * qz)).astype(F)
    e = [np.abs((d(x) * 180.0 / np.pi).astype(F)) for x in (e0, e1, e2)]
    for k in range(3):
        if sym[k] == 90:
            e[k] = np.abs(e[k] - F(90)); e[k] = np.minimum(e[k], F(90) - e[k])
        elif sym[k] == 180:
            e[k] = np.minimum(e[k], F(180) - e[k])
        elif sym[k] == 360:
            e[k] = np.zeros_like(e[k])
    rot = np.maximum(np.maximum(e[0], e[1]), e[2])
    dx, dy, dz = (d(a(Tb, r, 3) - a(Tt, r, 3)) for r in range(3))
    branch = np.where(tr > 0, 3, i_sel)            # 3: trace > 0, else the largest diagonal entry
    return rot, np.sqrt((dx * dx + dy * dy) + dz * dz).astype(F), branch, np.abs(sinp) >= 1


def _poses(rng, n):
    """pairs whose relative rotation is random, or near 180 degrees about x / y / z (every quaternion
    branch), or at exactly +-90 degrees of pitch; translations from nearby to far"""
    Rt = synth.random_rotations(rng, n)
    kind = np.arange(n) % 6
    Rrel = synth.random_rotations(rng, n)
    for i in np.flatnonzero((kind >= 1) & (kind <= 3)):
        axis = np.zeros(3); axis[kind[i] - 1] = 1.0
        Rrel[i] = synth.axis_angle(axis + rng.normal(0, 0.02, 3), np.pi - abs(rng.normal(0, 0.05)))
    for i in np.flatnonzero(kind == 4):
        s = 1.0 if rng.random() < 0.5 else -1.0      # pitch of exactly +-90 degrees, roll / yaw random
        Rrel[i] = synth.axis_angle([0, 0, 1], rng.uniform(-np.pi, np.pi)) @ np.array([[0, 0, s], [0, 1, 0], [-s, 0, 0]])
    Tt, Tb = np.zeros((n, 4, 4), F), np.zeros((n, 4, 4), F)
    Tt[:, :3, :3] = Rt
    Tb[:, :3, :3] = Rt @ Rrel
    # kind 5: the base is the test pose rotated by a small angle (the clustering's deciding range)
    for i in np.flatnonzero(kind == 5):
        Tb[i, :3, :3] = synth.axis_angle(rng.normal(size=3), np.deg2rad(rng.uniform(0, 20))) @ Rt[i]
    Tt[:, :3, 3] = rng.uniform(-0.5, 0.5, (n, 3))
    Tb[:, :3, 3] = Tt[:, :3, 3] + rng.normal(0, 10.0 ** rng.uniform(-4, 0, (n, 1)), (n, 3))
    Tt[:, 3, 3] = Tb[:, 3, 3] = 1
    # exact +-90 degree pitch with exact matrices: test = identity
    Tt[:8, :3, :3] = np.eye(3)
    for i in range(8):
        s = 1.0 if i % 2 == 0 else -1.0
        Tb[i, :3, :3] = np.array([[0, 0, s], [0, 1, 0], [-s, 0, 0]])
    col = lambda T: np.ascontiguousarray(T.transpose(0, 2, 1).reshape(n, 16))
    return col(Tt), col(Tb)


@pytest.mark.parametrize("sym", [(0, 0, 0), (90, 90, 90), (180, 180, 180), (360, 360, 360), (90, 180, 360), (0, 180, 90)])
def test_pinned_pose_diff_matches_libm(sym):
    if not os.path.exists(EXE):
        pytest.skip("host layer not built")
    rng = np.random.Generator(np.random.Philox(11 + int(sum(sym))))
    n = 20000
    Tt, Tb = _poses(rng, n)
    r, t = _pinned(Tt, Tb, sym)
    wr, wt, branch, clamped = _libm(Tt, Tb, sym)
    assert np.bincount(branch, minlength=4).min() >= 1000 and clamped.sum() >= 4   # every branch is exercised
    assert np.array_equal(t.view(np.uint32), wt.view(np.uint32))
    assert np.isfinite(r).all() and np.isfinite(wr).all()
    err = np.abs(r.astype(np.float64) - wr)
    assert err.max() <= 1e-4, err.max()
    differ = int((r != wr).sum())
    print(f"sym {sym}: {differ} of {n} rotation errors differ from libm's in binary32, max {err.max():.3g} degree")
    assert differ <= n // 1000
