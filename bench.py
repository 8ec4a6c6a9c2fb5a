#!/usr/bin/env python
"""bench.py -- hypotheses scored / second on the synthetic S1 workload (BASELINE.json configs[3]).

One "step" = one pass of the hot path over one batch: score H = 10^6 rigid-transform hypotheses
(|M| = 512 model points each) against the 1,048,576-point scene and reduce them to the K = 32 best
64-byte records.  With N > 1 GPUs the 10^6 hypotheses are SHARDED (strong scaling, the named
config): every rank holds a replica of the scene index, scores ceil(H/N) hypotheses, and ONE
ncclAllGather + a device merge give every rank the global top-K -- all inside the C ABI call
stocs_b200_score_sharded_device.  The weak-scaling figure (10^6 per GPU) is reported under `extra`.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload s1|s2]
                  [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for how each field is produced.
--dump-outputs DIR writes what the last timed step returned to its caller as DIR/<name>.npy
(rank 0; integers widened to float64, which holds them exactly).  The inputs are seeded, so two
builds run with the same arguments can be compared output for output.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the tree may be read-only: nothing is cached in it

N_SCENE = 1 << 20
N_MODEL = 512
H_TOTAL = 1_000_000
TOPK = 32
METRIC = "hypotheses_scored_per_second"
UNIT = "hypotheses/s"


def algorithmic_bytes_per_hypothesis(M):
    # SURVEY.md section 8(d): 64 B per NN query (8 cell descriptors x 4 B + one 16 B candidate
    # position + one 16 B attribute record) x |M| queries + 48 B transform in + 8 B results out.
    return 56 + 64 * M


def dump_outputs(dirname, arrays):
    """--dump-outputs: each array as <dirname>/<name>.npy, float32 / float64 only."""
    if not dirname:
        return
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        if a.dtype not in (np.float32, np.float64):
            a = a.astype(np.float64)
        np.save(os.path.join(dirname, name + ".npy"), a)


def record_arrays(rec, prefix=""):
    """the fields of a RECORD array (the top-K a scoring call returns), one array per field"""
    return {f"{prefix}topk_{f}": rec[f] for f in ("index", "lcp", "inliers", "T")}


def workload(rank, H):
    from model_matching_b200 import synth
    sc = synth.make_scene(n_points=N_SCENE, seed=1234)
    mpos, mnrm = synth.make_model(N_MODEL)
    T, _ = synth.make_hypotheses(H, sc["pos"], mpos, sc["gt_R"], sc["gt_t"], seed=4321 + rank)
    return sc, mpos, mnrm, T


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 50 ms.  Started before the warm-up (its
    first sample can take a second); only samples stamped inside the timed region are reported."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-i", str(self.gpu), "-lms", "50"], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def wait_first_sample(self, timeout=3.0):
        t0 = time.time()
        while self.p is not None and time.time() - t0 < timeout:
            if os.path.getsize(self.f.name) > 0:
                return
            time.sleep(0.02)

    def stop(self, t_begin=None, t_end=None):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)
        self.p.terminate()
        self.p.wait()
        self.f.flush()
        self.f.seek(0)
        import datetime
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = []
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                ts = None
                try:
                    ts = datetime.datetime.strptime(c[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                except ValueError:
                    pass
                rows.append((ts, float(c[1]), float(c[2]),
                             [nm for nm, v in zip(names, c[5:9]) if v.lower().startswith("active")]))
            except ValueError:
                continue
        os.unlink(self.f.name)
        inside = [r for r in rows if t_begin is not None and r[0] is not None and t_begin - 0.05 <= r[0] <= t_end + 0.05]
        window = "timed region"
        if not inside:  # clock skew / unparsable stamps: fall back to every sample (warm-up included)
            inside, window = rows, "whole run"
        sm, smax = [r[1] for r in inside], [r[2] for r in inside]
        reasons = sorted({nm for r in inside for nm in r[3]})
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(smax)) if smax else None, "reasons": reasons,
                "samples": len(sm), "window": window}


def cpu_baseline(sc, mpos, mnrm, T, seconds_target=15.0):
    """The CPU oracle (port of the reference's kd-tree LCP loop) on all host cores, bounded sample."""
    import oracle
    cores = os.cpu_count() or 1
    est = oracle.Estimator(sc["pos"], sc["nrm"], sc["cls"], mpos, mnrm)
    n0 = min(len(T), 2000 * cores)
    t0 = time.perf_counter()
    est.score(T[:n0], threads=cores)
    dt = time.perf_counter() - t0
    n = int(min(len(T), max(n0, n0 * seconds_target / max(dt, 1e-6))))
    t0 = time.perf_counter()
    lcp, inl = est.score(T[:n], threads=cores)
    dt = time.perf_counter() - t0
    n1 = min(len(T), 20000)   # the reference itself is single-threaded: report that figure too
    t0 = time.perf_counter()
    est.score(T[:n1], threads=1)
    dt1 = time.perf_counter() - t0
    return est, {"value": n / dt, "unit": UNIT, "cores": cores, "kind": "port",
                 "sample": f"first {n} of the {len(T)} hypotheses of the same workload, {cores} threads, {dt:.1f} s",
                 "single_thread": {"value": n1 / dt1, "unit": UNIT, "sample": f"first {n1} hypotheses, 1 thread, {dt1:.1f} s"}}, (lcp, inl, n)


def pose_latency_fixture(ctx, name, label):
    """GPU-only figures for another of the reference's example scenes (tests/golden/golden_<name>.npz):
    upload + index, model table, fused pipeline, and scoring-only rate on the fixture's own
    hypothesis list (a few thousand transforms: the launch-bound regime of the reference CLI)."""
    path = os.path.join(ROOT, "tests", "golden", f"golden_{name}.npz")
    if not os.path.exists(path):
        return None
    with np.load(path) as z:
        g = {k: np.ascontiguousarray(z[k]) for k in ("mpos", "mnrm", "spos", "snrm", "scls", "spix", "T", "inliers")}
    ctx.upload_model(g["mpos"], g["mnrm"])
    ctx.upload_scene(g["spos"], g["snrm"], g["scls"], g["spix"])
    tm, tu = [], []
    for _ in range(5):
        t0 = time.perf_counter(); ctx.upload_model(g["mpos"], g["mnrm"]); tm.append(time.perf_counter() - t0)
        t0 = time.perf_counter(); ctx.upload_scene(g["spos"], g["snrm"], g["scls"], g["spix"]); tu.append(time.perf_counter() - t0)
    ctx.run_pipeline(1, 100, 200)
    tp, res = [], None
    for seed in range(2, 12):
        best = 1e9
        for _ in range(3):
            t0 = time.perf_counter(); res = ctx.run_pipeline(seed, 100, 200); best = min(best, time.perf_counter() - t0)
        tp.append(best)
    T = np.ascontiguousarray(g["T"], np.float32)
    lcp, inl = ctx.score_lcp(T)
    ts = []
    for _ in range(10):
        t0 = time.perf_counter(); ctx.score_lcp(T); ts.append(time.perf_counter() - t0)
    return {"workload": "%s (|S|=%d, |M|=%d), 100 bases, <=200 sets/base" % (label, len(g["spos"]), len(g["mpos"])),
            "gpu_ms_per_pose": 1e3 * float(np.median(tp)), "gpu_upload_index_ms": 1e3 * float(np.median(tu)),
            "gpu_model_table_ms": 1e3 * float(np.median(tm)), "transforms_scored": int(res.n_transforms),
            "scoring_only_hyp_per_s": len(T) / float(np.median(ts)), "scoring_only_hypotheses": int(len(T)),
            "scoring_matches_fixture": bool(np.array_equal(inl, g["inliers"]))}


def pose_latency_packed(ctx):
    """configs[2]: the reference's `packed` example, INSTANCE mode (edge map present): bases are
    sequentially coupled (src/stocs.cpp:572-580), so sampling is one launch per base; congruent sets,
    <= 200 fits per base, scoring and the best-pose reduction are batched as in class mode."""
    import cv2
    path = os.path.join(ROOT, "tests", "golden", "golden_packed.npz")
    ef = os.path.join(ROOT, "tests", "golden", "examples", "packed", "probability_maps", "edge.png")
    if not (os.path.exists(path) and os.path.exists(ef)):
        return None
    with np.load(path) as z:
        g = {k: np.ascontiguousarray(z[k]) for k in ("mpos", "mnrm", "spos", "snrm", "scls", "spix")}
    edge = cv2.imread(ef, cv2.IMREAD_GRAYSCALE)

    def once(seed):
        t = {}
        t0 = time.perf_counter()
        ctx.upload_model(g["mpos"], g["mnrm"]); ctx.upload_scene(g["spos"], g["snrm"], g["scls"], g["spix"]); ctx.upload_edge_map(edge)
        t["upload_index_ms"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        bases, invs = [], []
        for b in range(1, 101):
            ok, ids, inv, _ = ctx.sample_instance_base(seed, b, 0.9, want_mask=False)
            if ok:
                bases.append(ids.copy()); invs.append(inv.copy())
        t["sampling_ms"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        n_sets = n_T = 0
        best = (-1, 0.0)
        if bases:
            bases, invs = np.array(bases), np.array(invs)
            quads, offs = ctx.find_congruent(bases, invs, cap=1 << 22)
            cnt = np.diff(offs)
            take = np.minimum(cnt, 200)
            b = np.repeat(np.arange(len(bases)), take)
            k = np.arange(int(take.sum())) - np.repeat(np.cumsum(take) - take, take)
            src = np.where(cnt[b] < 200, k, (k * cnt[b]) // 200)
            n_sets = int(cnt.sum())
            t["congruent_ms"] = time.perf_counter() - t0
            t0 = time.perf_counter()
            if len(b):
                Tc, _, ok = ctx.fit_transforms(bases[b], quads[offs[b] + src])
                lcp, _ = ctx.score_lcp(Tc[ok])
                best = ctx.reduce_best(None, K=1)[:2]
                n_T = int(ok.sum())
            t["fit_score_best_ms"] = time.perf_counter() - t0
        t.update(valid_bases=len(bases), congruent_sets=n_sets, transforms_scored=n_T, best_lcp=float(best[1]))
        return t

    once(1)
    runs = [once(s) for s in range(2, 7)]
    out = {"workload": "packed/dove example scene, instance mode (|S|=%d, |M|=%d), 100 bases, <=200 sets/base" % (len(g["spos"]), len(g["mpos"]))}
    for k in ("upload_index_ms", "sampling_ms", "congruent_ms", "fit_score_best_ms"):
        out["per_stage_driver_" + k] = 1e3 * float(np.median([r.get(k, 0.0) for r in runs]))
    out["per_stage_driver_ms_per_pose"] = out["per_stage_driver_sampling_ms"] + out["per_stage_driver_congruent_ms"] + out["per_stage_driver_fit_score_best_ms"]
    for k in ("valid_bases", "congruent_sets", "transforms_scored", "best_lcp"):
        out[k] = runs[-1][k]
    # the fused device pipeline: the 100 coupled bases enqueued back to back, quads stay on the device
    tf, tu, res = [], [], None
    for s in range(2, 9):
        t0 = time.perf_counter()
        ctx.upload_scene(g["spos"], g["snrm"], g["scls"], g["spix"]); ctx.upload_edge_map(edge)
        tu.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        res = ctx.run_pipeline_instance(s, 100, 200, 0.9)
        tf.append(time.perf_counter() - t0)
    out["gpu_ms_per_pose"] = 1e3 * float(np.median(tf[1:]))
    out["gpu_upload_index_ms"] = 1e3 * float(np.median(tu[1:]))
    out["fused"] = {"valid_bases": int(res.n_valid_bases), "congruent_sets": int(res.n_congruent_sets),
                    "transforms_scored": int(res.n_transforms), "best_lcp": float(res.best_lcp)}
    out["note"] = ("gpu_ms_per_pose: stocs_b200_run_pipeline_instance (bases are sequentially coupled -- prior decay + cached masks -- "
                   "so sampling is 100 dependent launches, enqueued back to back); per_stage_driver_*: the same work through the "
                   "per-call ABI the class shim uses (a host round trip per base, every quad returned to the host)")
    return out


def pose_latency(ctx_factory, with_cpu):
    """Secondary BASELINE metric: end-to-end ms per object pose on the reference's YCB example
    (configs[0]): 100 bases -> congruent sets -> <=200 transforms per base -> score -> best, all on
    the device (stocs_b200_run_pipeline), inputs = the scene/model point sets stocs_single uploads
    (tests/golden/golden_ycb.npz).  CPU figure: the oracle on a bounded number of bases, scaled."""
    path = os.path.join(ROOT, "tests", "golden", "golden_ycb.npz")
    if not os.path.exists(path):
        return None
    with np.load(path) as z:  # materialise: an NpzFile decompresses on every access
        g = {k: np.ascontiguousarray(z[k]) for k in ("mpos", "mnrm", "spos", "snrm", "scls", "spix")}
    ctx = ctx_factory()
    ctx.upload_model(g["mpos"], g["mnrm"])                       # first call allocates
    ctx.upload_scene(g["spos"], g["snrm"], g["scls"], g["spix"])
    tm, tu = [], []
    for _ in range(5):
        t0 = time.perf_counter()
        ctx.upload_model(g["mpos"], g["mnrm"])
        tm.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        ctx.upload_scene(g["spos"], g["snrm"], g["scls"], g["spix"])
        tu.append(time.perf_counter() - t0)
    t_model, t_upload = float(np.median(tm)), float(np.median(tu))
    ctx.run_pipeline(1, 100, 200)
    times, res = [], None
    for seed in range(2, 12):      # per seed: best of 3 (host jitter); reported: median over the 10 seeds
        best = 1e9
        for _ in range(3):
            t0 = time.perf_counter()
            res = ctx.run_pipeline(seed, 100, 200)
            best = min(best, time.perf_counter() - t0)
        times.append(best)
    # upload + pose back to back, as a frame loop runs them (upload_scene returns while the reference
    # kd-tree is still being built on a host thread; the pipeline's scoring launch collects it)
    both = []
    for seed in range(2, 12):
        best = 1e9
        for _ in range(3):
            t0 = time.perf_counter()
            ctx.upload_scene(g["spos"], g["snrm"], g["scls"], g["spix"])
            res = ctx.run_pipeline(seed, 100, 200)
            best = min(best, time.perf_counter() - t0)
        both.append(best)
    out = {"workload": "YCB 024_bowl example scene (|S|=%d, |M|=%d), 100 bases, <=200 sets/base" % (len(g["spos"]), len(g["mpos"])),
           "gpu_ms_per_pose": 1e3 * float(np.median(times)), "gpu_upload_index_ms": 1e3 * t_upload, "gpu_model_table_ms": 1e3 * t_model,
           "gpu_upload_plus_pose_ms": 1e3 * float(np.median(both)),
           "transforms_scored": int(res.n_transforms), "congruent_sets": int(res.n_congruent_sets)}
    try:  # frame -> scene cloud (src/rgbd.cpp:190-279) on the device, PNG decoding excluded
        import cv2
        d = os.path.join(ROOT, "tests", "golden", "examples", "ycb")
        depth = cv2.imread(os.path.join(d, "depth.png"), cv2.IMREAD_UNCHANGED)
        bgr = cv2.imread(os.path.join(d, "rgb.png"), cv2.IMREAD_COLOR)
        prob = cv2.imread(os.path.join(d, "probability_maps", "024_bowl.png"), cv2.IMREAD_UNCHANGED)
        K = [1066.778, 312.986, 1067.487, 241.310]
        ctx.build_scene_cloud(depth, bgr, prob, None, K, 1 / 10000.0, 0.005, 0.10)
        ts = []
        for _ in range(5):
            t0 = time.perf_counter()
            sc = ctx.build_scene_cloud(depth, bgr, prob, None, K, 1 / 10000.0, 0.005, 0.10)
            ts.append(time.perf_counter() - t0)
        out["gpu_scene_cloud_ms"] = 1e3 * float(np.median(ts))
        out["scene_cloud_points"] = int(len(sc["pos"]))
    except Exception as e:  # cv2 missing or data absent: the headline numbers do not depend on it
        out["gpu_scene_cloud_ms"] = None
        out["scene_cloud_error"] = str(e)[:100]
    try:  # a1 alone (SURVEY 8d, S1): synthetic 640x480 depth frame, plane at 1 m + 3 boxes + 1 mm noise
        rng = np.random.Generator(np.random.Philox(1234))
        z = np.full((480, 640), 1.0)
        for (r0, r1, c0, c1, zz) in ((100, 220, 80, 240, 0.80), (250, 400, 300, 420, 0.70), (60, 160, 450, 600, 0.85)):
            z[r0:r1, c0:c1] = zz
        depth16 = np.clip((z + rng.normal(0, 0.001, z.shape)) * 1000.0, 0, 65535).astype(np.uint16)
        bgr8 = rng.integers(0, 256, (480, 640, 3), dtype=np.uint8)
        kk = (572.4114, 325.2611, 573.57043, 242.04899)
        xyz, _ = ctx.backproject(depth16, bgr8, *kk, 0.001)
        ts = []
        for _ in range(10):
            t0 = time.perf_counter(); ctx.backproject(depth16, bgr8, *kk, 0.001); ts.append(time.perf_counter() - t0)
        tb = float(np.median(ts))
        out["backproject"] = {"frame": "640x480 synthetic (Philox 1234), host buffers in and out", "ms": 1e3 * tb,
                              "pixels_per_s": 307200 / tb, "algorithmic_GBps": 21 * 307200 / tb / 1e9,
                              "note": "21 B per pixel (SURVEY 8d); the call is PCIe/launch bound: 1.5 MB in, 4.9 MB out"}
        if with_cpu:
            import oracle
            oxyz, _ = oracle.backproject(depth16, bgr8, *kk, 0.001)
            out["backproject"]["bit_exact_vs_oracle"] = bool(np.array_equal(xyz.view(np.uint32), np.asarray(oxyz, np.float32).reshape(xyz.shape).view(np.uint32)))
    except Exception as e:
        out["backproject_error"] = str(e)[:100]
    try:  # the other class-mode example of the reference (configs[1] of its README: LINEMOD obj_06)
        out["linemod"] = pose_latency_fixture(ctx, "linemod", "LINEMOD obj_06 example scene")
        out["ycb_scoring_only"] = {k: v for k, v in (pose_latency_fixture(ctx, "ycb", "YCB 024_bowl example scene") or {}).items()
                                   if k.startswith("scoring")}
    except Exception as e:
        out["linemod_error"] = str(e)[:100]
    try:
        out["packed"] = pose_latency_packed(ctx)
    except Exception as e:
        out["packed_error"] = str(e)[:200]
    ctx.close()
    if with_cpu:
        import oracle
        omap = oracle.PPFMap(g["mpos"], g["mnrm"])
        est = oracle.Estimator(g["spos"], g["snrm"], g["scls"], g["mpos"], g["mnrm"], ppfmap=omap)
        nb = 8
        t0 = time.perf_counter()
        Ts = []
        for b in range(nb):
            ok, ids, inv, _ = est.sample_class_base(2, b)
            if not ok:
                continue
            q, _, _ = est.find_congruent(ids, inv[0], inv[1])
            sel = range(len(q)) if len(q) < 200 else [(k * len(q)) // 200 for k in range(200)]
            Ts += [est.fit(ids, q[k])[1] for k in sel]
        if Ts:
            est.score(np.array(Ts, np.float32), threads=1)
        dt = time.perf_counter() - t0
        out["cpu_ms_per_pose"] = 1e3 * dt * 100 / nb
        out["cpu_sample"] = f"oracle, 1 thread, {nb} of 100 bases timed and scaled (PPF map build excluded)"
    return out


def bind_to_gpu_numa_node(local):
    """Multi-rank runs: pin this process to the CPUs next to its GPU (sysfs local_cpulist of the
    PCI device) so that the pinned host buffers the kernels read in place are allocated on that
    NUMA node.  Best effort: returns the CPU list used, or None."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local).pci_bus_id
        dom = torch.cuda.get_device_properties(local).pci_domain_id
        devid = torch.cuda.get_device_properties(local).pci_device_id
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/local_cpulist" % (dom, bus, devid)
        txt = open(path).read().strip()
        cpus = set()
        for part in txt.split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        allowed = os.sched_getaffinity(0)
        cpus &= allowed
        if cpus and cpus != allowed:
            os.sched_setaffinity(0, cpus)
            return txt
    except Exception:
        pass
    return None


WORKLOAD_S1 = "S1: 1,048,576-point synthetic scene, |M|=512, 1e6 hypotheses (1% near-truth), hypothesis-sharded over the GPUs"
WORKLOAD_S2 = "S2: 8 models (|M| 384..1024) x 1e7 hypotheses each, 1,048,576-point scene with per-object class maps, hypothesis-sharded"
S2_MODEL_POINTS = (384, 448, 512, 576, 640, 768, 896, 1024)
S2_H_PER_OBJECT = 10_000_000


def s1_config(world, H=H_TOTAL):
    """The `config` object of the S1 line -- identical in the b200 and the reference arm."""
    return {"workload": WORKLOAD_S1, "scene_points": N_SCENE, "model_points": N_MODEL, "hypotheses": H,
            "hypotheses_per_gpu": -(-H // world),
            "parallelism": f"hypothesis-sharded x{world}, replicated scene index, one all-gather of top-{TOPK} 64-byte records",
            "l2": "inputs larger than L2 (64 MB of transforms per 1e6 hypotheses + ~1.7 GB scene index)"}


def s2_config(world):
    return {"workload": WORKLOAD_S2, "scene_points": N_SCENE, "model_points": list(S2_MODEL_POINTS),
            "hypotheses": 8 * S2_H_PER_OBJECT, "hypotheses_per_gpu": 8 * -(-S2_H_PER_OBJECT // world),
            "parallelism": f"every object hypothesis-sharded x{world}, one all-gather of top-{TOPK} records per object",
            "l2": "inputs larger than L2"}


def run_reference(args):
    """--impl reference: the reference algorithm's CPU implementation (oracle port; the reference
    itself cannot be compiled here: no Eigen/PCL/OpenCV/Boost) on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    from model_matching_b200 import synth
    cores = os.cpu_count() or 1
    if args.workload == "s2":
        sc = synth.make_scene(n_points=N_SCENE, seed=1234)
        ests, Ts = [], []
        for k, m in enumerate(S2_MODEL_POINTS[:2]):   # bounded: two of the eight objects
            mpos, mnrm = synth.make_model(m)
            cls = synth.class_map(len(sc["pos"]), 1000 + k)
            T, _ = synth.make_hypotheses(20000, sc["pos"], mpos, sc["gt_R"], sc["gt_t"], seed=1000 + k)
            ests.append(oracle.Estimator(sc["pos"], sc["nrm"], cls, mpos, mnrm)); Ts.append(T)
        n = min(1000 * cores, 10000)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            last = [e.score(T[:n], threads=cores) for e, T in zip(ests, Ts)]
        dt = time.perf_counter() - t0
        dump_outputs(args.dump_outputs, {f"obj{k}_{name}": a for k, (lcp, inl) in enumerate(last)
                                         for name, a in (("lcp", lcp), ("inliers", inl))})
        v = n * len(ests) * args.steps / dt
        cfg, sample = s2_config(args.gpus), f"{n} hypotheses of each of 2 of the 8 objects per step, {cores} threads"
    else:
        sc, mpos, mnrm, T = workload(0, 200_000)
        est = oracle.Estimator(sc["pos"], sc["nrm"], sc["cls"], mpos, mnrm)
        n = min(2500 * cores, len(T) // 2)  # per step; sized so that steps+warmup end within a few minutes
        for w in range(args.warmup):
            est.score(T[:n // 4], threads=cores)
        t0 = time.perf_counter()
        for k in range(args.steps):
            off = (k * n) % (len(T) - n)
            lcp, inl = est.score(T[off:off + n], threads=cores)
        dt = time.perf_counter() - t0
        dump_outputs(args.dump_outputs, {"lcp": lcp, "inliers": inl})
        v = n * args.steps / dt
        cfg, sample = s1_config(args.gpus), f"{n} hypotheses per step ({args.steps} steps) of the S1 list, {cores} threads"
    out = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
           "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
           "data": "synthetic", "config": cfg,
           "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
           "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out), flush=True)


def source_stamp():
    """sha256 over the sources that define the scoring kernel and the index it reads: an ncu capture
    (profiles/score_kernel_traffic.json) is only quoted when it was taken on these sources."""
    import hashlib
    h = hashlib.sha256()
    for f in ("score.cu", "scene_index.cu", "stocs_ctx.h", "stocs_math.h"):
        h.update(open(os.path.join(ROOT, "model_matching_b200", "csrc", f), "rb").read())
    return h.hexdigest()[:16]


def fitted_hypotheses(ctx, H, seed=20260, max_sets=2000, batch=256, budget_s=90.0):
    """H hypotheses as StoCS produces them (src/stocs.cpp:871-941): bases sampled on the uploaded
    scene, congruent sets on the model, one 3-point fit per (base, quad) -- every transform lands
    the model on scene surface.  Uses the repo's own GPU stages; not timed."""
    out, n, base_no, nb_valid, t0 = [], 0, 0, 0, time.time()
    while n < H and time.time() - t0 < budget_s:
        ids, inv, valid = ctx.sample_bases(seed, base_no, batch)
        base_no += batch
        ids, inv = ids[valid], inv[valid]
        if len(ids) == 0:
            continue
        quads, offs = ctx.find_congruent(ids, inv, cap=1 << 22)
        cnt = np.diff(offs)
        take = np.minimum(cnt, max_sets)
        tot = int(take.sum())
        if tot == 0:
            continue
        b = np.repeat(np.arange(len(ids)), take)
        k = np.arange(tot) - np.repeat(np.cumsum(take) - take, take)
        src = np.where(cnt[b] < max_sets, k, (k * cnt[b]) // max_sets)   # the CLI's even spread
        Tc, _, ok = ctx.fit_transforms(ids[b], quads[offs[b] + src])
        out.append(Tc[ok]); n += int(ok.sum()); nb_valid += len(ids)
    if not out:
        return None, {}
    T = np.concatenate(out)
    info = {"unique": int(min(len(T), H)), "bases_sampled": base_no, "bases_valid": nb_valid, "max_sets": max_sets,
            "generation_s": round(time.time() - t0, 1)}
    if len(T) < H:   # generation budget exhausted: repeat what there is (stated in the line)
        T = np.concatenate([T] * (-(-H // len(T))))
    return np.ascontiguousarray(T[:H], np.float32), info


def counter_bytes(c):
    """Data-dependent byte figures from the kernel's exact work counters.
    survey: SURVEY 8(d)'s formula 32 B per query + 16 B per candidate examined + 16 B per hit.
    kernel_min: what THIS kernel must fetch from beyond shared memory: transform in / results out,
    4 B of brick bitmap per coarse survivor, 16 B per brick record, 8 B of offsets per queued query,
    16 B per candidate examined, 16 B of scene attributes + 16 B of model normal per hit."""
    survey = 32 * c["queries"] + 16 * c["candidates"] + 16 * c["hits"]
    kmin = (56 * c["hypotheses"] + 4 * c["coarse_survivors"] + 16 * c["brick_records"] + 8 * c["queued"]
            + 16 * c["candidates"] + 32 * c["hits"])
    return survey, kmin


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="s1", choices=["s1", "s2"])
    ap.add_argument("--hyp", type=int, default=H_TOTAL, help="hypotheses in the list (default: the named config)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip S1-fit, weak scaling and pose latency")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist
    import model_matching_b200 as mm
    from model_matching_b200 import Context, RECORD, synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: libstocs_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(local) if world > 1 else None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL writes its version / debug lines to stdout by default; stdout carries the JSON line.
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev)   # plumbing: barrier, max-over-ranks, id broadcast

    def new_comm(ctx):
        """library-level communicator: rank 0 makes the NCCL id, torch.distributed only carries it"""
        if world == 1:
            return
        box = [mm.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        ctx.comm_init(box[0], rank, world)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(*vals):
        t = torch.tensor(list(vals), dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t]

    stream = torch.cuda.Stream(dev)   # a dedicated (non-default) stream: NULL means "the context's own" to the ABI
    torch.cuda.set_stream(stream)
    sptr = ctypes.c_void_p(stream.cuda_stream)
    warm = max(args.warmup, 3)

    def timed_steps(step, steps, ctxs):
        """warm-up, then `steps` steps between barriers; -> (ms total max over ranks, mean kernel ms max over ranks)"""
        for _ in range(warm):
            step()
        barrier()
        for c in ctxs:
            c.kernel_ms_stats(reset=True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_begin = time.time()
        e0.record(stream)
        for _ in range(steps):
            step()
        e1.record(stream)
        barrier()
        t_end = time.time()
        kms = float(np.sum([c.kernel_ms_stats()[1] for c in ctxs]))   # per step: one launch per context
        ms_total, kms = max_over_ranks(e0.elapsed_time(e1), kms)
        return ms_total, kms, t_begin, t_end

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
        sampler.wait_first_sample()

    if args.workload == "s2":
        run_s2(args, locals())
        return

    # ---------------------------------------------------------------- S1, strong scaling (the named config)
    H = args.hyp
    sc, mpos, mnrm, T = workload(0, H)            # every rank builds the same list and takes its block
    lo, hi = mm.shard_range(H, rank, world)
    Hl = hi - lo
    ctx = Context(local)
    ctx.upload_model(mpos, mnrm)
    ctx.upload_scene(sc["pos"], sc["nrm"], sc["cls"])
    new_comm(ctx)
    dT = torch.from_numpy(T[lo:hi]).to(dev)
    drec = torch.zeros(TOPK * 64, dtype=torch.uint8, device=dev)

    def step():
        ctx.score_sharded_device(dT.data_ptr(), Hl, lo, TOPK, drec.data_ptr(), sptr)

    ms_total, kernel_ms, t_begin, t_end = timed_steps(step, args.steps, [ctx])
    clocks = sampler.stop(t_begin, t_end) if sampler else None
    value = H * args.steps / (ms_total * 1e-3)
    rec = drec.cpu().numpy().view(RECORD).copy()
    if rank == 0:
        dump_outputs(args.dump_outputs, record_arrays(rec))

    # ---- merged result == single-GPU result of the whole list (asserted on every run)
    dTf = torch.from_numpy(T).to(dev) if world > 1 else dT
    dlcp = torch.empty(H, dtype=torch.float32, device=dev)
    dinl = torch.empty(H, dtype=torch.int32, device=dev)
    dti = torch.empty(TOPK, dtype=torch.int64, device=dev)
    dtv = torch.empty(TOPK, dtype=torch.float32, device=dev)
    ctx.score_lcp_device(dTf.data_ptr(), H, dlcp.data_ptr(), dinl.data_ptr(), sptr)
    ctx.reduce_best_device(dlcp.data_ptr(), H, TOPK, 0, dti.data_ptr(), dtv.data_ptr(), sptr)
    torch.cuda.synchronize(dev)
    ti, tv, inl_full = dti.cpu().numpy(), dtv.cpu().numpy(), dinl.cpu().numpy()
    live = ti >= 0
    T34 = T.reshape(-1, 4, 4).transpose(0, 2, 1)[:, :3, :].reshape(-1, 12)
    merge_ok = bool(np.array_equal(rec["index"], ti) and np.array_equal(rec["lcp"].view(np.uint32), tv.view(np.uint32))
                    and np.array_equal(rec["inliers"][live], inl_full[ti[live]])
                    and np.array_equal(rec["T"][live].view(np.uint32), T34[ti[live]].view(np.uint32)))
    if world > 1:   # every rank must hold the same merged records
        allrec = [None] * world
        dist.all_gather_object(allrec, rec.tobytes())
        merge_ok = merge_ok and all(b == allrec[0] for b in allrec)
    if not merge_ok:
        raise SystemExit(f"rank {rank}: merged top-{TOPK} differs from the single-GPU result of the whole list")
    del dTf

    # ---- e2e: the host-buffer call (pinned host memory in, records + per-hypothesis results out)
    hT = torch.from_numpy(T[lo:hi]).pin_memory()
    hlcp = torch.empty(Hl, dtype=torch.float32).pin_memory()
    hinl = torch.empty(Hl, dtype=torch.int32).pin_memory()
    hrec = np.zeros(TOPK, RECORD)
    e2e_steps = max(1, min(args.steps, 20))

    def e2e_step(hT=hT, n=Hl, off=lo):
        ctx.score_sharded_ptr(hT.data_ptr(), n, off, TOPK, hrec, hlcp.data_ptr(), hinl.data_ptr())

    def e2e_measure(stepfn, Htot):
        stepfn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            stepfn()
        torch.cuda.synchronize(dev)
        dt, = max_over_ranks(time.perf_counter() - t0)
        return Htot * e2e_steps / dt

    def h2d_probe():
        """every rank copies its pinned block to its GPU at the same time: the platform's host->device ceiling"""
        dst = torch.empty_like(dT)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        dst.copy_(hT, non_blocking=True)
        barrier()
        a.record(stream)
        for _ in range(10):
            dst.copy_(hT, non_blocking=True)
        b.record(stream)
        torch.cuda.synchronize(dev)
        ms, = max_over_ranks(a.elapsed_time(b) / 10)
        per_rank = hT.numel() * 4 / (ms * 1e-3) / 1e9
        return {"bytes_per_rank": hT.numel() * 4, "per_rank_GBps": per_rank, "aggregate_GBps": per_rank * world,
                "note": "all ranks copy at once (cudaMemcpyAsync from pinned memory, max over ranks): an upper bound on any "
                        "end-to-end rate that ingests 64 B per hypothesis = aggregate_GBps / 64 B"}

    h2d = h2d_probe()
    e2e_value = e2e_measure(e2e_step, H)
    e2e_rec = hrec.copy()
    os.environ["STOCS_NO_ZERO_COPY"] = "1"
    e2e_staged = e2e_measure(e2e_step, H)
    del os.environ["STOCS_NO_ZERO_COPY"]
    if not (np.array_equal(e2e_rec["index"], rec["index"]) and np.array_equal(hrec["index"], rec["index"])):
        raise SystemExit("e2e records differ from the device-resident run")

    # ---- weak scaling (N > 1): 1e6 hypotheses PER GPU
    extra = {}
    if world > 1 and not args.no_extras:
        Tw, _ = synth.make_hypotheses(H, sc["pos"], mpos, sc["gt_R"], sc["gt_t"], seed=4321 + rank)
        dTw = torch.from_numpy(Tw).to(dev)
        wsteps = max(1, min(args.steps, 50))

        def wstep():
            ctx.score_sharded_device(dTw.data_ptr(), H, rank * H, TOPK, drec.data_ptr(), sptr)

        wms, wk, _, _ = timed_steps(wstep, wsteps, [ctx])
        hTw = torch.from_numpy(Tw).pin_memory()
        hlcp = torch.empty(H, dtype=torch.float32).pin_memory()
        hinl = torch.empty(H, dtype=torch.int32).pin_memory()
        we2e = e2e_measure(lambda: e2e_step(hTw, H, rank * H), world * H)
        extra["weak"] = {"workload": "1e6 hypotheses per GPU (round-1 configuration)", "value": world * H * wsteps / (wms * 1e-3),
                         "ms_per_step": wms / wsteps, "steps": wsteps, "kernel_ms": wk, "e2e_value": we2e, "scaling": "weak"}
        del dTw, hTw

    if rank == 0:
        M = N_MODEL
        peaks = {}
        pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(pk):
            peaks = json.load(open(pk))
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        stamp = source_stamp()

        def roofline_of(kms, n_hyp, counters, traffic_key):
            alg = n_hyp * algorithmic_bytes_per_hypothesis(M)
            r = {"bound": "hbm", "achieved": alg / (kms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                 "kernel": "score_lcp_kernel", "kernel_ms": kms, "hypotheses_per_launch": n_hyp,
                 "algorithmic_bytes_per_launch": alg, "peak_source": peak_src, "traffic": None}
            r["frac"] = r["achieved"] / peak
            if counters:
                survey, kmin = counter_bytes(counters)
                r["counters"] = counters
                r["data_bytes_per_launch"] = survey
                r["frac_data"] = survey / (kms * 1e-3) / 1e9 / peak
                r["kernel_min_bytes_per_launch"] = kmin
                r["frac_kernel_min"] = kmin / (kms * 1e-3) / 1e9 / peak
            tp = os.path.join(ROOT, "profiles", "score_kernel_traffic.json")
            if os.path.exists(tp):
                t = json.load(open(tp)).get(traffic_key)
                if t and t.get("hypotheses_per_launch") == n_hyp:
                    r["traffic"] = t["dram_bytes_per_launch"]
                    r["traffic_capture"] = {k: t.get(k) for k in ("source_stamp", "workload", "captured", "file")}
                    r["traffic_capture"]["current_source_stamp"] = stamp
                    r["traffic_capture"]["stale"] = t.get("source_stamp") != stamp
                    r["dram_achieved"] = r["traffic"] / (kms * 1e-3) / 1e9
                    r["dram_frac"] = r["dram_achieved"] / peak
            return r

        cnt = ctx.score_counters(dT.data_ptr(), Hl)
        roof = roofline_of(kernel_ms, Hl, cnt, "s1")
        roof["note"] = ("frac: contract accounting of SURVEY 8(d), 64 B for EVERY (hypothesis, model point) query -- not a "
                        "physical fraction (the kernel answers most queries from an on-chip occupancy map); frac_data: "
                        "SURVEY 8(d)'s data-dependent counter 32 B/query + 16 B/candidate examined + 16 B/hit from the kernel's "
                        "exact work counters; frac_kernel_min: bytes this kernel must fetch from beyond shared memory; "
                        "dram_frac: DRAM bytes of the committed ncu capture (stamped) over the live kernel time")
        out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
               "warmup": warm, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
               "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
               "config": s1_config(world, H),
               "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": Hl * 64, "d2h_bytes_per_step": Hl * 8 + TOPK * 64,
                       "bytes_note": "per rank", "steps": e2e_steps, "best_index": int(rec["index"][0]), "best_lcp": float(rec["lcp"][0]),
                       "input_path": "pinned host transforms read in place by the kernel over PCIe (zero-copy); per-hypothesis "
                                     "lcp + inlier counts and the merged top-K records copied back",
                       "staged_copy_value": e2e_staged, "numa_cpus": numa, "h2d_probe": h2d},
               # per step: [probe_order_kernel for 32 768..300 000 hypotheses per launch] + score_lcp_kernel +
               # topk_kernel [+ merge_records_kernel after the all-gather]
               "gpu_launches": args.steps * (2 + (1 if world > 1 else 0) + (1 if 32768 <= Hl <= 300000 and not os.environ.get("STOCS_NO_LPT") else 0)),
               "collectives_per_step": 1 if world > 1 else 0,
               "merge_check": {"merged_topk_equals_single_gpu_topk_of_whole_list": merge_ok, "ranks_agree": True, "K": TOPK},
               "roofline": roof, "clocks": clocks, "ties_resolved_by_kdtree": int(ctx.counters()[1]), "extra": extra}
        if world == 1 and not args.no_extras:
            try:
                extra["s1_fit"] = s1_fit(ctx, H, stream, sptr, dev, timed_steps, e2e_measure, roofline_of, min(args.steps, 50),
                                         sc, mpos, mnrm, not args.no_cpu_baseline)
            except Exception as e:  # the headline does not depend on it
                extra["s1_fit"] = {"error": str(e)[:300]}
            out["pose_latency"] = pose_latency(lambda: Context(local), not args.no_cpu_baseline)
        if world == 1 and not args.no_cpu_baseline:
            est, cb, (olcp, oinl, n) = cpu_baseline(sc, mpos, mnrm, T)
            out["cpu_baseline"] = cb
            # parity gate run with the measurement (SURVEY 8d): the sample must match bit for bit
            glcp, ginl = hlcp.numpy()[:n], hinl.numpy()[:n]
            out["parity"] = {"checked": int(n), "inliers_equal": bool(np.array_equal(ginl, oinl)),
                             "lcp_bits_equal": bool(np.array_equal(glcp.view(np.uint32), olcp.view(np.uint32)))}
            # the same data-dependent counter on the reference's own structure (kd-tree), same prefix
            npre = min(n, 20000)
            oc = est.score_counters(T[:npre], threads=os.cpu_count() or 1)
            gc = ctx.score_counters(dT.data_ptr(), npre)
            out["roofline"]["oracle_counter"] = {"prefix": npre, "kdtree": oc, "grid_hits": gc["hits"], "grid_inliers": gc["inliers"],
                                                 "grid_candidates": gc["candidates"],
                                                 "hits_equal": oc["hits"] == gc["hits"], "inliers_equal": oc["inliers"] == gc["inliers"],
                                                 "kdtree_bytes_per_query": oc["bytes"] / oc["queries"],
                                                 "grid_bytes_per_query": counter_bytes(gc)[0] / gc["queries"]}
        print(json.dumps(out), flush=True)
    barrier()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def s1_fit(ctx, H, stream, sptr, dev, timed_steps, e2e_measure, roofline_of, steps, sc, mpos, mnrm, with_cpu):
    """Second named workload: 1e6 hypotheses produced by the repo's own pipeline on the S1 scene --
    every one a 3-point fit onto scene surface, as src/stocs.cpp:871-941 produces them."""
    import torch
    from model_matching_b200 import RECORD
    T, info = fitted_hypotheses(ctx, H)
    if T is None:
        return {"error": "no fitted hypotheses (no valid base)"}
    dT = torch.from_numpy(T).to(dev)
    drec = torch.zeros(TOPK * 64, dtype=torch.uint8, device=dev)

    def step():
        ctx.score_sharded_device(dT.data_ptr(), H, 0, TOPK, drec.data_ptr(), sptr)

    ms, kms, _, _ = timed_steps(step, steps, [ctx])
    hT = torch.from_numpy(T).pin_memory()
    hlcp = torch.empty(H, dtype=torch.float32).pin_memory()
    hinl = torch.empty(H, dtype=torch.int32).pin_memory()
    hrec = np.zeros(TOPK, RECORD)
    e2e = e2e_measure(lambda: ctx.score_sharded_ptr(hT.data_ptr(), H, 0, TOPK, hrec, hlcp.data_ptr(), hinl.data_ptr()), H)
    cnt = ctx.score_counters(dT.data_ptr(), H)
    out = {"workload": "S1-fit: the S1 scene and model, 1e6 hypotheses fitted by the repo's own sampling -> congruent sets -> "
                       "3-point fit stages (all land the model on scene surface)",
           "generation": info, "value": H * steps / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / steps, "steps": steps,
           "e2e_value": e2e, "roofline": roofline_of(kms, H, cnt, "s1_fit"),
           "mean_inliers": float(hinl.numpy().mean()), "best_lcp": float(hrec["lcp"][0]),
           "target_1e8_met": bool(H * steps / (ms * 1e-3) >= 1e8)}
    if with_cpu:
        import oracle
        est = oracle.Estimator(sc["pos"], sc["nrm"], sc["cls"], mpos, mnrm)
        n = 4000
        olcp, oinl = est.score(T[:n], threads=os.cpu_count() or 1)
        out["parity"] = {"checked": n, "inliers_equal": bool(np.array_equal(hinl.numpy()[:n], oinl)),
                         "lcp_bits_equal": bool(np.array_equal(hlcp.numpy()[:n].view(np.uint32), olcp.view(np.uint32)))}
    return out


def run_s2(args, env):
    """BASELINE.json configs[4]: 8 models x 1e7 hypotheses each, every object hypothesis-sharded over
    the GPUs (SURVEY 8e: balanced, rather than object-per-GPU).  One context per object and rank (the
    class map, hence the scene attributes, differ per object); one all-gather per object and step."""
    import torch
    import torch.distributed as dist
    import model_matching_b200 as mm
    from model_matching_b200 import Context, RECORD, synth
    rank, world, local, dev, stream, sptr = (env[k] for k in ("rank", "world", "local", "dev", "stream", "sptr"))
    timed_steps, new_comm, sampler, warm = env["timed_steps"], env["new_comm"], env["sampler"], env["warm"]
    Hobj = args.hyp if args.hyp != H_TOTAL else S2_H_PER_OBJECT
    sc = synth.make_scene(n_points=N_SCENE, seed=1234)
    lo, hi = mm.shard_range(Hobj, rank, world)
    Hl = hi - lo
    ctxs, dTs, drecs = [], [], []
    for k, m in enumerate(S2_MODEL_POINTS):
        mpos, mnrm = synth.make_model(m)
        c = Context(local)
        c.upload_model(mpos, mnrm)
        c.upload_scene(sc["pos"], sc["nrm"], synth.class_map(len(sc["pos"]), 1000 + k))
        new_comm(c)
        # each rank generates only its own block (seeded by object and rank)
        T, _ = synth.make_hypotheses(Hl, sc["pos"], mpos, sc["gt_R"], sc["gt_t"], seed=1000 + k + 100 * rank)
        ctxs.append(c); dTs.append(torch.from_numpy(T).to(dev))
        drecs.append(torch.zeros(TOPK * 64, dtype=torch.uint8, device=dev))
        del T

    def step():
        for c, dT, dr in zip(ctxs, dTs, drecs):
            c.score_sharded_device(dT.data_ptr(), Hl, lo, TOPK, dr.data_ptr(), sptr)

    ms_total, kernel_ms, t_begin, t_end = timed_steps(step, args.steps, ctxs)
    clocks = sampler.stop(t_begin, t_end) if sampler else None
    recs = [dr.cpu().numpy().view(RECORD).copy() for dr in drecs]
    if rank == 0:
        dump_outputs(args.dump_outputs, {k: a for i, r in enumerate(recs) for k, a in record_arrays(r, f"obj{i}_").items()})
    if world > 1:
        allrec = [None] * world
        dist.all_gather_object(allrec, b"".join(r.tobytes() for r in recs))
        if not all(b == allrec[0] for b in allrec):
            raise SystemExit("S2: ranks disagree on the merged records")
    if rank == 0:
        Htot = len(S2_MODEL_POINTS) * Hobj
        alg = sum(Hl * algorithmic_bytes_per_hypothesis(m) for m in S2_MODEL_POINTS)
        peaks = {}
        pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(pk):
            peaks = json.load(open(pk))
        peak = float(peaks.get("hbm_gbs", 6650.0))
        out = {"metric": METRIC, "value": Htot * args.steps / (ms_total * 1e-3), "unit": UNIT, "n_gpus": world,
               "steps": args.steps, "warmup": warm, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
               "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": s2_config(world),
               "gpu_launches": args.steps * len(ctxs) * (3 + (1 if world > 1 else 0)),
               "collectives_per_step": len(ctxs) if world > 1 else 0,
               "roofline": {"bound": "hbm", "achieved": alg / (kernel_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                            "frac": alg / (kernel_ms * 1e-3) / 1e9 / peak, "traffic": None, "kernel": "score_lcp_kernel",
                            "kernel_ms": kernel_ms, "note": "sum over the 8 per-object launches of one step; contract accounting (see the S1 line)"},
               "best_per_object": [{"model_points": m, "index": int(r["index"][0]), "lcp": float(r["lcp"][0]), "inliers": int(r["inliers"][0])}
                                   for m, r in zip(S2_MODEL_POINTS, recs)],
               "clocks": clocks}
        print(json.dumps(out), flush=True)
    env["barrier"]()
    for c in ctxs:
        c.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
