"""ctypes binding of libstocs_b200.so (include/stocs_b200.h).

The library is the product; this module only marshals numpy / torch buffers into it.  There is
no CPU fallback: importing works without a GPU (so that the symbol table can be checked), but
creating a Context without a B200 raises, and a missing .so raises at import of `lib()`.
"""
import ctypes as C
import itertools
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("STOCS_B200_LIB", os.path.join(_HERE, "libstocs_b200.so"))
_LIB = None

# every symbol include/stocs_b200.h declares (checked by tests/test_abi.py)
SYMBOLS = [
    "stocs_b200_abi_version", "stocs_b200_create", "stocs_b200_destroy", "stocs_b200_last_error",
    "stocs_b200_set_params", "stocs_b200_backproject", "stocs_b200_build_scene_cloud", "stocs_b200_build_scene_clouds",
    "stocs_b200_build_scene_clouds_device", "stocs_b200_upload_model",
    "stocs_b200_upload_scene", "stocs_b200_get_centroids", "stocs_b200_get_centred",
    "stocs_b200_ppf_num_pairs", "stocs_b200_ppf_num_expanded_keys", "stocs_b200_ppf_export",
    "stocs_b200_ppf_lookup", "stocs_b200_upload_ppf_table", "stocs_b200_sample_bases",
    "stocs_b200_upload_edge_map", "stocs_b200_sample_instance_base", "stocs_b200_get_class_probability",
    "stocs_b200_set_class_probability",
    "stocs_b200_find_congruent", "stocs_b200_fit_transforms", "stocs_b200_score_lcp",
    "stocs_b200_score_lcp_device", "stocs_b200_reduce_best", "stocs_b200_reduce_best_device", "stocs_b200_select_above",
    "stocs_b200_icp_point_to_plane",
    "stocs_b200_run_pipeline", "stocs_b200_run_pipeline_instance", "stocs_b200_cluster_poses",
    "stocs_b200_run_pipeline_clustered", "stocs_b200_run_pipeline_instance_clustered",
    "stocs_b200_upload_scenes", "stocs_b200_upload_scenes_device", "stocs_b200_run_pipelines", "stocs_b200_get_counters", "stocs_b200_last_kernel_ms",
    "stocs_b200_score_counters", "stocs_b200_kernel_ms_stats", "stocs_b200_host_kdtree_order", "stocs_b200_debug_kdtree",
    "stocs_b200_debug_angle_estimates", "stocs_b200_debug_survivor_counts", "stocs_b200_debug_fine_survivor_counts",
    "stocs_b200_comm_unique_id", "stocs_b200_comm_init", "stocs_b200_comm_destroy", "stocs_b200_shard_range",
    "stocs_b200_score_sharded_device", "stocs_b200_score_sharded",
    "stocs_b200_group_create", "stocs_b200_group_destroy", "stocs_b200_group_size", "stocs_b200_group_ctx",
    "stocs_b200_group_last_error", "stocs_b200_group_set_params", "stocs_b200_group_upload_model",
    "stocs_b200_group_upload_scene", "stocs_b200_group_score_best",
]


class StocsError(RuntimeError):
    pass


class PipelineResult(C.Structure):
    _fields_ = [("n_valid_bases", C.c_int32), ("n_congruent_sets", C.c_int64),
                ("n_transforms", C.c_int64), ("best_index", C.c_int64), ("best_lcp", C.c_float),
                ("best_base", C.c_int32), ("best_T_centred", C.c_float * 16),
                ("best_T_world", C.c_float * 16)]


class ClusterParams(C.Structure):
    _fields_ = [("acceptable_fraction", C.c_float), ("maximum_pose_count", C.c_int32), ("min_distance", C.c_float),
                ("min_angle", C.c_float), ("sym_info", C.c_float * 3)]


# stocs_b200_pose (include/stocs_b200.h): one pose kept by the clustered pipeline
POSE = np.dtype([("index", np.int64), ("lcp", np.float32), ("base", np.int32), ("T_centred", np.float32, (16,)),
                 ("T_world", np.float32, (16,))])
assert POSE.itemsize == 144


def lib():
    """Load libstocs_b200.so; raise loudly when it has not been built."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise StocsError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, f32, u64, u32 = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_uint64, C.c_uint32
    L.stocs_b200_abi_version.restype = i32
    L.stocs_b200_create.argtypes = [C.POINTER(vp), i32]
    L.stocs_b200_destroy.argtypes = [vp]
    L.stocs_b200_destroy.restype = None
    L.stocs_b200_last_error.argtypes = [vp]
    L.stocs_b200_last_error.restype = C.c_char_p
    L.stocs_b200_set_params.argtypes = [vp, f32, i32, i32]
    L.stocs_b200_backproject.argtypes = [vp, vp, vp, i32, i32, f32, f32, f32, f32, f32, vp, vp]
    L.stocs_b200_build_scene_cloud.argtypes = [vp, vp, vp, vp, vp, i32, i32, f32, f32, f32, f32, f32, f32, f32,
                                               vp, vp, vp, vp, vp, vp, i64, C.POINTER(i64)]
    L.stocs_b200_build_scene_clouds.argtypes = [vp, vp, vp, vp, vp, i32, vp, i32, i32, f32, f32, f32, f32, f32, f32,
                                                vp, vp, vp, vp, vp, vp, i64, vp]
    L.stocs_b200_build_scene_clouds_device.argtypes = [vp, vp, vp, vp, i32, vp, i32, vp, i32, i32, f32, f32, f32, f32, f32,
                                                       f32, vp, vp, vp, vp, vp, vp, i64, vp, vp]
    L.stocs_b200_upload_model.argtypes = [vp, vp, vp, i32]
    L.stocs_b200_upload_scene.argtypes = [vp, vp, vp, vp, vp, i32]
    L.stocs_b200_get_centroids.argtypes = [vp, vp, vp]
    L.stocs_b200_get_centred.argtypes = [vp, vp, vp]
    L.stocs_b200_ppf_num_pairs.argtypes = [vp, C.POINTER(i64), C.POINTER(i64)]
    L.stocs_b200_ppf_lookup.argtypes = [vp, vp, vp, i64, C.POINTER(i64)]
    L.stocs_b200_upload_ppf_table.argtypes = [vp, vp, vp, i64, i32, i32, i32]
    L.stocs_b200_ppf_num_expanded_keys.argtypes = [vp, C.POINTER(i64)]
    L.stocs_b200_ppf_export.argtypes = [vp, vp, vp, i64, C.POINTER(i64)]
    L.stocs_b200_sample_bases.argtypes = [vp, u64, u32, i32, vp, vp, vp]
    L.stocs_b200_upload_edge_map.argtypes = [vp, vp, i32, i32]
    L.stocs_b200_sample_instance_base.argtypes = [vp, u64, i32, f32, vp, vp, vp, vp, vp]
    L.stocs_b200_get_class_probability.argtypes = [vp, vp]
    L.stocs_b200_set_class_probability.argtypes = [vp, vp]
    L.stocs_b200_find_congruent.argtypes = [vp, i32, vp, vp, vp, i64, vp]
    L.stocs_b200_fit_transforms.argtypes = [vp, i64, vp, vp, vp, vp, vp]
    L.stocs_b200_score_lcp.argtypes = [vp, vp, i64, vp, vp]
    L.stocs_b200_score_lcp_device.argtypes = [vp, vp, i64, vp, vp, vp]
    L.stocs_b200_reduce_best.argtypes = [vp, vp, i64, i32, C.POINTER(i64), C.POINTER(f32), vp, vp]
    L.stocs_b200_reduce_best_device.argtypes = [vp, vp, i64, i32, i64, vp, vp, vp]
    L.stocs_b200_select_above.argtypes = [vp, vp, i64, f32, vp, vp, i64, C.POINTER(i64)]
    L.stocs_b200_icp_point_to_plane.argtypes = [vp, vp, i32, vp, vp, i32, i32, f32, vp, vp, vp, C.POINTER(i32), C.POINTER(i32)]
    L.stocs_b200_run_pipeline.argtypes = [vp, u64, i32, i32, C.POINTER(PipelineResult)]
    L.stocs_b200_run_pipeline_instance.argtypes = [vp, u64, i32, i32, f32, C.POINTER(PipelineResult)]
    L.stocs_b200_cluster_poses.argtypes = [vp, vp, vp, i64, f32, C.POINTER(ClusterParams), vp, i64, C.POINTER(i64)]
    L.stocs_b200_run_pipeline_clustered.argtypes = [vp, u64, i32, i32, C.POINTER(ClusterParams), C.POINTER(PipelineResult),
                                                    vp, i32, C.POINTER(i32)]
    L.stocs_b200_run_pipeline_instance_clustered.argtypes = [vp, u64, i32, i32, f32, C.POINTER(ClusterParams),
                                                             C.POINTER(PipelineResult), vp, i32, C.POINTER(i32)]
    L.stocs_b200_upload_scenes.argtypes = [vp, i32, vp, vp, vp, vp, vp]
    L.stocs_b200_upload_scenes_device.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp]
    L.stocs_b200_run_pipelines.argtypes = [vp, i32, vp, i32, i32, i32, f32, vp, vp, vp, i32, vp]
    L.stocs_b200_get_counters.argtypes = [vp, vp, i32]
    L.stocs_b200_last_kernel_ms.argtypes = [vp, C.POINTER(f32)]
    L.stocs_b200_score_counters.argtypes = [vp, vp, i64, vp, i32]
    L.stocs_b200_kernel_ms_stats.argtypes = [vp, i32, C.POINTER(i32), C.POINTER(f32), C.POINTER(f32)]
    L.stocs_b200_host_kdtree_order.argtypes = [vp, i32, vp, C.POINTER(i32)]
    L.stocs_b200_debug_kdtree.argtypes = [vp, vp, i32, i32, vp, C.POINTER(i32), vp]
    L.stocs_b200_debug_angle_estimates.argtypes = [vp, vp, vp, i64, vp, vp, vp, vp, vp, vp]
    L.stocs_b200_debug_survivor_counts.argtypes = [vp, vp, i64, vp]
    L.stocs_b200_debug_fine_survivor_counts.argtypes = [vp, vp, i64, vp, vp]
    L.stocs_b200_comm_unique_id.argtypes = [vp]
    L.stocs_b200_comm_init.argtypes = [vp, vp, i32, i32]
    L.stocs_b200_comm_destroy.argtypes = [vp]
    L.stocs_b200_shard_range.argtypes = [i64, i32, i32, C.POINTER(i64), C.POINTER(i64)]
    L.stocs_b200_shard_range.restype = None
    L.stocs_b200_score_sharded_device.argtypes = [vp, vp, i64, i64, i32, vp, vp]
    L.stocs_b200_score_sharded.argtypes = [vp, vp, i64, i64, i32, vp, vp, vp]
    L.stocs_b200_group_create.argtypes = [C.POINTER(vp), C.POINTER(i32), i32]
    L.stocs_b200_group_destroy.argtypes = [vp]
    L.stocs_b200_group_destroy.restype = None
    L.stocs_b200_group_size.argtypes = [vp]
    L.stocs_b200_group_ctx.argtypes = [vp, i32]
    L.stocs_b200_group_ctx.restype = vp
    L.stocs_b200_group_last_error.argtypes = [vp]
    L.stocs_b200_group_last_error.restype = C.c_char_p
    L.stocs_b200_group_set_params.argtypes = [vp, f32, i32, i32]
    L.stocs_b200_group_upload_model.argtypes = [vp, vp, vp, i32]
    L.stocs_b200_group_upload_scene.argtypes = [vp, vp, vp, vp, vp, i32]
    L.stocs_b200_group_score_best.argtypes = [vp, vp, i64, i32, vp, vp, vp]
    _LIB = L
    return L


def _ptr(a):
    return None if a is None else a.ctypes.data


def _f32(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float32)
    return a if shape is None else a.reshape(shape)


# stocs_b200_record (include/stocs_b200.h): the 64-byte unit of the multi-GPU all-gather
RECORD = np.dtype([("lcp", np.float32), ("inliers", np.int32), ("index", np.int64), ("T", np.float32, (12,))])
assert RECORD.itemsize == 64


def _cluster_params(acceptable_fraction, maximum_pose_count, min_distance, min_angle, sym_info=(0, 0, 0)):
    return ClusterParams(acceptable_fraction, int(maximum_pose_count), min_distance, min_angle,
                         (C.c_float * 3)(*[float(v) for v in sym_info]))


def _handles(contexts):
    assert len(contexts) >= 1, "at least one context"
    return (C.c_void_p * len(contexts))(*[c.h for c in contexts])


def _has_scene(ctx):
    return lib().stocs_b200_get_centroids(ctx.h, _ptr(np.zeros(3, np.float32)), None) == 0


def _csr_device(clouds, key, cols, dtype, offs):
    """The CSR array of one key of CUDA-tensor clouds -> (device pointer, tensor to keep alive): the slices' own
    buffer when they are consecutive views of it (the outputs of Context.build_scene_clouds_device), else their
    concatenation."""
    import torch
    parts = [c[key] for c in clouds]
    used = [(p, int(o)) for p, o in zip(parts, offs[:-1]) if p.numel()]
    row = cols * torch.empty(0, dtype=dtype).element_size()
    if used and all(p.dtype == dtype and p.is_contiguous() and p.device == used[0][0].device for p, _ in used):
        base = used[0][0].data_ptr() - used[0][1] * row
        if all(p.data_ptr() == base + o * row for p, o in used):
            return base, None
    dev = parts[0].device
    cat = torch.cat([p.reshape(-1, cols).to(dev, dtype) for p in parts]) if used else torch.zeros((1, cols), dtype=dtype, device=dev)
    return cat.data_ptr(), cat


def _upload_scenes_device(contexts, clouds, offs, has_pix):
    import torch
    arrays = [_csr_device(clouds, "pos", 3, torch.float32, offs), _csr_device(clouds, "nrm", 3, torch.float32, offs),
              _csr_device(clouds, "cls", 1, torch.float32, offs)]
    arrays.append(_csr_device(clouds, "pix", 2, torch.int32, offs) if has_pix else (None, None))
    stream = torch.cuda.current_stream(clouds[0]["pos"].device).cuda_stream
    return lib().stocs_b200_upload_scenes_device(_handles(contexts), len(contexts), *[a[0] for a in arrays], _ptr(offs),
                                                 stream)


def upload_scenes(contexts, clouds):
    """Object k's cloud (a dict of Context.build_scene_clouds: pos, nrm, cls and optionally pix) to contexts[k],
    every object in one call (stocs_b200_upload_scenes); an empty cloud leaves its context with an empty scene.
    Clouds of torch CUDA tensors (Context.build_scene_clouds_device) go to stocs_b200_upload_scenes_device, ordered
    after torch's current stream; views of one output buffer are passed without a copy."""
    assert len(contexts) == len(clouds), "one cloud per context"
    n = [len(c["pos"]) for c in clouds]
    if len({id(c) for c in contexts}) < len(contexts) or any(not c.h for c in contexts) or max(n, default=0) > (1 << 27):
        raise StocsError("upload_scenes: a context given twice or closed, or a slice over 2^27 points")
    offs = np.fromiter(itertools.accumulate(n, initial=0), np.int64, len(n) + 1)
    has_pix = all(c.get("pix") is not None for c in clouds)
    if getattr(clouds[0]["pos"], "is_cuda", False):
        rc = _upload_scenes_device(contexts, clouds, offs, has_pix)
    else:
        if len(clouds) == 1:   # one object's arrays are passed as they are
            c = clouds[0]
            pos, nrm, cls = _f32(c["pos"], (-1, 3)), _f32(c["nrm"], (-1, 3)), _f32(c["cls"], (-1,))
            pix = np.ascontiguousarray(c["pix"], np.int32).reshape(-1, 2) if has_pix else None
        else:                  # the CSR concatenation
            pos = np.concatenate([_f32(c["pos"], (-1, 3)) for c in clouds])
            nrm = np.concatenate([_f32(c["nrm"], (-1, 3)) for c in clouds])
            cls = np.concatenate([_f32(c["cls"], (-1,)) for c in clouds])
            pix = np.concatenate([np.ascontiguousarray(c["pix"], np.int32).reshape(-1, 2) for c in clouds]) if has_pix else None
        assert pos.shape == nrm.shape and cls.shape[0] == pos.shape[0]
        rc = lib().stocs_b200_upload_scenes(_handles(contexts), len(contexts), _ptr(pos), _ptr(nrm), _ptr(cls), _ptr(pix),
                                            _ptr(offs))
    err = None
    try:
        contexts[0]._check(rc)
    except StocsError as e:
        err = e
    for c, k in zip(contexts, n):
        # the arguments passed the checks above, so a failure came after validation: the objects that
        # uploaded hold their slice, the failing one (and any empty slice) holds none
        c.S = k if err is None or _has_scene(c) else 0
    if err is not None:
        raise err


def run_pipelines(contexts, seeds, n_bases=100, max_sets=200, instance=False, dispersion=0.9, cluster=None):
    """run_pipeline[_instance][_clustered] on every context in one call (stocs_b200_run_pipelines), with seeds[k]
    on contexts[k].  cluster: None, or one dict of cluster parameters per object (acceptable_fraction,
    maximum_pose_count, min_distance, min_angle, sym_info).  -> [PipelineResult], or [(PipelineResult, POSE array)]."""
    n = len(contexts)
    seeds = np.ascontiguousarray(np.asarray(seeds, np.uint64).reshape(n))
    results = (PipelineResult * n)()
    if cluster is None:
        contexts[0]._check(lib().stocs_b200_run_pipelines(_handles(contexts), n, _ptr(seeds), n_bases, max_sets, int(instance),
                                                          dispersion, None, results, None, 0, None))
        return list(results)
    assert len(cluster) == n, "one cluster parameter record per object"
    params = (ClusterParams * n)(*[_cluster_params(**p) for p in cluster])
    cap = max(max(p.maximum_pose_count for p in params) + 1, 1)
    poses, n_poses = np.zeros((n, cap), POSE), np.zeros(n, np.int32)
    contexts[0]._check(lib().stocs_b200_run_pipelines(_handles(contexts), n, _ptr(seeds), n_bases, max_sets, int(instance),
                                                      dispersion, params, results, _ptr(poses), cap, _ptr(n_poses)))
    return [(results[k], poses[k, :n_poses[k]].copy()) for k in range(n)]


def host_kdtree_order(pos):
    """Host-only (no GPU): leaf order and node count of the reference kd-tree as upload_scene builds it."""
    pos = _f32(pos, (-1, 3))
    order, nn = np.empty(pos.shape[0], np.int32), C.c_int32(0)
    rc = lib().stocs_b200_host_kdtree_order(_ptr(pos), pos.shape[0], _ptr(order), C.byref(nn))
    if rc:
        raise StocsError("stocs_b200_host_kdtree_order failed: %d" % rc)
    return order, nn.value


def shard_range(H, rank, nranks):
    """[lo, hi) of ceil(H / nranks) hypotheses owned by `rank` (stocs_b200_shard_range)."""
    lo, hi = C.c_int64(0), C.c_int64(0)
    lib().stocs_b200_shard_range(H, rank, nranks, C.byref(lo), C.byref(hi))
    return lo.value, hi.value


def comm_unique_id():
    """128 bytes for Context.comm_init; rank 0 creates them, the caller distributes them."""
    buf = C.create_string_buffer(128)
    rc = lib().stocs_b200_comm_unique_id(buf)
    if rc != 0:
        raise StocsError(f"stocs_b200_comm_unique_id failed ({rc}): NCCL not loadable")
    return bytes(buf.raw)


class Context:
    """One stocs_b200_ctx (one GPU)."""

    def __init__(self, device=0, distance_threshold=0.005, ppf_tr_discretization=5,
                 ppf_rot_discretization=5):
        self._L = lib()
        h = C.c_void_p()
        rc = self._L.stocs_b200_create(C.byref(h), int(device))
        if rc != 0:
            msg = self._L.stocs_b200_last_error(None)
            raise StocsError(f"stocs_b200_create failed ({rc}): {msg.decode() if msg else ''}")
        self.h = h
        self.device = device
        self._check(self._L.stocs_b200_set_params(self.h, distance_threshold, ppf_tr_discretization,
                                                   ppf_rot_discretization))
        self.M = self.S = 0
        self._last_H = 0

    def close(self):
        if getattr(self, "h", None):
            self._L.stocs_b200_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            msg = self._L.stocs_b200_last_error(self.h)
            raise StocsError(f"libstocs_b200 error {rc}: {msg.decode() if msg else ''}")

    # ---- a1
    def backproject(self, depth, bgr, fx, cx, fy, cy, depth_scale):
        depth = np.ascontiguousarray(depth, np.uint16)
        H, W = depth.shape
        bgr = None if bgr is None else np.ascontiguousarray(bgr, np.uint8)
        xyz = np.empty((H * W, 3), np.float32)
        rgb = np.empty(H * W, np.uint32) if bgr is not None else None
        self._check(self._L.stocs_b200_backproject(self.h, _ptr(depth), _ptr(bgr), W, H, fx, cx, fy, cy,
                                                    depth_scale, _ptr(xyz), _ptr(rgb)))
        return xyz, rgb

    # ---- f1
    def build_scene_cloud(self, depth, bgr, prob, edge, K, depth_scale, voxel_size, class_threshold):
        depth = np.ascontiguousarray(depth, np.uint16)
        H, W = depth.shape
        bgr = None if bgr is None else np.ascontiguousarray(bgr, np.uint8)
        prob = np.ascontiguousarray(prob, np.uint16)
        edge = None if edge is None else np.ascontiguousarray(edge, np.uint8)
        cap = H * W
        pos, nrm, rgb = (np.empty((cap, 3), np.float32) for _ in range(3))
        pix = np.empty((cap, 2), np.int32)
        cls, ep = np.empty(cap, np.float32), np.empty(cap, np.float32)
        n = C.c_int64(0)
        self._check(self._L.stocs_b200_build_scene_cloud(self.h, _ptr(depth), _ptr(bgr), _ptr(prob), _ptr(edge), W, H,
                                                          K[0], K[1], K[2], K[3], depth_scale, voxel_size, class_threshold,
                                                          _ptr(pos), _ptr(nrm), _ptr(rgb), _ptr(pix), _ptr(cls), _ptr(ep),
                                                          cap, C.byref(n)))
        k = n.value
        return dict(pos=pos[:k].copy(), nrm=nrm[:k].copy(), rgb=rgb[:k].copy(), pix=pix[:k].copy(), cls=cls[:k].copy(),
                    edge=ep[:k].copy())

    def build_scene_clouds(self, depth, bgr, probs, edge, K, depth_scale, voxel_size, class_thresholds):
        """The scene clouds of n objects of one frame in one call: probs (n, H, W), class_thresholds a scalar or n
        values -> n dicts, each equal to build_scene_cloud with that object's map and threshold."""
        depth = np.ascontiguousarray(depth, np.uint16)
        H, W = depth.shape
        bgr = None if bgr is None else np.ascontiguousarray(bgr, np.uint8)
        probs = np.ascontiguousarray(probs, np.uint16)
        assert probs.ndim == 3 and probs.shape[1:] == (H, W), "probs must be (n, H, W)"
        n_obj = probs.shape[0]
        thr = np.ascontiguousarray(np.broadcast_to(np.asarray(class_thresholds, np.float32), (n_obj,)))
        edge = None if edge is None else np.ascontiguousarray(edge, np.uint8)
        offs = np.zeros(n_obj + 1, np.int64)
        cap = H * W   # one object's bound; a frame with more points in all is run again at its exact size
        while True:
            pos, nrm, rgb = (np.empty((cap, 3), np.float32) for _ in range(3))
            pix = np.empty((cap, 2), np.int32)
            cls, ep = np.empty(cap, np.float32), np.empty(cap, np.float32)
            rc = self._L.stocs_b200_build_scene_clouds(self.h, _ptr(depth), _ptr(bgr), _ptr(probs), _ptr(thr), n_obj,
                                                       _ptr(edge), W, H, K[0], K[1], K[2], K[3], depth_scale, voxel_size,
                                                       _ptr(pos), _ptr(nrm), _ptr(rgb), _ptr(pix), _ptr(cls), _ptr(ep),
                                                       cap, _ptr(offs))
            if rc == -5:  # STOCS_E_CAPACITY: offsets are filled
                cap = int(offs[-1])
                continue
            self._check(rc)
            return [dict(pos=pos[a:b].copy(), nrm=nrm[a:b].copy(), rgb=rgb[a:b].copy(), pix=pix[a:b].copy(),
                         cls=cls[a:b].copy(), edge=ep[a:b].copy()) for a, b in zip(offs[:-1], offs[1:])]

    def build_scene_clouds_device(self, depth, bgr, maps, edge, K, depth_scale, voxel_size, class_thresholds, cap=None,
                                  stream=None):
        """build_scene_clouds from a frame already on this context's GPU (stocs_b200_build_scene_clouds_device).  torch
        CUDA tensors: depth [H, W] and maps 2-byte (read as uint16), bgr [H, W, 3] and edge [H, W] uint8 or None; maps
        is a [n, H, W] tensor or a list of n [H, W] tensors, all float32 (used as given) or all 2-byte (converted as
        build_scene_clouds does), and may repeat.  stream (torch.cuda.Stream or a raw handle; default: torch's current
        stream) is the one the inputs were written on.  -> n dicts of CUDA tensor views (pos nrm rgb pix cls edge),
        shaped as build_scene_clouds returns them; cap: rows of the output buffers (default H * W, grown to the
        frame's size when more are needed)."""
        import torch
        two_byte = (torch.uint16, torch.int16)

        def image(t, name, dtypes):
            if t is None:
                return None
            if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype in dtypes):
                raise StocsError(f"build_scene_clouds_device: {name} must be a CUDA tensor of {dtypes}")
            return t.contiguous()

        depth = image(depth, "depth", two_byte)
        H, W = depth.shape
        bgr, edge = image(bgr, "bgr", (torch.uint8,)), image(edge, "edge", (torch.uint8,))
        maps = [image(m, "maps", two_byte + (torch.float32,)) for m in maps]
        if len({m.dtype == torch.float32 for m in maps}) != 1 or any(tuple(m.shape) != (H, W) for m in maps):
            raise StocsError("build_scene_clouds_device: maps must be [H, W] each, all float32 or all 2-byte")
        n_obj = len(maps)
        map_type = 1 if maps[0].dtype == torch.float32 else 0   # STOCS_B200_MAP_F32 / _U16
        table = (C.c_void_p * n_obj)(*[m.data_ptr() for m in maps])
        thr = np.ascontiguousarray(np.broadcast_to(np.asarray(class_thresholds, np.float32), (n_obj,)))
        if stream is None:
            stream = torch.cuda.current_stream(depth.device)
        stream = getattr(stream, "cuda_stream", stream)
        dev = torch.device("cuda", self.device)
        offs = np.zeros(n_obj + 1, np.int64)
        cap = H * W if cap is None else int(cap)
        while True:
            c = max(cap, 1)
            pos, nrm, rgb = (torch.empty((c, 3), dtype=torch.float32, device=dev) for _ in range(3))
            pix = torch.empty((c, 2), dtype=torch.int32, device=dev)
            cls, ep = torch.empty(c, dtype=torch.float32, device=dev), torch.empty(c, dtype=torch.float32, device=dev)
            ptr = [None if t is None else t.data_ptr() for t in (depth, bgr)]
            rc = self._L.stocs_b200_build_scene_clouds_device(
                self.h, ptr[0], ptr[1], table, map_type, _ptr(thr), n_obj, None if edge is None else edge.data_ptr(), W, H,
                K[0], K[1], K[2], K[3], depth_scale, voxel_size, pos.data_ptr(), nrm.data_ptr(), rgb.data_ptr(),
                pix.data_ptr(), cls.data_ptr(), ep.data_ptr(), cap, _ptr(offs), stream)
            if rc == -5:  # STOCS_E_CAPACITY: offsets are filled
                cap = int(offs[-1])
                continue
            self._check(rc)
            return [dict(pos=pos[a:b], nrm=nrm[a:b], rgb=rgb[a:b], pix=pix[a:b], cls=cls[a:b], edge=ep[a:b])
                    for a, b in zip(offs[:-1], offs[1:])]

    # ---- uploads
    def upload_model(self, pos, nrm):
        pos, nrm = _f32(pos, (-1, 3)), _f32(nrm, (-1, 3))
        assert pos.shape == nrm.shape
        self._check(self._L.stocs_b200_upload_model(self.h, _ptr(pos), _ptr(nrm), pos.shape[0]))
        self.M = pos.shape[0]

    def upload_scene(self, pos, nrm, cls, pix=None):
        pos, nrm, cls = _f32(pos, (-1, 3)), _f32(nrm, (-1, 3)), _f32(cls, (-1,))
        pix = None if pix is None else np.ascontiguousarray(pix, np.int32).reshape(-1, 2)
        assert pos.shape == nrm.shape and cls.shape[0] == pos.shape[0]
        self._check(self._L.stocs_b200_upload_scene(self.h, _ptr(pos), _ptr(nrm), _ptr(cls), _ptr(pix),
                                                     pos.shape[0]))
        self.S = pos.shape[0]

    def centroids(self):
        s, m = np.zeros(3, np.float32), np.zeros(3, np.float32)
        self._check(self._L.stocs_b200_get_centroids(self.h, _ptr(s) if self.S else None,
                                                      _ptr(m) if self.M else None))
        return s, m

    def centred(self):
        s = np.empty((self.S, 3), np.float32) if self.S else None
        m = np.empty((self.M, 3), np.float32) if self.M else None
        self._check(self._L.stocs_b200_get_centred(self.h, _ptr(s), _ptr(m)))
        return s, m

    # ---- PPF table
    def ppf_num_pairs(self):
        a, b = C.c_int64(0), C.c_int64(0)
        self._check(self._L.stocs_b200_ppf_num_pairs(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def ppf_num_expanded_keys(self):
        a = C.c_int64(0)
        self._check(self._L.stocs_b200_ppf_num_expanded_keys(self.h, C.byref(a)))
        return a.value

    def ppf_export(self):
        n = C.c_int64(0)
        self._check(self._L.stocs_b200_ppf_export(self.h, None, None, 0, C.byref(n)))
        keys, pairs = np.empty((n.value, 4), np.int32), np.empty((n.value, 2), np.int32)
        self._check(self._L.stocs_b200_ppf_export(self.h, _ptr(keys), _ptr(pairs), n.value, C.byref(n)))
        return keys, pairs

    def upload_ppf_table(self, keys4, pairs2, tr, rot, num_model_points):
        keys4 = np.ascontiguousarray(keys4, np.int32).reshape(-1, 4)
        pairs2 = np.ascontiguousarray(pairs2, np.int32).reshape(-1, 2)
        assert keys4.shape[0] == pairs2.shape[0]
        try:
            self._check(self._L.stocs_b200_upload_ppf_table(self.h, _ptr(keys4), _ptr(pairs2), keys4.shape[0], tr, rot,
                                                             num_model_points))
        except StocsError:
            self.M = 0
            raise

    def ppf_lookup(self, key):
        key = np.ascontiguousarray(key, np.int32).reshape(4)
        n = C.c_int64(0)
        self._check(self._L.stocs_b200_ppf_lookup(self.h, _ptr(key), None, 0, C.byref(n)))
        if n.value < 0:
            return None
        out = np.empty((max(n.value, 1), 2), np.int32)
        self._check(self._L.stocs_b200_ppf_lookup(self.h, _ptr(key), _ptr(out), n.value, C.byref(n)))
        return out[:n.value]

    # ---- sampling / congruent sets / fit
    def sample_bases(self, seed, first_base_no, n_bases):
        ids = np.empty((n_bases, 4), np.int32)
        inv = np.empty((n_bases, 2), np.float32)
        valid = np.empty(n_bases, np.uint8)
        self._check(self._L.stocs_b200_sample_bases(self.h, int(seed), int(first_base_no), n_bases,
                                                     _ptr(ids), _ptr(inv), _ptr(valid)))
        return ids, inv, valid.astype(bool)

    def upload_edge_map(self, edge):
        edge = np.ascontiguousarray(edge, np.uint8)
        self._edge_shape = edge.shape
        self._check(self._L.stocs_b200_upload_edge_map(self.h, _ptr(edge), edge.shape[1], edge.shape[0]))

    def sample_instance_base(self, seed, base_num, dispersion=0.9, want_mask=True):
        ids, inv, valid = np.empty(4, np.int32), np.empty(2, np.float32), np.zeros(1, np.uint8)
        shape = getattr(self, "_edge_shape", None)
        mask = np.zeros(shape, np.uint8) if (want_mask and shape is not None) else None
        self._check(self._L.stocs_b200_sample_instance_base(self.h, int(seed), int(base_num), dispersion, _ptr(ids),
                                                             _ptr(inv), _ptr(valid), _ptr(mask), None))
        return bool(valid[0]), ids, inv, mask

    def class_probability(self):
        out = np.empty(self.S, np.float32)
        self._check(self._L.stocs_b200_get_class_probability(self.h, _ptr(out)))
        return out

    def set_class_probability(self, cls):
        cls = _f32(cls, (-1,))
        assert cls.shape[0] == self.S
        self._check(self._L.stocs_b200_set_class_probability(self.h, _ptr(cls)))

    def find_congruent(self, base_idx, inv, cap=1 << 20):
        base_idx = np.ascontiguousarray(base_idx, np.int32).reshape(-1, 4)
        inv = _f32(inv, (-1, 2))
        nb = base_idx.shape[0]
        offs = np.zeros(nb + 1, np.int64)
        while True:
            quads = np.empty((max(cap, 1), 4), np.int32)
            rc = self._L.stocs_b200_find_congruent(self.h, nb, _ptr(base_idx), _ptr(inv), _ptr(quads), cap,
                                                   _ptr(offs))
            if rc == -5:  # STOCS_E_CAPACITY: offsets are filled, retry with the exact size
                cap = int(offs[-1])
                continue
            self._check(rc)
            return quads[:offs[-1]].copy(), offs

    def fit_transforms(self, base_idx, quads):
        base_idx = np.ascontiguousarray(base_idx, np.int32).reshape(-1, 4)
        quads = np.ascontiguousarray(quads, np.int32).reshape(-1, 4)
        n = quads.shape[0]
        assert base_idx.shape[0] == n
        Tc, Tw = np.empty((n, 16), np.float32), np.empty((n, 16), np.float32)
        ok = np.empty(n, np.uint8)
        self._check(self._L.stocs_b200_fit_transforms(self.h, n, _ptr(base_idx), _ptr(quads), _ptr(Tc),
                                                       _ptr(Tw), _ptr(ok)))
        return Tc, Tw, ok.astype(bool)

    # ---- scoring
    def score_lcp(self, T):
        """Host buffers in, host buffers out (the drop-in call)."""
        T = _f32(T, (-1, 16))
        H = T.shape[0]
        lcp, inl = np.empty(H, np.float32), np.empty(H, np.int32)
        self._check(self._L.stocs_b200_score_lcp(self.h, _ptr(T), H, _ptr(lcp), _ptr(inl)))
        self._last_H = H
        return lcp, inl

    def score_lcp_ptr(self, T_ptr, H, lcp_ptr, inl_ptr):
        """Raw host pointers (e.g. pinned torch tensors)."""
        self._check(self._L.stocs_b200_score_lcp(self.h, T_ptr, H, lcp_ptr, inl_ptr))
        self._last_H = H

    def score_lcp_device(self, dT_ptr, H, dlcp_ptr, dinl_ptr, stream=None):
        self._check(self._L.stocs_b200_score_lcp_device(self.h, dT_ptr, H, dlcp_ptr, dinl_ptr, stream))

    def reduce_best(self, lcp, K=32):
        lcp = None if lcp is None else _f32(lcp, (-1,))
        H = self._last_H if lcp is None else lcp.shape[0]
        bi, bl = C.c_int64(0), C.c_float(0)
        ti, tl = np.empty(K, np.int64), np.empty(K, np.float32)
        self._check(self._L.stocs_b200_reduce_best(self.h, _ptr(lcp), H, K, C.byref(bi), C.byref(bl),
                                                    _ptr(ti), _ptr(tl)))
        return bi.value, bl.value, ti, tl

    def select_above(self, lcp, threshold):
        lcp = _f32(lcp, (-1,))
        n = C.c_int64(0)
        idx, val = np.empty(lcp.size, np.int64), np.empty(lcp.size, np.float32)
        self._check(self._L.stocs_b200_select_above(self.h, _ptr(lcp), lcp.size, threshold, _ptr(idx), _ptr(val),
                                                     lcp.size, C.byref(n)))
        return idx[:n.value].copy(), val[:n.value].copy()

    def icp_point_to_plane(self, src, tgt, tgt_nrm, max_iterations=5, max_dist=0.035):
        """-> (T 4x4, aligned source, pairs per iteration, iterations done, converged)"""
        src, tgt, tgt_nrm = _f32(src, (-1, 3)), _f32(tgt, (-1, 3)), _f32(tgt_nrm, (-1, 3))
        assert tgt.shape == tgt_nrm.shape
        T = np.zeros(16, np.float32)
        out = np.empty_like(src)
        pairs = np.zeros(max(max_iterations, 1), np.int32)
        done, conv = C.c_int32(0), C.c_int32(0)
        self._check(self._L.stocs_b200_icp_point_to_plane(self.h, _ptr(src), src.shape[0], _ptr(tgt), _ptr(tgt_nrm),
                                                           tgt.shape[0], max_iterations, max_dist, _ptr(T), _ptr(out),
                                                           _ptr(pairs), C.byref(done), C.byref(conv)))
        return T.reshape(4, 4).T.copy(), out, pairs, done.value, bool(conv.value)

    def reduce_best_device(self, dlcp_ptr, H, K, index_offset, didx_ptr, dval_ptr, stream=None):
        self._check(self._L.stocs_b200_reduce_best_device(self.h, dlcp_ptr, H, K, index_offset, didx_ptr,
                                                           dval_ptr, stream))

    # ---- multi-GPU (one process per GPU)
    def comm_init(self, unique_id, rank, nranks):
        buf = C.create_string_buffer(bytes(unique_id), 128)
        self._check(self._L.stocs_b200_comm_init(self.h, buf, int(rank), int(nranks)))

    def comm_destroy(self):
        self._check(self._L.stocs_b200_comm_destroy(self.h))

    def score_sharded_device(self, dT_ptr, H_local, index_offset, K, dout_ptr, stream=None):
        """Device pointers; enqueues score -> local top-K records -> ONE all-gather -> merge."""
        self._check(self._L.stocs_b200_score_sharded_device(self.h, dT_ptr, H_local, index_offset, K, dout_ptr, stream))

    def score_sharded(self, T_local, index_offset, K=32, want_local=False):
        """Host buffers -> K best records of the whole list (numpy RECORD array) [, local lcp, inliers]."""
        T_local = _f32(T_local, (-1, 16))
        H = T_local.shape[0]
        out = np.zeros(K, RECORD)
        lcp = np.empty(H, np.float32) if want_local else None
        inl = np.empty(H, np.int32) if want_local else None
        self._check(self._L.stocs_b200_score_sharded(self.h, _ptr(T_local), H, int(index_offset), K, _ptr(out),
                                                      _ptr(lcp), _ptr(inl)))
        return (out, lcp, inl) if want_local else out

    def score_sharded_ptr(self, T_ptr, H_local, index_offset, K, out, lcp_ptr=None, inl_ptr=None):
        """Raw host pointers (e.g. pinned torch tensors); out: RECORD array of K."""
        self._check(self._L.stocs_b200_score_sharded(self.h, T_ptr, H_local, int(index_offset), K, _ptr(out),
                                                      lcp_ptr, inl_ptr))

    def run_pipeline(self, seed, n_bases=100, max_sets=200):
        r = PipelineResult()
        self._check(self._L.stocs_b200_run_pipeline(self.h, int(seed), n_bases, max_sets, C.byref(r)))
        return r

    def run_pipeline_instance(self, seed, n_bases=100, max_sets=200, dispersion=0.9):
        r = PipelineResult()
        self._check(self._L.stocs_b200_run_pipeline_instance(self.h, int(seed), n_bases, max_sets, dispersion, C.byref(r)))
        return r

    # ---- f3: greedy pose clustering
    def cluster_poses(self, T_world, lcp, best_score, acceptable_fraction, maximum_pose_count, min_distance, min_angle,
                      sym_info=(0, 0, 0)):
        """clustering::greedy_clustering on the device -> int64 array of the kept indices, in the order kept
        (T_world: H world poses, 4x4 row-major or 16 column-major floats each)."""
        lcp = _f32(lcp, (-1,))
        T = np.asarray(T_world, np.float32)
        T = _f32(T.transpose(0, 2, 1) if T.ndim == 3 else T, (-1, 16))
        assert T.shape[0] == lcp.shape[0]
        p = _cluster_params(acceptable_fraction, maximum_pose_count, min_distance, min_angle, sym_info)
        cap = max(int(maximum_pose_count) + 1, 1)
        out, n = np.empty(cap, np.int64), C.c_int64(0)
        self._check(self._L.stocs_b200_cluster_poses(self.h, _ptr(T), _ptr(lcp), lcp.shape[0], best_score, C.byref(p),
                                                      _ptr(out), cap, C.byref(n)))
        return out[:n.value].copy()

    def run_pipeline_clustered(self, seed, n_bases=100, max_sets=200, **params):
        """run_pipeline + greedy clustering of its scored list -> (PipelineResult, POSE array).
        params: acceptable_fraction, maximum_pose_count, min_distance, min_angle, sym_info=(0, 0, 0)"""
        p = _cluster_params(**params)
        r, poses, n = PipelineResult(), np.zeros(max(p.maximum_pose_count + 1, 1), POSE), C.c_int32(0)
        self._check(self._L.stocs_b200_run_pipeline_clustered(self.h, int(seed), n_bases, max_sets, C.byref(p), C.byref(r),
                                                               _ptr(poses), poses.shape[0], C.byref(n)))
        return r, poses[:n.value].copy()

    def run_pipeline_instance_clustered(self, seed, n_bases=100, max_sets=200, dispersion=0.9, **params):
        """run_pipeline_instance + greedy clustering of its scored list -> (PipelineResult, POSE array)"""
        p = _cluster_params(**params)
        r, poses, n = PipelineResult(), np.zeros(max(p.maximum_pose_count + 1, 1), POSE), C.c_int32(0)
        self._check(self._L.stocs_b200_run_pipeline_instance_clustered(self.h, int(seed), n_bases, max_sets, dispersion,
                                                                        C.byref(p), C.byref(r), _ptr(poses), poses.shape[0],
                                                                        C.byref(n)))
        return r, poses[:n.value].copy()

    def counters(self):
        c = np.zeros(9, np.int64)
        self._check(self._L.stocs_b200_get_counters(self.h, _ptr(c), 9))
        return c

    SCORE_COUNTER_NAMES = ("queries", "coarse_survivors", "brick_records", "queued", "candidates", "hits",
                           "inliers", "drains", "hypotheses")

    def score_counters(self, dT_ptr, H):
        """Exact data-dependent work of one scoring launch (device transforms) -> dict."""
        c = np.zeros(9, np.int64)
        self._check(self._L.stocs_b200_score_counters(self.h, dT_ptr, H, _ptr(c), 9))
        return dict(zip(self.SCORE_COUNTER_NAMES, (int(v) for v in c)))

    def kernel_ms_stats(self, reset=False):
        """(launches, mean ms, max ms) of the scoring kernel since the last reset (<= 512 launches)."""
        n, mean, mx = C.c_int32(0), C.c_float(0), C.c_float(0)
        self._check(self._L.stocs_b200_kernel_ms_stats(self.h, int(reset), C.byref(n), C.byref(mean), C.byref(mx)))
        return n.value, mean.value, mx.value

    def debug_angle_estimates(self, y, x):
        """-> dict: fp32 estimate / pinned value of atan2(y, x) in degrees, both integer parts, and both forms
        of the 30-degree predicate on d = x (test hook, see include/stocs_b200.h)"""
        y, x = _f32(y, (-1,)), _f32(x, (-1,))
        n = y.shape[0]
        assert x.shape[0] == n
        est, pin = np.empty(n, np.float32), np.empty(n, np.float64)
        ff, pf = np.empty(n, np.int32), np.empty(n, np.int32)
        bf, bp = np.empty(n, np.uint8), np.empty(n, np.uint8)
        self._check(self._L.stocs_b200_debug_angle_estimates(self.h, _ptr(y), _ptr(x), n, _ptr(est), _ptr(pin), _ptr(ff),
                                                             _ptr(pf), _ptr(bf), _ptr(bp)))
        return {"est": est, "pinned": pin, "fast_floor": ff, "pinned_floor": pf, "below30_fast": bf, "below30_pinned": bp}

    def debug_survivor_counts(self, dT_ptr, H, fine=False):
        """survivor count of each of H device transforms (test hook, see include/stocs_b200.h) -> int32
        array: loop 1's count on the coarse map, or with fine=True the count on the fine map that a large
        top-K launch orders and stops its claims by, returned with (fine_shift, coarse_shift)"""
        ns = np.empty(H, np.int32)
        if not fine:
            self._check(self._L.stocs_b200_debug_survivor_counts(self.h, dT_ptr, H, _ptr(ns)))
            return ns
        shifts = np.zeros(2, np.int32)
        self._check(self._L.stocs_b200_debug_fine_survivor_counts(self.h, dT_ptr, H, _ptr(ns), _ptr(shifts)))
        return ns, (int(shifts[0]), int(shifts[1]))

    def debug_kdtree(self, pos, on_device):
        """the reference kd-tree over pos as built on the device (on_device) or on the host (test hook, see
        include/stocs_b200.h) -> (leaf order, node count, int32 [nodes, 3] pre-order dump)"""
        pos = _f32(pos, (-1, 3))
        n = pos.shape[0]
        order, nn, nodes = np.empty(n, np.int32), C.c_int32(0), np.empty((n + 3, 3), np.int32)
        self._check(self._L.stocs_b200_debug_kdtree(self.h, _ptr(pos), n, int(bool(on_device)), _ptr(order), C.byref(nn),
                                                    _ptr(nodes)))
        return order, nn.value, nodes[:nn.value].copy()

    def last_kernel_ms(self):
        ms = C.c_float(0)
        self._check(self._L.stocs_b200_last_kernel_ms(self.h, C.byref(ms)))
        return ms.value


class _BorrowedContext(Context):
    """A context owned by a Group (never destroyed from Python)."""

    def __init__(self, handle, device):
        self._L = lib()
        self.h = C.c_void_p(handle)
        self.device = device
        self.M = self.S = 0
        self._last_H = 0

    def close(self):
        self.h = None


class Group:
    """stocs_b200_group: one process driving several GPUs (hypothesis sharding + one all-gather)."""

    def __init__(self, device_ids, distance_threshold=0.005, ppf_tr_discretization=5, ppf_rot_discretization=5):
        self._L = lib()
        ids = (C.c_int * len(device_ids))(*device_ids)
        g = C.c_void_p()
        rc = self._L.stocs_b200_group_create(C.byref(g), ids, len(device_ids))
        if rc != 0:
            msg = self._L.stocs_b200_last_error(None)
            raise StocsError(f"stocs_b200_group_create failed ({rc}): {msg.decode() if msg else ''}")
        self.g = g
        self.n = len(device_ids)
        self._check(self._L.stocs_b200_group_set_params(self.g, distance_threshold, ppf_tr_discretization,
                                                         ppf_rot_discretization))

    def _check(self, rc):
        if rc != 0:
            msg = self._L.stocs_b200_group_last_error(self.g)
            raise StocsError(f"libstocs_b200 group error {rc}: {msg.decode() if msg else ''}")

    def ctx(self, i):
        return _BorrowedContext(self._L.stocs_b200_group_ctx(self.g, i), i)

    def upload_model(self, pos, nrm):
        pos, nrm = _f32(pos, (-1, 3)), _f32(nrm, (-1, 3))
        self._check(self._L.stocs_b200_group_upload_model(self.g, _ptr(pos), _ptr(nrm), pos.shape[0]))

    def upload_scene(self, pos, nrm, cls, pix=None):
        pos, nrm, cls = _f32(pos, (-1, 3)), _f32(nrm, (-1, 3)), _f32(cls, (-1,))
        pix = None if pix is None else np.ascontiguousarray(pix, np.int32).reshape(-1, 2)
        self._check(self._L.stocs_b200_group_upload_scene(self.g, _ptr(pos), _ptr(nrm), _ptr(cls), _ptr(pix), pos.shape[0]))

    def score_best(self, T, K=32, want_all=False):
        T = _f32(T, (-1, 16))
        H = T.shape[0]
        out = np.zeros(K, RECORD)
        lcp = np.empty(H, np.float32) if want_all else None
        inl = np.empty(H, np.int32) if want_all else None
        self._check(self._L.stocs_b200_group_score_best(self.g, _ptr(T), H, K, _ptr(out), _ptr(lcp), _ptr(inl)))
        return (out, lcp, inl) if want_all else out

    def close(self):
        if getattr(self, "g", None):
            self._L.stocs_b200_group_destroy(self.g)
            self.g = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
