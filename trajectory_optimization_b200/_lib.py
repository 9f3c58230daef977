"""ctypes binding of libcovb200.so (C ABI: include/coverage_b200.h).

The library is built in-tree by `csrc/build.sh` (or `__graft_entry__.build()`); it is never
pip-installed.  Loading is lazy so that importing the package works on a box without the
build, but every op calls `lib()` and therefore fails loudly when the library is missing.
"""
import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
# COV_B200_LIB: another build of the same library (A/B experiments with kernel variants); default: the in-tree build
LIB_PATH = os.environ.get("COV_B200_LIB") or os.path.join(_HERE, "libcovb200.so")
_lock = threading.Lock()
_lib = None

ACC_STRIDE = 22   # COV_ACC_STRIDE
POSE_ACC = 8      # COV_POSE_ACC


class Camera(C.Structure):
    """struct cov_camera."""
    _fields_ = [("img_width", C.c_float), ("img_height", C.c_float), ("min_dist", C.c_float),
                ("max_dist", C.c_float), ("eps", C.c_float)]


class TrajOpts(C.Structure):
    """struct cov_traj_opts (per-call options; all zero = defaults)."""
    _fields_ = [("dense", C.c_int), ("rewards_prefilled", C.c_int), ("prefill_dev", C.c_void_p), ("stats_dev", C.c_void_p)]


MAX_PEERS = 16          # COV_MAX_PEERS
PEER_MAX_F32, PEER_SUM_F64, PEER_MINMAX_F32 = 0, 1, 2


class Peers(C.Structure):
    """struct cov_peers: the world's exchange buffers as addressable from this device."""
    _fields_ = [("ptr", C.c_void_p * MAX_PEERS), ("world", C.c_int), ("rank", C.c_int)]


_vp, _i64, _int, _f, _sz = C.c_void_p, C.c_int64, C.c_int, C.c_float, C.c_size_t
_cam = C.POINTER(Camera)
_opts = C.POINTER(TrajOpts)

# name -> (restype, argtypes); must list every symbol include/coverage_b200.h declares
PROTOTYPES = {
    "cov_version": (_int, []),
    "cov_last_error": (C.c_char_p, []),
    "cov_device_sm_count": (_int, []),
    "cov_pose_workspace_bytes": (_sz, [_i64]),
    "cov_pose_fused": (_int, [_vp, _i64, _vp, _vp, _vp, _vp, _cam, _vp, _vp, _vp, _sz, _vp]),
    "cov_pose_epilogue": (_int, [_vp, _vp, _vp, _vp, _vp]),
    "cov_pose_batch_workspace_bytes": (_sz, [_i64, _int, _opts]),
    "cov_pose_batch_fused": (_int, [_vp, _i64, _vp, _vp, _vp, _int, _vp, _cam, _vp, _vp, _opts, _vp, _sz, _vp]),
    "cov_pose_batch_epilogue": (_int, [_vp, _vp, _int, _vp, _vp]),
    "cov_traj_max_poses": (_int, []),
    "cov_traj_max_poses_pruned": (_int, []),
    "cov_traj_workspace_bytes": (_sz, [_i64, _int]),
    "cov_traj_prefill_applies": (_int, [_i64, _opts]),
    "cov_traj_minmax": (_int, [_vp, _i64, _vp, _vp, _int, _vp, _cam, _vp, _vp, _opts, _vp, _sz, _vp]),
    "cov_traj_fused": (_int, [_vp, _i64, _vp, _vp, _int, _vp, _cam, _vp, _vp, _vp, _vp, _vp, _vp, _opts, _vp, _sz, _vp]),
    "cov_traj_epilogue": (_int, [_vp, _vp, _vp, _int, _i64, _int, _vp, _vp]),
    "cov_traj_regularizers": (_int, [_vp, _vp, _int, _f, _f, _f, _vp, _vp]),
    "cov_sweep_workspace_bytes": (_sz, [_i64, _int, _int]),
    "cov_sweep_rewards": (_int, [_vp, _i64, _vp, _vp, _int, _int, _vp, _cam, _vp, _vp, _vp, _opts, _vp, _sz, _vp]),
    "cov_sweep_fused_workspace_bytes": (_sz, [_i64, _int, _int, _opts]),
    "cov_sweep_fused": (_int, [_vp, _i64, _vp, _vp, _int, _int, _vp, _cam, _vp, _vp, _vp, _opts, _vp, _sz, _vp]),
    "cov_sweep_epilogue": (_int, [_vp, _vp, _vp, _int, _int, _i64, _vp, _vp]),
    "cov_prior_reward_sum": (_int, [_vp, _i64, _vp, _vp]),
    "cov_traj_minmax_prior": (_int, [_vp, _i64, _vp, _vp, _int, _vp, _cam, _vp, _vp, _vp, _opts, _vp, _sz, _vp]),
    "cov_traj_fused_prior": (_int, [_vp, _i64, _vp, _vp, _int, _vp, _cam, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _opts,
                                    _vp, _sz, _vp]),
    "cov_traj_logodds": (_int, [_vp, _i64, _vp, _vp, _int, _vp, _cam, _vp, _vp, _vp, _vp, _opts, _vp, _sz, _vp]),
    "cov_sweep_rewards_prior": (_int, [_vp, _i64, _vp, _vp, _int, _int, _vp, _cam, _vp, _vp, _vp, _vp, _vp, _opts, _vp,
                                       _sz, _vp]),
    "cov_sweep_fused_prior": (_int, [_vp, _i64, _vp, _vp, _int, _int, _vp, _cam, _vp, _vp, _vp, _vp, _vp, _opts, _vp, _sz,
                                     _vp]),
    "cov_weight_sums": (_int, [_vp, _vp, _i64, _vp, _vp]),
    "cov_traj_fused_weighted": (_int, [_vp, _i64, _vp, _vp, _int, _vp, _cam, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                       _opts, _vp, _sz, _vp]),
    "cov_sweep_rewards_weighted": (_int, [_vp, _i64, _vp, _vp, _int, _int, _vp, _cam, _vp, _vp, _vp, _vp, _vp, _vp,
                                          _opts, _vp, _sz, _vp]),
    "cov_sweep_fused_weighted": (_int, [_vp, _i64, _vp, _vp, _int, _int, _vp, _cam, _vp, _vp, _vp, _vp, _vp, _vp, _opts,
                                        _vp, _sz, _vp]),
    "cov_traj_epilogue_dev": (_int, [_vp, _vp, _vp, _int, _vp, _vp, _vp]),
    "cov_sweep_epilogue_dev": (_int, [_vp, _vp, _vp, _int, _int, _vp, _vp, _vp]),
    "cov_sweep_prefix_rewards": (_int, [_vp, _i64, _vp, _vp, _int, _int, _vp, _cam, _vp, _vp, _vp, _vp, _vp, _vp, _opts,
                                        _vp, _sz, _vp]),
    "cov_traj_long_workspace_bytes": (_sz, [_i64, _int, _int]),
    "cov_traj_fused_long": (_int, [_vp, _i64, _vp, _vp, _int, _vp, _cam, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _int,
                                   _opts, _vp, _sz, _vp]),
    "cov_traj_logodds_long": (_int, [_vp, _i64, _vp, _vp, _int, _vp, _cam, _vp, _vp, _vp, _vp, _int, _opts, _vp, _sz, _vp]),
    "cov_peer_region_bytes": (_sz, [_int, _i64, _int]),
    "cov_peer_allreduce": (_int, [_int, _vp, _i64, C.POINTER(Peers), _sz, _vp]),
    "cov_rig_poses": (_int, [_vp, _int, _vp, _int, _vp, _vp, _vp]),
    "cov_rig_poses_backward": (_int, [_vp, _int, _vp, _int, _vp, _vp, _f, _vp, _vp]),
    "cov_cull_workspace_bytes": (_sz, [_i64]),
    "cov_frustum_cull": (_int, [_vp, _i64, _vp, _f, _f, _f, _f, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "cov_hpr_flip": (_int, [_vp, _i64, _f, _vp, _vp, _vp]),
    "cov_hpr_hull_workspace_bytes": (_sz, [_i64]),
    "cov_hpr_hull": (_int, [_vp, _i64, _vp, _vp, _vp, _sz, _vp]),
    "cov_pc2_workspace_bytes": (_sz, [_i64]),
    "cov_pc2_to_xyz": (_int, [_vp, _i64, _int, _int, _int, _int, _int, _int, _vp, _vp, _vp, _sz, _vp]),
    "cov_xyz_to_pc2": (_int, [_vp, _vp, _i64, _vp, _vp, _vp]),
    "cov_voxel_grid_workspace_bytes": (_sz, [_i64]),
    "cov_voxel_grid": (_int, [_vp, _i64, _f, _int, _f, _f, _vp, _vp, _vp, _vp, _sz, _vp]),
    "cov_spatial_sort_workspace_bytes": (_sz, [_i64]),
    "cov_spatial_sort": (_int, [_vp, _i64, _vp, _vp, _vp, _sz, _vp]),
    "cov_sort_pairs_workspace_bytes": (_sz, [_i64]),
    "cov_sort_pairs": (_int, [_vp, _vp, _i64, _int, _int, _vp, _sz, _vp]),
    "cov_tile_boxes_count": (_i64, [_i64]),
    "cov_tile_boxes": (_int, [_vp, _i64, _vp, _vp]),
    "cov_probe_fma": (_i64, [_int, _vp, _vp]),
    "cov_probe_fma2": (_i64, [_int, _vp, _vp]),
    "cov_probe_ex2": (_i64, [_int, _vp, _vp]),
}


def lib():
    """The loaded library; raises RuntimeError if it has not been built."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise RuntimeError(
                        f"{LIB_PATH} not found: build it with trajectory_optimization_b200/csrc/build.sh "
                        "(there is no CPU or PyTorch fallback for the coverage ops)")
                handle = C.CDLL(LIB_PATH)
                for name, (res, args) in PROTOTYPES.items():
                    fn = getattr(handle, name)
                    fn.restype, fn.argtypes = res, args
                _lib = handle
    return _lib


def check(rc, what):
    if rc != 0:
        msg = lib().cov_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed (code {rc}): {msg}")


def camera(img_width, img_height, min_dist, max_dist, eps):
    return Camera(float(img_width), float(img_height), float(min_dist), float(max_dist), float(eps))


def traj_opts(dense=False, rewards_prefilled=False, stats=None, prefill=None):
    """cov_traj_opts; `stats`: None or a CUDA int64/uint64 tensor of 8 counters the evaluation kernels add to;
    `prefill`: None or the fp32 rewards tensor pass A should fill with 1/2 for the pass B that follows."""
    return TrajOpts(1 if dense else 0, 1 if rewards_prefilled else 0, None if prefill is None else prefill.data_ptr(),
                    None if stats is None else stats.data_ptr())
