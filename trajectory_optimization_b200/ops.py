"""torch.autograd.Function wrappers over the C ABI (include/coverage_b200.h).

PyTorch is plumbing here: it owns device memory, streams and (when the cloud is sharded over
ranks) the NCCL communicator.  Every numeric result comes from libcovb200.so.

Sharded use: each rank passes ITS slice of the cloud plus a `group`; the per-pose normalisers
are all-reduced with MIN/MAX, the accumulators with SUM (a few KB), so every rank ends up with
the same scalar and the same pose gradients, while per-point outputs stay sharded.
"""
import contextlib
import ctypes
import os
import threading

import torch

from . import _lib


def _stream(device=None):
    """The caller's current stream ON THE TENSORS' DEVICE (not on whatever device happens to be current)."""
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _guard(t):
    """Device guard for a C-ABI call: the library launches on the CUDA device that is current, so the tensors'
    device is made current for the duration of the call (`ModelPose(..., device='cuda:1')` while cuda:0 is current)."""
    return torch.cuda.device(t.device)


def _call(name, on, *args):
    """One C-ABI call on the device of tensor `on` and on that device's current stream (every entry point takes the
    stream last); raises RuntimeError with the library's message on a non-zero return code.  The device guard is only
    entered when the tensor's device is not the current one (the common case pays two cheap queries)."""
    fn = getattr(_lib.lib(), name)
    dev = on.device
    if dev.index == torch.cuda.current_device():
        rc = fn(*args, ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
    else:
        with torch.cuda.device(dev):
            rc = fn(*args, ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
    if rc:
        _lib.check(rc, name)


def _dev_f32(t, device=None, what="tensor"):
    """fp32, contiguous, on a CUDA device, 16-byte aligned (clones only when it has to)."""
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{what} must be a torch.Tensor")
    if device is not None and t.device != device:
        t = t.to(device)
    if not t.is_cuda:
        raise RuntimeError(f"{what} is on {t.device}: the coverage ops are CUDA-only (no CPU fallback)")
    t = t.detach()
    if t.dtype != torch.float32:
        t = t.float()
    if not t.is_contiguous():
        t = t.contiguous()
    if t.data_ptr() % 16:
        t = t.clone()
    return t


class _Mode(threading.local):
    dense = False      # evaluate every (point, pose) pair (cov_traj_opts.dense)
    stats = None       # CUDA int64 tensor of 8 work counters, or None (cov_traj_opts.stats_dev)


_MODE = _Mode()


@contextlib.contextmanager
def evaluation(dense=None, stats=None):
    """Per-thread defaults of the trajectory ops inside the block: `dense=True` switches the exact pruning off
    (A/B measurements, unordered clouds); `stats` = a CUDA int64 tensor of 8 counters the kernels add to.  Python-side
    only: the C ABI takes these per call (cov_traj_opts) and keeps no process-wide switch."""
    old = (_MODE.dense, _MODE.stats)
    if dense is not None:
        _MODE.dense = bool(dense)
    if stats is not None:
        _MODE.stats = stats
    try:
        yield
    finally:
        _MODE.dense, _MODE.stats = old


def _opts(dense=None, rewards_prefilled=False, prefill=None):
    return _lib.traj_opts(_MODE.dense if dense is None else dense, rewards_prefilled, _MODE.stats, prefill)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr() if t is not None else 0)


def _max_poses_pruned():
    """Poses one pruned call takes (cov_traj_max_poses_pruned); trajectory calls with more take the long path."""
    return _lib.lib().cov_traj_max_poses_pruned()


def _takes_long_path(W, dense):
    return not dense and W > _max_poses_pruned()


def _check_prior(prior, n, device, what="prior_logodds", unit="log-odds"):
    """A per-point prior log-odds tensor (or point weight) as the kernels take it: fp32, shape (n,), on the cloud's
    device; made contiguous and 16-byte aligned (a copy only when it has to).  Shape, dtype and device errors raise
    ValueError naming `what`."""
    if prior is None:
        return None
    if not isinstance(prior, torch.Tensor):
        raise ValueError(f"{what} must be a torch.Tensor, got {type(prior).__name__}")
    if prior.dtype != torch.float32:
        raise ValueError(f"{what} must be float32, got {prior.dtype}")
    if tuple(prior.shape) != (n,):
        raise ValueError(f"{what} must have shape ({n},) (one {unit} per point), got {tuple(prior.shape)}")
    if prior.device != device:
        raise ValueError(f"{what} is on {prior.device}, the cloud on {device}")
    prior = prior.detach()
    if not prior.is_contiguous():
        prior = prior.contiguous()
    if prior.is_cuda and prior.data_ptr() % 16:
        prior = prior.clone()
    return prior


def _check_weight(weight, n, device, what="weight"):
    """A per-point weight as the kernels take it (see _check_prior), or None.  Values are not checked here (that would
    synchronise with the host): finite, >= 0 and a positive sum are the caller's to ensure."""
    return _check_prior(weight, n, device, what, unit="weight")


def _all_reduce(t, op, group):
    if group is not None:
        import torch.distributed as dist
        dist.all_reduce(t, op=op, group=group)


def _reduce_ops():
    import torch.distributed as dist
    return dist.ReduceOp.MIN, dist.ReduceOp.MAX, dist.ReduceOp.SUM


class PeerExchange:
    """The world's exchange buffers for the in-kernel NVLink all-reduces of one (group, device, pose count): symmetric
    memory allocated and rendezvoused ONCE (outside any graph capture), then used by `cov_peer_allreduce`
    (csrc/cov_peer.cu) for the 2 W normalisers and the 22 W + 1 accumulator doubles of every step."""

    def __init__(self, group, device, W):
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        L = _lib.lib()
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        if self.world > _lib.MAX_PEERS:
            raise RuntimeError(f"peer exchange supports up to {_lib.MAX_PEERS} ranks")
        self.n_mm, self.n_acc = 2 * W, W * _lib.ACC_STRIDE + 1
        b_mm = (L.cov_peer_region_bytes(_lib.PEER_MINMAX_F32, self.n_mm, self.world) + 255) // 256 * 256
        b_acc = (L.cov_peer_region_bytes(_lib.PEER_SUM_F64, self.n_acc, self.world) + 255) // 256 * 256
        self.off_mm, self.off_acc = 0, b_mm
        with torch.cuda.device(device):
            self.buf = symm.empty(b_mm + b_acc, dtype=torch.uint8, device=device)
            self.buf.zero_()
            self.handle = symm.rendezvous(self.buf, group)
            torch.cuda.synchronize(device)
        dist.barrier(group)      # every rank's buffer is zeroed before anybody pushes into it
        self.peers = _lib.Peers()
        for r, ptr in enumerate(self.handle.buffer_ptrs):
            self.peers.ptr[r] = ptr
        self.peers.world, self.peers.rank = self.world, self.rank

    def reduce(self, kind, t, offset):
        _call("cov_peer_allreduce", t, kind, _ptr(t), t.numel(), ctypes.byref(self.peers), offset)


_PEER_CACHE = {}
_PEER_STATE = {"enabled": os.environ.get("COV_PEER_EXCHANGE", "1") != "0", "warned": False}


def peer_exchange(group, device, W):
    """The PeerExchange for (group, device, W), or None when the in-kernel exchange is off or unavailable (then the
    collectives are NCCL all-reduces).  Created on first use, which must happen outside CUDA-graph capture (any eager
    warm-up step does it)."""
    if group is None or not _PEER_STATE["enabled"] or device.type != "cuda" or W > 2048:
        return None
    key = (id(group), device.index, W)
    if key not in _PEER_CACHE:
        try:
            import torch.distributed as dist
            if dist.get_backend(group) != "nccl":
                raise RuntimeError("peer exchange needs one CUDA device per rank (nccl group)")
            if torch.cuda.is_current_stream_capturing():
                raise RuntimeError("first use inside a CUDA-graph capture")
            _PEER_CACHE[key] = PeerExchange(group, device, W)
        except Exception as exc:   # no P2P / symmetric memory on this box: the NCCL path is equivalent
            _PEER_CACHE[key] = None
            if not _PEER_STATE["warned"]:
                _PEER_STATE["warned"] = True
                import warnings
                warnings.warn(f"in-kernel NVLink exchange unavailable ({str(exc).splitlines()[0][:160]}); using NCCL all-reduces")
    return _PEER_CACHE[key]


def _all_reduce_minmax(minmax, W, group):
    """Global per-pose minima (first W) and maxima (last W) in ONE exchange: the in-kernel NVLink all-reduce
    (MIN | MAX halves) when available, else one NCCL MAX with the minima negated (MIN(x) = -MAX(-x), exact)."""
    if group is None:
        return
    px = peer_exchange(group, minmax.device, W) if minmax.is_cuda and minmax.dtype == torch.float32 else None
    if px is not None and px.n_mm == minmax.numel():
        px.reduce(_lib.PEER_MINMAX_F32, minmax, px.off_mm)
        return
    minmax[:W].neg_()
    _all_reduce(minmax, _reduce_ops()[1], group)
    minmax[:W].neg_()


def _all_reduce_acc(acc, W, group):
    """SUM of the 22 W + 1 accumulator doubles over the ranks (in rank order: identical on every rank)."""
    if group is None:
        return
    px = peer_exchange(group, acc.device, W) if acc.is_cuda and acc.dtype == torch.float64 else None
    if px is not None and px.n_acc == acc.numel():
        px.reduce(_lib.PEER_SUM_F64, acc, px.off_acc)
        return
    _all_reduce(acc, _reduce_ops()[2], group)


class CudaBackend:
    """The five C-ABI calls of the coverage path on device tensors.  `ops._BACKEND` is the only instance the
    product uses; the N>1 CPU tests swap in a stand-in with the same methods to exercise the collective
    plumbing below over gloo."""

    def prepare(self, t, device=None, what="tensor"):
        return _dev_f32(t, device, what)

    def order_cloud(self, pts, spatial_sort_cloud=True):
        """Once per cloud (ModelTraj): Morton-ordered copy, its permutation and the 128-point boxes."""
        perm = None
        if spatial_sort_cloud and pts.shape[0] > 0:
            pts, perm = spatial_sort(pts)
        return pts, perm, tile_boxes(pts)

    def pose_fused(self, pts, t, q, Kd, cam, w, obs):
        L = _lib.lib()
        n = pts.shape[0]
        acc = torch.empty(_lib.POSE_ACC, dtype=torch.float64, device=pts.device)
        ws_bytes = L.cov_pose_workspace_bytes(n)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=pts.device)
        _call("cov_pose_fused", pts, _ptr(pts), n, _ptr(w), _ptr(t), _ptr(q), _ptr(Kd), ctypes.byref(cam), _ptr(obs),
                                    _ptr(acc), _ptr(ws), ws_bytes)
        return acc

    def pose_epilogue(self, acc, t, q):
        out = torch.empty(8, dtype=torch.float32, device=acc.device)
        _call("cov_pose_epilogue", acc, _ptr(acc), _ptr(t), _ptr(q), _ptr(out))
        return out

    def pose_batch_workspace_bytes(self, pts, K):
        opts = _opts()
        return _lib.lib().cov_pose_batch_workspace_bytes(pts.shape[0], K, ctypes.byref(opts))

    def pose_batch_fused(self, pts, T, Q, Kd, cam, w, boxes=None, ws=None):
        """This cloud's COV_POSE_ACC sums of each of the K poses: (K * 8) fp64 (cov_pose_batch_fused)."""
        K, n, dev = T.shape[0], pts.shape[0], pts.device
        ws_bytes = self.pose_batch_workspace_bytes(pts, K)
        if ws is None or ws.numel() < ws_bytes or ws.device != dev:
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        acc = torch.empty(K * _lib.POSE_ACC, dtype=torch.float64, device=dev)
        opts = _opts()
        _call("cov_pose_batch_fused", pts, _ptr(pts), n, _ptr(w), _ptr(T), _ptr(Q), K, _ptr(Kd), ctypes.byref(cam),
              _ptr(boxes), _ptr(acc), ctypes.byref(opts), _ptr(ws), ws.numel())
        return acc

    def pose_batch_epilogue(self, acc, Q):
        """(K, 8) fp32: per pose [total | d total/d trans (3) | d total/d quat (4)] from the summed sums."""
        K = Q.shape[0]
        out = torch.empty(K, 8, dtype=torch.float32, device=acc.device)
        _call("cov_pose_batch_epilogue", acc, _ptr(acc), _ptr(Q), K, _ptr(out))
        return out

    def traj_workspace_bytes(self, pts, W):
        """Workspace of both passes of a W-pose call; above cov_traj_max_poses_pruned() poses, of the long path."""
        if W > _max_poses_pruned():
            return _lib.lib().cov_traj_long_workspace_bytes(pts.shape[0], W, 0)
        return _lib.lib().cov_traj_workspace_bytes(pts.shape[0], W)

    def traj_workspace(self, pts, W):
        return torch.empty(self.traj_workspace_bytes(pts, W), dtype=torch.uint8, device=pts.device)

    def prefill_applies(self, pts, dense=None):
        """Will pass A on this cloud honour a `prefill` buffer (pruned path)?"""
        opts = _opts(dense)
        return bool(_lib.lib().cov_traj_prefill_applies(pts.shape[0], ctypes.byref(opts)))

    def prior_sum(self, prior):
        """sum_j sigmoid(prior_j) in fp64 on the device, (1,) (cov_prior_reward_sum): the reward-sum base of a prior."""
        out = torch.empty(1, dtype=torch.float64, device=prior.device)
        _call("cov_prior_reward_sum", prior, _ptr(prior), prior.shape[0], _ptr(out))
        return out

    def weight_sums(self, weight, prior=None):
        """[sum_j w_j r0_j, sum_j w_j] in fp64 on the device, (2,) (cov_weight_sums); r0_j = sigmoid(prior_j) or 1/2: the
        reward-sum base and the denominator of the weighted calls."""
        out = torch.empty(2, dtype=torch.float64, device=weight.device)
        _call("cov_weight_sums", weight, _ptr(weight), _ptr(prior), weight.shape[0], _ptr(out))
        return out

    def traj_minmax(self, pts, P, Q, Kd, cam, boxes=None, ws=None, dense=None, prefill=None, prior=None):
        """`prior` (indexed like `prefill`): the pre-fill writes sigmoid(prior_i) instead of 1/2."""
        W = P.shape[0]
        minmax = torch.empty(2 * W, dtype=torch.float32, device=pts.device)
        ws = self.traj_workspace(pts, W) if ws is None else ws
        opts = _opts(dense, prefill=prefill)
        if prior is not None and prefill is not None:
            _call("cov_traj_minmax_prior", pts, _ptr(pts), pts.shape[0], _ptr(P), _ptr(Q), W, _ptr(Kd), ctypes.byref(cam),
                  _ptr(boxes), _ptr(minmax), _ptr(prior), ctypes.byref(opts), _ptr(ws), ws.numel())
            return minmax
        _call("cov_traj_minmax", pts, _ptr(pts), pts.shape[0], _ptr(P), _ptr(Q), W, _ptr(Kd), ctypes.byref(cam),
              _ptr(boxes), _ptr(minmax), ctypes.byref(opts), _ptr(ws), ws.numel())
        return minmax

    def traj_fused(self, pts, P, Q, Kd, cam, minmax, upstream, rewards, reward_index=None, boxes=None, ws=None,
                   dense=None, prefilled=False, prior=None, prior_sum=None, weight=None, wsums=None):
        """`weight` (with `wsums` from weight_sums): the weighted sums of cov_traj_fused_weighted (no upstream)."""
        W, n = P.shape[0], pts.shape[0]
        acc = torch.empty(W * _lib.ACC_STRIDE + 1, dtype=torch.float64, device=pts.device)
        ws = self.traj_workspace(pts, W) if ws is None else ws
        opts = _opts(dense, rewards_prefilled=prefilled)
        if weight is not None:
            _call("cov_traj_fused_weighted", pts, _ptr(pts), n, _ptr(P), _ptr(Q), W, _ptr(Kd), ctypes.byref(cam),
                  _ptr(boxes), _ptr(minmax), _ptr(reward_index), _ptr(rewards), _ptr(acc), _ptr(prior), _ptr(weight),
                  _ptr(wsums), ctypes.byref(opts), _ptr(ws), ws.numel())
            return acc
        if prior is not None:
            _call("cov_traj_fused_prior", pts, _ptr(pts), n, _ptr(P), _ptr(Q), W, _ptr(Kd), ctypes.byref(cam), _ptr(boxes),
                  _ptr(minmax), _ptr(upstream), _ptr(reward_index), _ptr(rewards), _ptr(acc), _ptr(prior), _ptr(prior_sum),
                  ctypes.byref(opts), _ptr(ws), ws.numel())
            return acc
        _call("cov_traj_fused", pts, _ptr(pts), n, _ptr(P), _ptr(Q), W, _ptr(Kd), ctypes.byref(cam), _ptr(boxes),
              _ptr(minmax), _ptr(upstream), _ptr(reward_index), _ptr(rewards), _ptr(acc), ctypes.byref(opts), _ptr(ws),
              ws.numel())
        return acc

    def traj_logodds(self, pts, P, Q, Kd, cam, minmax, out, reward_index=None, boxes=None, ws=None, dense=None):
        """out (pre-filled with the prior, indexed like the rewards) += L_j where L_j != 0 (cov_traj_logodds)."""
        W, n = P.shape[0], pts.shape[0]
        ws = self.traj_workspace(pts, W) if ws is None else ws
        opts = _opts(dense)
        _call("cov_traj_logodds", pts, _ptr(pts), n, _ptr(P), _ptr(Q), W, _ptr(Kd), ctypes.byref(cam), _ptr(boxes),
              _ptr(minmax), _ptr(reward_index), _ptr(out), ctypes.byref(opts), _ptr(ws), ws.numel())
        return out

    def sweep_minmax(self, pts, P, Q, Kd, cam, boxes=None, ws=None, dense=None, prefill=None, prior=None):
        """Per-pose minima and maxima of all T*P poses of a sweep, or of the W poses of a long trajectory (pass A, one
        pose-table-full at a time).  `ws`: a kept workspace of at least cov_traj_workspace_bytes(n, chunk) bytes;
        `prefill` (with `prior`, indexed like it): the first chunk pre-fills it as traj_minmax does."""
        L = _lib.lib()
        W, n, dev = P.shape[0], pts.shape[0], pts.device
        minmax = torch.empty(2 * W, dtype=torch.float32, device=dev)
        chunk = L.cov_traj_max_poses_pruned() if self.prefill_applies(pts, dense) else L.cov_traj_max_poses()
        ws_bytes = L.cov_traj_workspace_bytes(n, min(W, chunk))
        if ws is None or ws.numel() < ws_bytes:
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        for w0 in range(0, W, chunk):
            w1 = min(W, w0 + chunk)
            mm = torch.empty(2 * (w1 - w0), dtype=torch.float32, device=dev)
            fill = prefill if w0 == 0 else None
            opts = _opts(dense, prefill=fill)
            if prior is not None and fill is not None:
                _call("cov_traj_minmax_prior", pts, _ptr(pts), n, _ptr(P[w0:w1]), _ptr(Q[w0:w1]), w1 - w0, _ptr(Kd),
                      ctypes.byref(cam), _ptr(boxes), _ptr(mm), _ptr(prior), ctypes.byref(opts), _ptr(ws), ws.numel())
            else:
                _call("cov_traj_minmax", pts, _ptr(pts), n, _ptr(P[w0:w1]), _ptr(Q[w0:w1]), w1 - w0, _ptr(Kd),
                      ctypes.byref(cam), _ptr(boxes), _ptr(mm), ctypes.byref(opts), _ptr(ws), ws.numel())
            minmax[w0:w1] = mm[:w1 - w0]
            minmax[W + w0:W + w1] = mm[w1 - w0:]
        return minmax

    def traj_fused_long(self, pts, P, Q, Kd, cam, minmax, upstream, rewards, reward_index=None, boxes=None, ws=None,
                        prefilled=False, prior=None, base=None, weight=None, pose_chunk=0):
        """traj_fused over any number of poses, in chunks of `pose_chunk` (0: cov_traj_max_poses_pruned()) with the fused
        log-odds carried between them (cov_traj_fused_long).  `base`: prior_sum(prior) with a prior alone,
        weight_sums(weight, prior) with a weight, else None."""
        W, n = P.shape[0], pts.shape[0]
        acc = torch.empty(W * _lib.ACC_STRIDE + 1, dtype=torch.float64, device=pts.device)
        ws_bytes = _lib.lib().cov_traj_long_workspace_bytes(n, W, pose_chunk)
        if ws is None or ws.numel() < ws_bytes or ws.device != pts.device:
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=pts.device)
        opts = _opts(False, rewards_prefilled=prefilled)
        _call("cov_traj_fused_long", pts, _ptr(pts), n, _ptr(P), _ptr(Q), W, _ptr(Kd), ctypes.byref(cam), _ptr(boxes),
              _ptr(minmax), _ptr(upstream), _ptr(reward_index), _ptr(rewards), _ptr(acc), _ptr(prior), _ptr(base),
              _ptr(weight), int(pose_chunk), ctypes.byref(opts), _ptr(ws), ws.numel())
        return acc

    def traj_logodds_long(self, pts, P, Q, Kd, cam, minmax, out, reward_index=None, boxes=None, ws=None, pose_chunk=0):
        """traj_logodds over any number of poses, in chunks of `pose_chunk` (cov_traj_logodds_long)."""
        W, n = P.shape[0], pts.shape[0]
        ws_bytes = _lib.lib().cov_traj_long_workspace_bytes(n, W, pose_chunk)
        if ws is None or ws.numel() < ws_bytes or ws.device != pts.device:
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=pts.device)
        opts = _opts(False)
        _call("cov_traj_logodds_long", pts, _ptr(pts), n, _ptr(P), _ptr(Q), W, _ptr(Kd), ctypes.byref(cam), _ptr(boxes),
              _ptr(minmax), _ptr(reward_index), _ptr(out), int(pose_chunk), ctypes.byref(opts), _ptr(ws), ws.numel())
        return out

    def sweep_sums(self, pts, P, Q, T, Pn, Kd, cam, boxes, minmax, prior=None, prior_sum=None, weight=None, wsums=None):
        """sum_j rewards_j(t) over this cloud for every trajectory t (fp64); `prior` in the cloud's order.  `weight` (cloud's
        order, with `wsums`): sum_j w_j rewards_j(t)."""
        L = _lib.lib()
        n, dev = pts.shape[0], pts.device
        ws_bytes = L.cov_sweep_workspace_bytes(n, T, Pn)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        sums = torch.zeros(T, dtype=torch.float64, device=dev)
        opts = _opts()
        if weight is not None:
            _call("cov_sweep_rewards_weighted", pts, _ptr(pts), n, _ptr(P), _ptr(Q), T, Pn, _ptr(Kd), ctypes.byref(cam),
                  _ptr(boxes), _ptr(minmax), _ptr(sums), _ptr(prior), _ptr(weight), _ptr(wsums), ctypes.byref(opts),
                  _ptr(ws), ws_bytes)
            return sums
        if prior is not None:
            _call("cov_sweep_rewards_prior", pts, _ptr(pts), n, _ptr(P), _ptr(Q), T, Pn, _ptr(Kd), ctypes.byref(cam),
                  _ptr(boxes), _ptr(minmax), _ptr(sums), _ptr(prior), _ptr(prior_sum), ctypes.byref(opts), _ptr(ws), ws_bytes)
            return sums
        _call("cov_sweep_rewards", pts, _ptr(pts), n, _ptr(P), _ptr(Q), T, Pn, _ptr(Kd), ctypes.byref(cam), _ptr(boxes),
              _ptr(minmax), _ptr(sums), ctypes.byref(opts), _ptr(ws), ws_bytes)
        return sums

    def sweep_prefix_sums(self, pts, P, Q, T, Pn, Kd, cam, boxes, minmax, prior=None, base=None, weight=None):
        """(T Pn,) fp64: entry t Pn + i = sweep_sums of trajectory t cut after its pose i, over this cloud
        (cov_sweep_prefix_rewards).  `base`: prior_sum(prior) with a prior alone, weight_sums(weight, prior) with a
        weight, else None."""
        L = _lib.lib()
        n, dev = pts.shape[0], pts.device
        ws_bytes = L.cov_sweep_workspace_bytes(n, T, Pn)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        out = torch.empty(T * Pn, dtype=torch.float64, device=dev)
        opts = _opts()
        _call("cov_sweep_prefix_rewards", pts, _ptr(pts), n, _ptr(P), _ptr(Q), T, Pn, _ptr(Kd), ctypes.byref(cam),
              _ptr(boxes), _ptr(minmax), _ptr(prior), _ptr(weight), _ptr(base), _ptr(out), ctypes.byref(opts), _ptr(ws),
              ws_bytes)
        return out

    def traj_epilogue(self, acc, minmax, Q, n_total, upstream_mode, den=None):
        """`den` ((1,) fp64 on the device, sum_j w_j): the weighted mean's epilogue (cov_traj_epilogue_dev) in place of
        n_total."""
        W = Q.shape[0]
        out = torch.empty(1 + 7 * W, dtype=torch.float32, device=acc.device)
        if den is not None:
            _call("cov_traj_epilogue_dev", acc, _ptr(acc), _ptr(minmax), _ptr(Q), W, _ptr(den), _ptr(out))
            return out
        _call("cov_traj_epilogue", acc, _ptr(acc), _ptr(minmax), _ptr(Q), W, n_total, upstream_mode, _ptr(out))
        return out

    def sweep_fused_workspace_bytes(self, pts, T, Pn, dense=None):
        """Workspace of a cov_sweep_fused call on this cloud with the current (or the given) dense mode."""
        opts = _opts(dense)
        return _lib.lib().cov_sweep_fused_workspace_bytes(pts.shape[0], T, Pn, ctypes.byref(opts))

    def sweep_fused(self, pts, P, Q, T, Pn, Kd, cam, boxes, minmax, ws=None, prior=None, prior_sum=None, weight=None,
                    wsums=None):
        """This cloud's pass-B accumulators of every trajectory: T blocks of 22 Pn + 1 doubles (cov_sweep_fused);
        `prior` in the cloud's order; `weight` (cloud's order, with `wsums`): cov_sweep_fused_weighted."""
        n, dev = pts.shape[0], pts.device
        ws_bytes = self.sweep_fused_workspace_bytes(pts, T, Pn)
        if ws is None or ws.numel() < ws_bytes or ws.device != dev:
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        acc = torch.empty(T * (Pn * _lib.ACC_STRIDE + 1), dtype=torch.float64, device=dev)
        opts = _opts()
        if weight is not None:
            _call("cov_sweep_fused_weighted", pts, _ptr(pts), n, _ptr(P), _ptr(Q), T, Pn, _ptr(Kd), ctypes.byref(cam),
                  _ptr(boxes), _ptr(minmax), _ptr(acc), _ptr(prior), _ptr(weight), _ptr(wsums), ctypes.byref(opts),
                  _ptr(ws), ws.numel())
            return acc
        if prior is not None:
            _call("cov_sweep_fused_prior", pts, _ptr(pts), n, _ptr(P), _ptr(Q), T, Pn, _ptr(Kd), ctypes.byref(cam),
                  _ptr(boxes), _ptr(minmax), _ptr(acc), _ptr(prior), _ptr(prior_sum), ctypes.byref(opts), _ptr(ws),
                  ws.numel())
            return acc
        _call("cov_sweep_fused", pts, _ptr(pts), n, _ptr(P), _ptr(Q), T, Pn, _ptr(Kd), ctypes.byref(cam), _ptr(boxes),
              _ptr(minmax), _ptr(acc), ctypes.byref(opts), _ptr(ws), ws.numel())
        return acc

    def sweep_epilogue(self, acc, minmax, Q, T, Pn, n_total, den=None):
        """[T means | T Pn 3 d mean_t/d poses | T Pn 4 d mean_t/d quats] (fp32) from the summed accumulators; `den` ((1,)
        fp64 on the device): the denominator in place of n_total (cov_sweep_epilogue_dev, weighted means)."""
        out = torch.empty(T * (1 + 7 * Pn), dtype=torch.float32, device=acc.device)
        if den is not None:
            _call("cov_sweep_epilogue_dev", acc, _ptr(acc), _ptr(minmax), _ptr(Q), T, Pn, _ptr(den), _ptr(out))
            return out
        _call("cov_sweep_epilogue", acc, _ptr(acc), _ptr(minmax), _ptr(Q), T, Pn, n_total, _ptr(out))
        return out


_BACKEND = CudaBackend()


def _weight_sums(B, w, prior, group):
    """(this shard's cov_weight_sums (2,), the denominator sum_j w_j over every rank (1,)): with a group the denominator
    is all-reduced (SUM of one double); the base [0] stays per shard, the accumulators' all-reduce sums it."""
    wsums = B.weight_sums(w, prior)
    if group is None:
        return wsums, wsums[1:]
    den = wsums[1:].clone()
    _all_reduce(den, _reduce_ops()[2], group)
    return wsums, den


class CoveragePoseFn(torch.autograd.Function):
    """obs_j = dist_mask*fov_mask[*weight_j], total = sum_j obs_j (reference src/model.py:98-127)."""

    @staticmethod
    def forward(ctx, points, trans, quat, K, cam, weight, group):
        B = _BACKEND
        dev = points.device
        pts = B.prepare(points, what="points")
        t = B.prepare(trans, dev, "trans").reshape(3)
        q = B.prepare(quat, dev, "quat").reshape(4)
        Kd = B.prepare(K, dev, "intrins").reshape(9)
        w = None if weight is None else B.prepare(weight, dev, "weight").reshape(-1)
        n = pts.shape[0]
        obs = torch.empty(n, dtype=torch.float32, device=dev)
        out = CoveragePoseFn._run(pts, t, q, Kd, cam, w, obs, group)
        ctx.cam, ctx.group = cam, group
        ctx.shapes = (trans.shape, quat.shape)
        ctx.save_for_backward(pts, t, q, Kd, w, out)
        ctx.set_materialize_grads(False)
        return obs, out[0].clone()

    @staticmethod
    def _run(pts, t, q, Kd, cam, w, obs, group):
        acc = _BACKEND.pose_fused(pts, t, q, Kd, cam, w, obs)   # this shard's sums (8 doubles)
        if group is not None:
            _all_reduce(acc, _reduce_ops()[2], group)
        return _BACKEND.pose_epilogue(acc, t, q)

    @staticmethod
    def backward(ctx, g_obs, g_total):
        pts, t, q, Kd, w, out = ctx.saved_tensors
        g_t = g_q = None
        if g_total is not None:
            g_t = g_total * out[1:4]
            g_q = g_total * out[4:8]
        if g_obs is not None:
            # someone differentiated through the per-point vector: one more pass with
            # weight_j = upstream_j [* weight_j]
            up = _BACKEND.prepare(g_obs, pts.device, "grad_obs").reshape(-1)
            if w is not None:
                up = up * w
            o2 = CoveragePoseFn._run(pts, t, q, Kd, ctx.cam, up, None, ctx.group)
            g_t = o2[1:4] if g_t is None else g_t + o2[1:4]
            g_q = o2[4:8] if g_q is None else g_q + o2[4:8]
        ts, qs = ctx.shapes
        return (None, None if g_t is None else g_t.reshape(ts), None if g_q is None else g_q.reshape(qs),
                None, None, None, None)


class CoveragePoseBatchFn(torch.autograd.Function):
    """totals_k = sum_j obs_j(pose k) for K candidate poses on one cloud, each as CoveragePoseFn computes its total, and
    d totals_k / d (trans_k, quat_k) from the same pass (cov_pose_batch_fused).  No per-point output exists, so the
    backward is g_k times the stored gradient rows: no second pass."""

    @staticmethod
    def forward(ctx, pts, trans, quats, K, cam, weight, group, boxes, workspace):
        B = _BACKEND
        dev = pts.device
        T = B.prepare(trans, dev, "trans").reshape(-1, 3)
        Q = B.prepare(quats, dev, "quats").reshape(-1, 4)
        Kd = B.prepare(K, dev, "intrins").reshape(9)
        acc = B.pose_batch_fused(pts, T, Q, Kd, cam, weight, boxes, workspace)   # this shard's sums, K x 8 doubles
        if group is not None:
            _all_reduce(acc, _reduce_ops()[2], group)
        out = B.pose_batch_epilogue(acc, Q)
        ctx.shapes = (trans.shape, quats.shape)
        ctx.save_for_backward(out)
        return out[:, 0].clone()

    @staticmethod
    def backward(ctx, g_totals):
        (out,) = ctx.saved_tensors
        ts, qs = ctx.shapes
        g = g_totals.reshape(-1, 1).to(out.dtype)
        return None, (g * out[:, 1:4]).reshape(ts), (g * out[:, 4:8]).reshape(qs), None, None, None, None, None, None


class CoverageTrajFn(torch.autograd.Function):
    """rewards_j = sigmoid(sum_w logit(clip(normalised m_jw))), mean = mean_j rewards_j
    over the poses given (reference src/model.py:217-237, :246)."""

    @staticmethod
    def forward(ctx, points, poses, quats, K, cam, n_total, group, reward_index=None, boxes=None, dense=None,
                workspace=None, prior=None, prior_sum=None, weight=None, wsums=None, den=None):
        # prior / prior_sum: the checked (N,) prior log-odds in the order of the rewards and sum_j sigmoid(prior_j) of
        # this shard ((1,) fp64 on the device), or None.  weight / wsums / den: the checked (N,) point weight in the same
        # order, this shard's cov_weight_sums (2,) and the global sum_j w_j (1,): the mean is then the weighted mean
        # (prior_sum may be None: only the gradient through the rewards needs it, and computes it then)
        B = _BACKEND
        dev = points.device
        pts = B.prepare(points, what="points")
        if reward_index is not None and (reward_index.dtype != torch.int32 or reward_index.shape[0] != pts.shape[0]
                                         or reward_index.device != dev or not reward_index.is_contiguous()):
            raise ValueError("reward_index must be a contiguous int32 tensor with one entry per point, on the cloud's device")
        P = B.prepare(poses, dev, "poses").reshape(-1, 3)
        Q = B.prepare(quats, dev, "quats").reshape(-1, 4)
        Kd = B.prepare(K, dev, "intrins").reshape(9)
        W, n = P.shape[0], pts.shape[0]
        if Q.shape[0] != W:
            raise ValueError("poses and quats disagree on the number of waypoints")
        n_total = int(n if n_total is None else n_total)
        dense = _MODE.dense if dense is None else bool(dense)
        ws = workspace                                       # shared by both passes; a caller may keep one per cloud
        if ws is None or ws.numel() < B.traj_workspace_bytes(pts, W) or ws.device != dev:
            ws = B.traj_workspace(pts, W)
        rewards = torch.empty(n, dtype=torch.float32, device=dev)
        # the pruned pass A pre-fills pass B's rewards with 1/2 under its idle memory bandwidth
        prefill = rewards if B.prefill_applies(pts, dense) else None
        if _takes_long_path(W, dense):   # pass A one pose-table-full at a time (the first pre-fills)
            minmax = B.sweep_minmax(pts, P, Q, Kd, cam, boxes, ws, dense, prefill, prior)
        elif prior is None:
            minmax = B.traj_minmax(pts, P, Q, Kd, cam, boxes, ws, dense, prefill)   # pass A on this shard
        else:   # the pre-fill writes sigmoid(prior_i)
            minmax = B.traj_minmax(pts, P, Q, Kd, cam, boxes, ws, dense, prefill, prior)
        _all_reduce_minmax(minmax, W, group)                 # global normalisers: W minima, W maxima
        out = CoverageTrajFn._run(pts, P, Q, Kd, cam, minmax, None, rewards, n_total, group, reward_index, boxes, ws,
                                  dense, prefill is not None, prior, prior_sum, weight, wsums, den)
        ctx.cam, ctx.group, ctx.n_total, ctx.reward_index, ctx.boxes = cam, group, n_total, reward_index, boxes
        ctx.dense, ctx.prior, ctx.prior_sum = dense, prior, prior_sum
        ctx.shapes = (poses.shape, quats.shape)
        ctx.save_for_backward(pts, P, Q, Kd, minmax, out)
        ctx.set_materialize_grads(False)
        return rewards, out[0].clone()

    @staticmethod
    def _run(pts, P, Q, Kd, cam, minmax, upstream, rewards, n_total, group, reward_index=None, boxes=None, ws=None,
             dense=None, prefilled=False, prior=None, prior_sum=None, weight=None, wsums=None, den=None):
        if _takes_long_path(P.shape[0], _MODE.dense if dense is None else dense):   # pass B in pose chunks
            acc = _BACKEND.traj_fused_long(pts, P, Q, Kd, cam, minmax, upstream, rewards, reward_index, boxes, ws,
                                           prefilled, prior, wsums if weight is not None else prior_sum, weight)
        elif weight is not None:   # pass B, weighted sums (never with an upstream)
            acc = _BACKEND.traj_fused(pts, P, Q, Kd, cam, minmax, None, rewards, reward_index, boxes, ws, dense,
                                      prefilled, prior=prior, weight=weight, wsums=wsums)
        elif prior is None:
            acc = _BACKEND.traj_fused(pts, P, Q, Kd, cam, minmax, upstream, rewards, reward_index, boxes, ws, dense,
                                      prefilled)   # pass B
        else:
            acc = _BACKEND.traj_fused(pts, P, Q, Kd, cam, minmax, upstream, rewards, reward_index, boxes, ws, dense,
                                      prefilled, prior, prior_sum)
        _all_reduce_acc(acc, P.shape[0], group)
        if weight is not None:
            return _BACKEND.traj_epilogue(acc, minmax, Q, n_total, 0, den)
        return _BACKEND.traj_epilogue(acc, minmax, Q, n_total, 0 if upstream is None else 1)

    @staticmethod
    def backward(ctx, g_rewards, g_mean):
        pts, P, Q, Kd, minmax, out = ctx.saved_tensors
        W = P.shape[0]
        g_p = g_q = None
        if g_mean is not None:
            g_p = g_mean * out[1:1 + 3 * W]
            g_q = g_mean * out[1 + 3 * W:]
        if g_rewards is not None:
            up = _BACKEND.prepare(g_rewards, pts.device, "grad_rewards").reshape(-1)
            scratch = torch.empty(pts.shape[0], dtype=torch.float32, device=pts.device)
            # the rewards do not depend on the weight: the unweighted pass B with the upstream
            psum = ctx.prior_sum
            if ctx.prior is not None and psum is None:
                psum = _BACKEND.prior_sum(ctx.prior)
            o2 = CoverageTrajFn._run(pts, P, Q, Kd, ctx.cam, minmax, up, scratch, ctx.n_total, ctx.group,
                                     ctx.reward_index, ctx.boxes, None, ctx.dense, False, ctx.prior, psum)
            g_p = o2[1:1 + 3 * W] if g_p is None else g_p + o2[1:1 + 3 * W]
            g_q = o2[1 + 3 * W:] if g_q is None else g_q + o2[1 + 3 * W:]
        ps, qs = ctx.shapes
        return (None, None if g_p is None else g_p.reshape(ps), None if g_q is None else g_q.reshape(qs),
                None, None, None, None, None, None, None, None, None, None, None, None, None)


class CoverageSweepFn(torch.autograd.Function):
    """means_t = mean_j rewards_j(t) of T candidate trajectories on one cloud, each trajectory's poses evaluated as
    CoverageTrajFn evaluates them, and d means_t / d (poses_t, quats_t) from the same pass (cov_sweep_fused)."""

    @staticmethod
    def forward(ctx, pts, poses, quats, K, cam, n_total, group, boxes, shard, workspace, prior=None, prior_sum=None,
                weight=None, wsums=None, den=None):
        # weight / wsums / den (cloud's order): the checked point weight, cov_weight_sums of this rank's cloud and the
        # denominator sum_j w_j of the whole cloud (shard="points": all-reduced; "trajectories": this rank's own)
        B = _BACKEND
        dev = pts.device
        T, Pn = poses.shape[0], poses.shape[1]
        Kd = B.prepare(K, dev, "intrins").reshape(9)
        if group is not None and shard == "trajectories":
            # every rank holds the whole cloud and evaluates its contiguous block of trajectories; the per-rank outputs
            # [means | d/dposes | d/dquats] are gathered and reassembled in the layout of one unsharded call
            import torch.distributed as dist
            world, rank = dist.get_world_size(group), dist.get_rank(group)
            per = (T + world - 1) // world
            t0, t1 = min(T, rank * per), min(T, (rank + 1) * per)
            nt = t1 - t0
            mine = torch.zeros(per * (1 + 7 * Pn), dtype=torch.float32, device=dev)
            if nt > 0:
                o = CoverageSweepFn._run(pts, poses[t0:t1], quats[t0:t1], Kd, cam, n_total, None, boxes, workspace, prior,
                                         prior_sum, weight, wsums, den)
                mine[:nt] = o[:nt]
                mine[per:per + 3 * nt * Pn] = o[nt:nt + 3 * nt * Pn]
                mine[per + 3 * per * Pn:per + 3 * per * Pn + 4 * nt * Pn] = o[nt + 3 * nt * Pn:]
            every = torch.empty(world * mine.numel(), dtype=mine.dtype, device=dev)
            dist.all_gather_into_tensor(every, mine, group=group)
            every = every.view(world, -1)
            out = torch.cat([every[:, :per].reshape(-1)[:T], every[:, per:per + 3 * per * Pn].reshape(-1)[:3 * T * Pn],
                             every[:, per + 3 * per * Pn:].reshape(-1)[:4 * T * Pn]])
        else:
            out = CoverageSweepFn._run(pts, poses, quats, Kd, cam, n_total, group, boxes, workspace, prior, prior_sum,
                                       weight, wsums, den)
        ctx.shapes = (poses.shape, quats.shape)
        ctx.save_for_backward(out)
        return out[:T].clone()

    @staticmethod
    def _run(pts, poses, quats, Kd, cam, n_total, group, boxes, workspace, prior=None, prior_sum=None, weight=None,
             wsums=None, den=None):
        B = _BACKEND
        dev = pts.device
        T, Pn = poses.shape[0], poses.shape[1]
        P = B.prepare(poses, dev, "poses").reshape(-1, 3)
        Q = B.prepare(quats, dev, "quats").reshape(-1, 4)
        minmax = B.sweep_minmax(pts, P, Q, Kd, cam, boxes)     # pass A on this shard, (2, T Pn)
        _all_reduce_minmax(minmax, T * Pn, group)
        if weight is not None:
            acc = B.sweep_fused(pts, P, Q, T, Pn, Kd, cam, boxes, minmax, workspace, prior=prior, weight=weight,
                                wsums=wsums)
        elif prior is None:
            acc = B.sweep_fused(pts, P, Q, T, Pn, Kd, cam, boxes, minmax, workspace)
        else:
            acc = B.sweep_fused(pts, P, Q, T, Pn, Kd, cam, boxes, minmax, workspace, prior, prior_sum)
        if group is not None:
            # plain all-reduce: the in-kernel exchange buffers are sized for the 22 W + 1 doubles of one trajectory
            _all_reduce(acc, _reduce_ops()[2], group)
        if weight is not None:
            return B.sweep_epilogue(acc, minmax, Q, T, Pn, n_total, den)
        return B.sweep_epilogue(acc, minmax, Q, T, Pn, n_total)

    @staticmethod
    def backward(ctx, g_means):
        (out,) = ctx.saved_tensors
        ps, qs = ctx.shapes
        T, Pn = ps[0], ps[1]
        g = g_means.reshape(T, 1).to(out.dtype)
        g_p = (g * out[T:T + 3 * T * Pn].reshape(T, 3 * Pn)).reshape(ps)
        g_q = (g * out[T + 3 * T * Pn:].reshape(T, 4 * Pn)).reshape(qs)
        return None, g_p, g_q, None, None, None, None, None, None, None, None, None, None, None, None


class TrajRegularizersFn(torch.autograd.Function):
    """(l2, smooth, length) of ModelTraj.criterion (reference src/model.py:248-259) and their gradients w.r.t. the
    waypoints in one launch (cov_traj_regularizers)."""

    @staticmethod
    def forward(ctx, poses, poses0, smoothness_weight, traj_length_weight, eps):
        P = _dev_f32(poses, what="poses").reshape(-1, 3)
        P0 = _dev_f32(poses0, P.device, "poses0").reshape(-1, 3)
        W = P.shape[0]
        out = torch.empty(3 + 9 * W, dtype=torch.float32, device=P.device)
        _call("cov_traj_regularizers", P, _ptr(P), _ptr(P0), W, float(smoothness_weight), float(traj_length_weight),
                                                    float(eps), _ptr(out))
        ctx.save_for_backward(out)
        ctx.shape = poses.shape
        return out[:3].clone()

    @staticmethod
    def backward(ctx, g):
        (out,) = ctx.saved_tensors
        W = (out.numel() - 3) // 9
        grads = out[3:].reshape(3, W * 3)
        return (g.reshape(1, 3) @ grads).reshape(ctx.shape), None, None, None, None


def traj_regularizers(poses, poses0, smoothness_weight, traj_length_weight, eps=1e-6):
    """Returns a (3,) tensor (l2, smooth, length), differentiable w.r.t. `poses` ((W,3), W >= 3, CUDA)."""
    return TrajRegularizersFn.apply(poses, poses0, smoothness_weight, traj_length_weight, eps)


def coverage_pose(points, trans, quat, intrins, img_width, img_height, min_dist=1.0, max_dist=5.0, eps=1e-6,
                  weight=None, group=None):
    """Fused ModelPose objective.  Returns (observations (N,), total = sum(observations));
    differentiable w.r.t. trans (.., 3) and quat (.., 4) (w, x, y, z)."""
    cam = _lib.camera(img_width, img_height, min_dist, max_dist, eps)
    return CoveragePoseFn.apply(points, trans, quat, intrins, cam, weight, group)


def coverage_pose_batch(points, trans, quats, intrins, img_width, img_height, min_dist=1.0, max_dist=5.0, eps=1e-6,
                        weight=None, group=None, boxes=None, presorted=False, workspace=None):
    """The ModelPose objective of K candidate poses on one cloud: trans (K, 3), quats (K, 4) -> totals (K,) fp32, where
    totals[k] is the total `coverage_pose(points, trans[k], quats[k], weight=weight)` returns.  `totals` is differentiable
    w.r.t. `trans` and `quats`; all K totals and their gradients come from one pass over the cloud (cov_pose_batch_fused),
    so a backward of any weighted sum of the totals costs no further pass.
    The cloud is Morton-ordered first (no per-point output exists, so the order is free) unless `presorted` or `boxes`
    are given; `weight` (N,) is in the order of `points` as passed.  Callers that evaluate the same cloud repeatedly order
    it once (`spatial_sort`, `tile_boxes`), permute their weight with the same permutation and pass `presorted=True`
    and the boxes.  The boxes let the kernel skip (128-point box, pose) pairs that are exactly zero: that pays on clouds
    much larger than the ~27 m reach of the default clip limits.  Dense mode comes from `evaluation(dense=True)`.
    `group`: `points` (and `weight`) are THIS RANK'S slice of the cloud; the K x 8 sums are all-reduced.  No host
    synchronisation: capturable in a CUDA graph.  `workspace`: a uint8 CUDA tensor kept by the caller across calls."""
    B = _BACKEND
    if (not isinstance(trans, torch.Tensor) or not isinstance(quats, torch.Tensor) or trans.dim() != 2
            or quats.dim() != 2 or trans.shape[1] != 3 or quats.shape[1] != 4 or trans.shape[0] != quats.shape[0]
            or trans.shape[0] == 0):
        raise ValueError("coverage_pose_batch: trans must be (K, 3) and quats (K, 4) with the same K >= 1; got "
                         f"{tuple(getattr(trans, 'shape', ()))} and {tuple(getattr(quats, 'shape', ()))}")
    pts = B.prepare(points, what="points")
    dev = pts.device
    w = None if weight is None else B.prepare(weight, dev, "weight").reshape(-1)
    if w is not None and w.shape[0] != pts.shape[0]:
        raise ValueError(f"coverage_pose_batch: weight has {w.shape[0]} entries for {pts.shape[0]} points")
    if not presorted and boxes is None and pts.shape[0] > 0:
        pts, perm, boxes = B.order_cloud(pts, True)
        if w is not None and perm is not None:
            w = B.prepare(w.index_select(0, perm.long()), dev, "weight")   # weight[j] belongs to point perm[j]
    cam = _lib.camera(img_width, img_height, min_dist, max_dist, eps)
    return CoveragePoseBatchFn.apply(pts, trans, quats, intrins, cam, w, group, boxes, workspace)


def coverage_traj(points, poses, quats, intrins, img_width, img_height, min_dist=1.0, max_dist=5.0, eps=1e-6,
                  n_total=None, group=None, reward_index=None, boxes=None, dense=None, workspace=None,
                  prior_logodds=None, weight=None):
    """Fused ModelTraj visibility term over the W poses given.  Returns (rewards (N,), mean(rewards)).
    `reward_index` (int32, from `spatial_sort`): `points` is a reordered copy of the caller's cloud and
    rewards come back in the caller's order.  `boxes` (from `tile_boxes(points)`): built once per cloud so the
    pruned kernels do not rebuild them on every call.  `dense=True`: evaluate every pair (no pruning; what an unordered
    cloud should ask for).  `workspace`: a uint8 CUDA tensor kept by the caller across calls (one per cloud).
    `prior_logodds` (N,) fp32: what earlier paths observed (map memory, e.g. `traj_logodds` of an executed path);
    rewards_j = sigmoid(prior_j + sum_w lo_jw), indexed like the rewards (the caller's order when `reward_index` is
    given).  With a `group` it is this rank's slice.  None = an empty map (exactly the rewards of a zero prior).
    `weight` (N,) fp32, finite and >= 0 with a positive sum (not checked: no host synchronisation): per-point importance,
    indexed like the rewards.  The mean is then sum_j w_j r_j / sum_j w_j (its gradient from the same pass); the rewards
    are unchanged.  With a `group` it is this rank's slice (the denominator is all-reduced); `n_total` is not used."""
    cam = _lib.camera(img_width, img_height, min_dist, max_dist, eps)
    prior = psum = w = wsums = den = None
    if prior_logodds is not None or weight is not None:
        pts = _BACKEND.prepare(points, what="points")
        prior = _check_prior(prior_logodds, pts.shape[0], pts.device)
        w = _check_weight(weight, pts.shape[0], pts.device)
        if w is not None:
            wsums, den = _weight_sums(_BACKEND, w, prior, group)
        elif prior is not None:
            psum = _BACKEND.prior_sum(prior)
    return CoverageTrajFn.apply(points, poses, quats, intrins, cam, n_total, group, reward_index, boxes, dense, workspace,
                                prior, psum, w, wsums, den)


@torch.no_grad()
def traj_logodds(points, poses, quats, intrins, img_width, img_height, min_dist=1.0, max_dist=5.0, eps=1e-6,
                 prior_logodds=None, reward_index=None, boxes=None, group=None, dense=None, workspace=None):
    """The fused log-odds prior_j + sum_w lo_jw of the W poses given, (N,) fp32 in the caller's order (as `rewards` of
    `coverage_traj`), without gradients: sigmoid of it is `coverage_traj(..., prior_logodds=prior_logodds)`'s rewards,
    bit for bit.  Folding an executed path into the map is `prior = traj_logodds(..., prior_logodds=prior)`; clamping
    (OctoMap's thresholds) is the caller's, in torch.  Arguments as for `coverage_traj`; with a `group`, `points` and
    `prior_logodds` are this rank's slices (the normalisers are all-reduced) and so is the result."""
    B = _BACKEND
    pts = B.prepare(points, what="points")
    dev, n = pts.device, pts.shape[0]
    if reward_index is not None and (reward_index.dtype != torch.int32 or reward_index.shape[0] != n
                                     or reward_index.device != dev or not reward_index.is_contiguous()):
        raise ValueError("reward_index must be a contiguous int32 tensor with one entry per point, on the cloud's device")
    prior = _check_prior(prior_logodds, n, dev)
    P = B.prepare(poses, dev, "poses").reshape(-1, 3)
    Q = B.prepare(quats, dev, "quats").reshape(-1, 4)
    Kd = B.prepare(intrins, dev, "intrins").reshape(9)
    W = P.shape[0]
    if Q.shape[0] != W:
        raise ValueError("poses and quats disagree on the number of waypoints")
    cam = _lib.camera(img_width, img_height, min_dist, max_dist, eps)
    dense = _MODE.dense if dense is None else bool(dense)
    ws = workspace
    if ws is None or ws.numel() < B.traj_workspace_bytes(pts, W) or ws.device != dev:
        ws = B.traj_workspace(pts, W)
    long = _takes_long_path(W, dense)
    minmax = B.sweep_minmax(pts, P, Q, Kd, cam, boxes, ws, dense) if long else B.traj_minmax(pts, P, Q, Kd, cam, boxes,
                                                                                           ws, dense)
    _all_reduce_minmax(minmax, W, group)
    out = torch.zeros(n, dtype=torch.float32, device=dev) if prior is None else prior.clone()
    if long:
        return B.traj_logodds_long(pts, P, Q, Kd, cam, minmax, out, reward_index, boxes, ws)
    return B.traj_logodds(pts, P, Q, Kd, cam, minmax, out, reward_index, boxes, ws, dense)


@torch.no_grad()
def tile_boxes(points):
    """Bounding boxes of runs of 128 consecutive points (include/coverage_b200.h: cov_tile_boxes), (nb, 8) fp32."""
    L = _lib.lib()
    pts = _dev_f32(points, what="points")
    n = pts.shape[0]
    boxes = torch.empty(max(int(L.cov_tile_boxes_count(n)), 1), 8, dtype=torch.float32, device=pts.device)
    if n > 0:
        _call("cov_tile_boxes", pts, _ptr(pts), n, _ptr(boxes))
    return boxes


@torch.no_grad()
def spatial_sort(points):
    """Morton-order copy of a cloud, made once per cloud (see include/coverage_b200.h: cov_spatial_sort).
    Returns (sorted (N,3) fp32, perm (N,) int32) with sorted[j] = points[perm[j]]."""
    L = _lib.lib()
    pts = _dev_f32(points, what="points")
    n = pts.shape[0]
    out = torch.empty_like(pts)
    perm = torch.empty(n, dtype=torch.int32, device=pts.device)
    if n == 0:
        return out, perm
    ws_bytes = L.cov_spatial_sort_workspace_bytes(n)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=pts.device)
    _call("cov_spatial_sort", pts, _ptr(pts), n, _ptr(out), _ptr(perm), _ptr(ws), ws_bytes)
    return out, perm


@torch.no_grad()
def sort_pairs(keys, vals, begin_bit=0, end_bit=32):
    """Stable radix sort of (keys int32/uint32 bit patterns, vals int32) CUDA tensors by key bits [begin_bit, end_bit)
    (include/coverage_b200.h: cov_sort_pairs); returns sorted copies.  Keys compare as UNSIGNED 32-bit values."""
    L = _lib.lib()
    if not (keys.is_cuda and vals.is_cuda and keys.dtype == torch.int32 and vals.dtype == torch.int32 and keys.shape == vals.shape
            and keys.dim() == 1):
        raise RuntimeError("sort_pairs: keys and vals must be 1-D int32 CUDA tensors of equal length")
    k, v = keys.clone(), vals.clone()
    n = k.shape[0]
    if n == 0:
        return k, v
    ws_bytes = L.cov_sort_pairs_workspace_bytes(n)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=k.device)
    _call("cov_sort_pairs", k, _ptr(k), _ptr(v), n, int(begin_bit), int(end_bit), _ptr(ws), ws_bytes)
    return k, v


def _order_with_prior(B, pts, prior, boxes, presorted, weight=None):
    """The sweeps' cloud ordering (Morton order unless `presorted` or `boxes`), the prior and the weight permuted with
    the cloud."""
    if not presorted and boxes is None and pts.shape[0] > 0:
        pts, perm, boxes = B.order_cloud(pts, True)
        if perm is not None:
            if prior is not None:   # prior[j] of point perm[j]
                prior = _check_prior(prior.index_select(0, perm.long()), pts.shape[0], pts.device)
            if weight is not None:
                weight = _check_weight(weight.index_select(0, perm.long()), pts.shape[0], pts.device)
    return pts, prior, boxes, weight


def _sweep_sums(B, pts, P, Q, T, Pn, Kd, cam, boxes, minmax, prior, psum, w=None, wsums=None):
    if w is not None:
        return B.sweep_sums(pts, P, Q, T, Pn, Kd, cam, boxes, minmax, prior=prior, weight=w, wsums=wsums)
    if prior is None:
        return B.sweep_sums(pts, P, Q, T, Pn, Kd, cam, boxes, minmax)
    return B.sweep_sums(pts, P, Q, T, Pn, Kd, cam, boxes, minmax, prior, psum)


def _prefix_sums(B, pts, P, Q, T, Pn, Kd, cam, boxes, minmax, prior, psum, w=None, wsums=None):
    return B.sweep_prefix_sums(pts, P, Q, T, Pn, Kd, cam, boxes, minmax, prior=prior,
                               base=psum if w is None else wsums, weight=w)


def _sweep_forward(sums, k, points, poses, quats, intrins, cam, n_total, group, boxes, presorted, shard, prior_logodds,
                   weight):
    """The forward-only sweeps around one backend sum `sums` (`_sweep_sums`, `_prefix_sums`) that gives k fp64 values
    per trajectory: the cloud ordered, the prior and the weight checked and permuted with it, their sums, then
    `_sweep_run`."""
    B = _BACKEND
    if shard not in ("points", "trajectories"):
        raise ValueError("shard must be 'points' or 'trajectories'")
    pts = B.prepare(points, what="points")
    prior = _check_prior(prior_logodds, pts.shape[0], pts.device)
    w = _check_weight(weight, pts.shape[0], pts.device)
    pts, prior, boxes, w = _order_with_prior(B, pts, prior, boxes, presorted, w)
    psum = wsums = den = None
    if w is not None:
        wsums, den = _weight_sums(B, w, prior, group if shard == "points" else None)
    elif prior is not None:
        psum = B.prior_sum(prior)
    return _sweep_run(sums, k, pts, poses, quats, intrins, cam, n_total, group, boxes, shard, prior, psum, w, wsums, den)


def _sweep_run(sums, k, pts, poses, quats, intrins, cam, n_total, group, boxes, shard, prior, psum, w, wsums, den):
    """(T k,) fp64 means of the ordered cloud `pts` with its prior, weight and their sums: pass A, `sums`, the
    collectives of `shard` and the division by the point count or the weighted denominator `den`."""
    B = _BACKEND
    dev = pts.device
    T, Pn = poses.shape[0], poses.shape[1]
    n = pts.shape[0]
    Kd = B.prepare(intrins, dev, "intrins").reshape(9)
    if group is not None and shard == "trajectories":
        import torch.distributed as dist
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        per = (T + world - 1) // world
        t0, t1 = min(T, rank * per), min(T, (rank + 1) * per)
        mine = torch.zeros(per * k, dtype=torch.float64, device=dev)
        if t1 > t0:
            P = B.prepare(poses[t0:t1], dev, "poses").reshape(-1, 3)
            Q = B.prepare(quats[t0:t1], dev, "quats").reshape(-1, 4)
            minmax = B.sweep_minmax(pts, P, Q, Kd, cam, boxes)
            mine[:(t1 - t0) * k] = sums(B, pts, P, Q, t1 - t0, Pn, Kd, cam, boxes, minmax, prior, psum, w, wsums)
        out = torch.empty(world * per * k, dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(out, mine, group=group)
        return out[:T * k] / (float(n) if w is None else den)
    P = B.prepare(poses, dev, "poses").reshape(-1, 3)
    Q = B.prepare(quats, dev, "quats").reshape(-1, 4)
    minmax = B.sweep_minmax(pts, P, Q, Kd, cam, boxes)
    _all_reduce_minmax(minmax, T * Pn, group)
    out = sums(B, pts, P, Q, T, Pn, Kd, cam, boxes, minmax, prior, psum, w, wsums)
    if group is not None:
        _all_reduce(out, _reduce_ops()[2], group)
    if w is not None:
        return out / den
    return out / float(n if n_total is None else n_total)


@torch.no_grad()
def sweep_rewards(points, poses, quats, intrins, img_width, img_height, min_dist=1.0, max_dist=5.0, eps=1e-6,
                  n_total=None, group=None, boxes=None, presorted=False, shard="points", prior_logodds=None,
                  weight=None):
    """Forward-only mean reward of many candidate trajectories: poses (T, P, 3), quats (T, P, 4) -> (T,) fp64
    (semantics: ModelTraj.forward per trajectory with every pose evaluated, reference src/model.py:217-237).
    The cloud is Morton-ordered first (no per-point output exists, so the order is free) unless `presorted`;
    callers that sweep the same cloud repeatedly order it once (`spatial_sort`, `tile_boxes`) and pass both.

    With a `group` (one process per GPU) there are two ways to split the work (SURVEY.md 8e):
      shard="points"        `points` is THIS RANK'S slice of the cloud; the per-pose normalisers are all-reduced (MAX of
                            2 T P floats) and the per-trajectory sums are all-reduced (SUM of T doubles);
      shard="trajectories"  every rank holds the WHOLE cloud (it fits: 50 M points = 600 MB) and evaluates its own
                            contiguous block of T / world trajectories — no collective on the data path, one all-gather
                            of T doubles at the end.  The choice when the cloud fits one GPU.

    `prior_logodds` (N,) fp32: per-point prior log-odds (map memory), shared by every trajectory: each trajectory's
    rewards are sigmoid(prior_j + sum_w lo_jw).  In the order of `points` as passed (permuted with the cloud when the
    call orders it; with `presorted`, already in the cloud's order); shard="points": this rank's slice,
    shard="trajectories": the whole prior on every rank.
    `weight` (N,) fp32, finite and >= 0 with a positive sum (not checked): per-point importance shared by every
    trajectory; each result is then sum_j w_j r_j(t) / sum_j w_j.  Ordered and sharded like `prior_logodds` (with
    shard="points" the denominator is all-reduced); `n_total` is not used."""
    cam = _lib.camera(img_width, img_height, min_dist, max_dist, eps)
    return _sweep_forward(_sweep_sums, 1, points, poses, quats, intrins, cam, n_total, group, boxes, presorted, shard,
                          prior_logodds, weight)


@torch.no_grad()
def sweep_prefix_rewards(points, poses, quats, intrins, img_width, img_height, min_dist=1.0, max_dist=5.0, eps=1e-6,
                         n_total=None, group=None, boxes=None, presorted=False, shard="points", prior_logodds=None,
                         weight=None):
    """The mean reward of every prefix of every candidate trajectory: poses (T, P, 3), quats (T, P, 4) -> (T, P) fp64,
    where [t, i] is what `sweep_rewards(points, poses[:, :i+1], quats[:, :i+1], ...)` returns for trajectory t, with the
    same prior and weight, up to the order of fp64 additions; [:, P-1] is `sweep_rewards`'s result.  One pass over the
    cloud per chunk of poses, as `sweep_rewards` (cov_sweep_prefix_rewards), in place of P sweeps.
    Rows are non-decreasing (up to the fp32 rounding of single terms).  Uses: how far along a candidate to commit
    (receding horizon), gain per path cost at every node of a branch, and candidates of different lengths: pad each to P
    (e.g. by repeating its last pose) and read column len_t - 1.  With a multi-camera rig (pose index body * n_cams +
    cam, `multicam`) the prefix after waypoint k is column (k + 1) * n_cams - 1.  A pose that sees nothing has 0/0
    normalisers: its prefix and every later one of its trajectory are NaN, as the truncated sweeps are.
    Arguments, ordering, prior, weight and sharding as for `sweep_rewards` (shard="points": the T P sums are
    all-reduced; "trajectories": the rank blocks are all-gathered).  Without gradients."""
    if (not isinstance(poses, torch.Tensor) or not isinstance(quats, torch.Tensor) or poses.dim() != 3
            or quats.dim() != 3 or poses.shape[2] != 3 or quats.shape[2] != 4 or poses.shape[:2] != quats.shape[:2]
            or poses.shape[0] == 0 or poses.shape[1] == 0):
        raise ValueError("sweep_prefix_rewards: poses must be (T, P, 3) and quats (T, P, 4) with the same T, P >= 1; got "
                         f"{tuple(getattr(poses, 'shape', ()))} and {tuple(getattr(quats, 'shape', ()))}")
    T, Pn = poses.shape[0], poses.shape[1]
    cam = _lib.camera(img_width, img_height, min_dist, max_dist, eps)
    return _sweep_forward(_prefix_sums, Pn, points, poses, quats, intrins, cam, n_total, group, boxes, presorted, shard,
                          prior_logodds, weight).reshape(T, Pn)


def coverage_sweep(points, poses, quats, intrins, img_width, img_height, min_dist=1.0, max_dist=5.0, eps=1e-6,
                   n_total=None, group=None, boxes=None, presorted=False, shard="points", workspace=None,
                   prior_logodds=None, weight=None):
    """Differentiable candidate sweep: poses (T, P, 3), quats (T, P, 4) -> means (T,) fp32, where means[t] is the mean
    reward of trajectory t as `coverage_traj(points, poses[t], quats[t])` computes it.  `means` is differentiable w.r.t.
    `poses` and `quats`; each trajectory's gradient comes from the same pass over the cloud (cov_sweep_fused), so a
    backward of any weighted sum of the means costs no further pass.
    The cloud is ordered as in `sweep_rewards` (Morton order, unless `presorted` or `boxes` are given); dense mode comes
    from `evaluation(dense=True)`.  No host synchronisation: capturable in a CUDA graph.  `workspace`: a uint8 CUDA tensor
    kept by the caller across calls (grown when too small).
    Sharding as in `sweep_rewards`: shard="points" (this rank's slice of the cloud; normalisers and accumulators are
    all-reduced) or shard="trajectories" (the whole cloud on every rank; means and gradients are all-gathered).
    `prior_logodds`: per-point prior log-odds shared by every trajectory, ordered and sharded as in `sweep_rewards`.
    `weight`: per-point importance as in `sweep_rewards`: means[t] = sum_j w_j r_j(t) / sum_j w_j and its gradient."""
    B = _BACKEND
    if shard not in ("points", "trajectories"):
        raise ValueError("shard must be 'points' or 'trajectories'")
    if (not isinstance(poses, torch.Tensor) or not isinstance(quats, torch.Tensor) or poses.dim() != 3
            or quats.dim() != 3 or poses.shape[2] != 3 or quats.shape[2] != 4 or poses.shape[:2] != quats.shape[:2]
            or poses.shape[0] == 0 or poses.shape[1] == 0):
        raise ValueError("coverage_sweep: poses must be (T, P, 3) and quats (T, P, 4) with the same T, P >= 1; got "
                         f"{tuple(getattr(poses, 'shape', ()))} and {tuple(getattr(quats, 'shape', ()))}")
    pts = B.prepare(points, what="points")
    prior = _check_prior(prior_logodds, pts.shape[0], pts.device)
    w = _check_weight(weight, pts.shape[0], pts.device)
    pts, prior, boxes, w = _order_with_prior(B, pts, prior, boxes, presorted, w)
    psum = wsums = den = None
    if w is not None:
        wsums, den = _weight_sums(B, w, prior, group if shard == "points" else None)
    elif prior is not None:
        psum = B.prior_sum(prior)
    n_total = int(pts.shape[0] if n_total is None else n_total)
    cam = _lib.camera(img_width, img_height, min_dist, max_dist, eps)
    return CoverageSweepFn.apply(pts, poses, quats, intrins, cam, n_total, group, boxes, shard, workspace, prior, psum, w,
                                 wsums, den)


@torch.no_grad()
def frustum_cull(points_nx3, intrins, img_width, img_height, min_dist=1.0, max_dist=10.0):
    """Binary frustum test + ordered compaction (reference src/tools.py:176-187).
    Returns (idx int64 (M,), dist_mask bool (N,), fov_mask bool (N,))."""
    L = _lib.lib()
    pts = _dev_f32(points_nx3, what="points")
    dev = pts.device
    Kd = _dev_f32(intrins, dev, "intrins")[:3, :3].contiguous().reshape(9)
    n = pts.shape[0]
    dm = torch.empty(n, dtype=torch.uint8, device=dev)
    fm = torch.empty(n, dtype=torch.uint8, device=dev)
    idx = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
    cnt = torch.zeros(1, dtype=torch.int64, device=dev)
    ws_bytes = L.cov_cull_workspace_bytes(n)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    _call("cov_frustum_cull", pts, _ptr(pts), n, _ptr(Kd), float(img_width), float(img_height), float(min_dist),
                                  float(max_dist), _ptr(dm), _ptr(fm), _ptr(idx), _ptr(cnt), _ptr(ws), ws_bytes)
    m = int(cnt.item())
    return idx[:m].long(), dm.view(torch.bool), fm.view(torch.bool)   # the masks hold 0/1 bytes: zero-copy views


@torch.no_grad()
def spherical_flip(points, param):
    """Bit-exact fp32 spherical flip (reference src/tools.py:38-53). Returns (flipped (N,3), radius 0-dim)."""
    L = _lib.lib()
    pts = _dev_f32(points, what="points")
    n = pts.shape[0]
    out = torch.empty_like(pts)
    rad = torch.empty(2, dtype=torch.float32, device=pts.device)
    _call("cov_hpr_flip", pts, _ptr(pts), n, float(10.0 ** param), _ptr(out), _ptr(rad))
    return out, rad[0]


@torch.no_grad()
def hpr_hull_mask(flipped, return_info=False):
    """Vertex mask of conv(flipped U {origin}) (reference src/tools.py:56-64 + the vertex set of :79).
    Returns (mask uint8 (N,), origin_is_vertex bool, n_exact_fallback int) [+ the raw 4-int info when `return_info`]."""
    L = _lib.lib()
    f = _dev_f32(flipped, what="flipped points")
    n = f.shape[0]
    mask = torch.empty(n, dtype=torch.uint8, device=f.device)
    info = torch.zeros(4, dtype=torch.int32, device=f.device)
    ws_bytes = L.cov_hpr_hull_workspace_bytes(n)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=f.device)
    _call("cov_hpr_hull", f, _ptr(f), n, _ptr(mask), _ptr(info), _ptr(ws), ws_bytes)
    info_h = info.tolist()
    if return_info:
        return mask, bool(info_h[0]), int(info_h[1]), info_h
    return mask, bool(info_h[0]), int(info_h[1])
