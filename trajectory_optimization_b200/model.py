"""Drop-in for the reference's `src/model.py`: same names, signatures, attributes and asserts,
with the N-sized arithmetic replaced by the fused sm_100a kernels in libcovb200.so.

Reference citations are relative to the reference repository root.  The callers
(`src/pose_optimization.py:82-137`, `src/trajectory_optimization.py:83-127`) construct the
models, put `.trans/.quat` (or `.poses/.quats`) in Adam parameter groups, call `model()`,
`loss.backward()`, and read `.observations` / `.rewards` / `.loss[...]` — all of that works
unchanged.  The helper functions operate on CUDA tensors only (no CPU fallback).
"""
from copy import deepcopy
from time import time

import torch
import torch.nn as nn

from . import ops
from .tools import hidden_pts_removal, load_intrinsics  # noqa: F401  (re-exported like the reference does)


# ------------------------------------------------------------------------------------------
# helper functions (src/model.py:13-57)
# ------------------------------------------------------------------------------------------
def _unit_pose(like):
    t = torch.zeros(1, 3, device=like.device)
    q = torch.tensor([[1.0, 0.0, 0.0, 0.0]], device=like.device)
    return t, q


def to_camera_frame(verts, quat, trans):
    """src/model.py:50-57.  R(q)^T (v - t) with q = normalize(quat); small differentiable torch
    helper kept for API parity (the fused ops do this in-kernel)."""
    assert verts.dim() == trans.dim()
    assert quat.size() == torch.Size([1, 4])
    q = torch.nn.functional.normalize(quat)
    w, x, y, z = q[0, 0], q[0, 1], q[0, 2], q[0, 3]
    R = torch.stack([
        torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)]),
        torch.stack([2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)]),
        torch.stack([2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]),
    ]).to(verts.dtype)
    return (verts - trans) @ R


def get_dist_mask(points, min_dist=1.0, max_dist=5.0):
    """src/model.py:13-24: Gaussian about the camera-frame point (mu, mu, mu)."""
    assert isinstance(points, torch.Tensor)
    assert points.size()[1] == 3
    mean = (min_dist + max_dist) / 2.0
    std = (max_dist - min_dist) / 2.0
    sq = ((points - mean) ** 2).sum(dim=1)
    return torch.exp(-0.5 * sq / (std * std))


def get_fov_mask(points, img_height, img_width, intrins, eps=1e-6, binary=False):
    """src/model.py:27-47.  `binary=True` runs the bit-exact CUDA cull test; the smooth branch is a
    small differentiable torch helper kept for API parity (the fused ops do this in-kernel)."""
    assert isinstance(points, torch.Tensor)
    assert points.size()[1] == 3
    assert isinstance(intrins, torch.Tensor)
    assert intrins.size() == torch.Size([3, 3])
    if binary:
        _, _, fov = ops.frustum_cull(points, intrins, img_width, img_height, min_dist=float("-inf"),
                                     max_dist=float("inf"))
        return fov
    h = points @ intrins.t().to(points.dtype)
    z = h[:, 2]
    u = h[:, 0] / (z + eps)
    v = h[:, 1] / (z + eps)
    return (torch.sigmoid(z) * torch.exp(-0.5 * ((u - img_width / 2.0) / img_width) ** 2)
            * torch.exp(-0.5 * ((v - img_height / 2.0) / img_height) ** 2))


# ------------------------------------------------------------------------------------------
# single pose (src/model.py:65-127)
# ------------------------------------------------------------------------------------------
class ModelPose(nn.Module):
    def __init__(self, points, trans0, q0, intrins, img_width, img_height, min_dist=1.0, max_dist=5.0,
                 device=torch.device("cuda:0"), group=None):
        super().__init__()
        assert trans0.size() == torch.Size([1, 3])
        assert q0.size() == torch.Size([1, 4])
        assert intrins.size() == torch.Size([3, 3])

        self.device = device
        self.points = points.to(self.device)
        self.rewards = None
        self.observations = None
        self.lo_sum = 0.0
        self.trans = nn.Parameter(torch.as_tensor(trans0, dtype=torch.float32).to(self.device))
        self.quat = nn.Parameter(torch.as_tensor(q0, dtype=torch.float32).to(self.device))
        self.K = torch.as_tensor(intrins, dtype=torch.float32).to(self.device)
        self.img_width, self.img_height = float(img_width), float(img_height)
        self.eps = 1e-6
        self.pc_clip_limits = [min_dist, max_dist]
        self.group = group            # torch.distributed group when `points` is this rank's shard
        self._total = None
        self._pts32 = None
        self.to(self.device)

    def _cloud(self):
        # fp32, contiguous, aligned copy made once per cloud (the reference keeps whatever dtype it was given); the
        # cache follows `self.points` by identity AND by torch's version counter, so an in-place edit is seen too
        key = (id(self.points), self.points._version)
        if self._pts32 is None or self._pts32_key != key:
            self._pts32 = ops._BACKEND.prepare(self.points, what="points")
            self._pts32_key = key
        return self._pts32

    def set_points(self, points):
        """Replace the cloud (same as assigning `model.points`; the fp32 working copy is rebuilt on the next forward)."""
        self.points = points.to(self.device)
        self._pts32 = None

    def detach_state(self):
        """Drop the references this model keeps into the last autograd graph (`_total`) so that the graph — and the
        gradient-accumulation nodes bound to the stream it ran on — can be freed (graphs.GraphedStep calls this before
        it warms up on its capture stream)."""
        self._total = None
        if self.observations is not None:
            self.observations = self.observations.detach()

    def forward(self, debug=False, hpr=False):
        t0 = time()
        weight = None
        if hpr:  # src/model.py:112-115 — HPR of the untransformed cloud, mask multiplies the observations
            weight = hidden_pts_removal(self.points.detach(), device=self.device)[1]
        obs, total = ops.coverage_pose(self._cloud(), self.trans, self.quat, self.K, self.img_width, self.img_height,
                                       self.pc_clip_limits[0], self.pc_clip_limits[1], self.eps, weight=weight,
                                       group=self.group)
        self.observations = obs
        self._total = total
        if debug:
            if obs.is_cuda:
                torch.cuda.synchronize(obs.device)
            print(f"\nFused transformation + visibility estimation took: {1000 * (time() - t0)} msec")
            print(f"Point cloud size {self.points.size()}")
        return self.criterion(self.observations)

    def criterion(self, observations):
        # 1 / (sum + eps); the sum of the tensor produced by forward() was already reduced in-kernel
        if observations is self.observations and self._total is not None:
            total = self._total
        else:
            total = torch.sum(observations)
        return 1.0 / (total + self.eps)


# ------------------------------------------------------------------------------------------
# trajectory (src/model.py:135-260)
# ------------------------------------------------------------------------------------------
def length_calc(traj):
    """src/model.py:135-139 — sum of segment lengths (vectorised, same arithmetic per segment)."""
    if len(traj) < 2:
        return 0.0
    return torch.linalg.norm(traj[1:] - traj[:-1], dim=-1).sum()


def mean_angle_calc(traj_wps, eps=1e-6):
    """src/model.py:142-155 — mean interior angle at the waypoints."""
    n_wps = len(traj_wps)
    traj = torch.as_tensor(traj_wps).reshape(n_wps, -1)
    if n_wps <= 2:
        return 0.0 / (n_wps - 2)  # ZeroDivisionError for 2 waypoints, 0.0/-1 for one: as the reference
    ab = traj[:-2] - traj[1:-1]
    ac = traj[2:] - traj[1:-1]
    cosang = (ab * ac).sum(dim=1) / (torch.linalg.norm(ab, dim=1) * torch.linalg.norm(ac, dim=1) + eps)
    return torch.arccos(cosang).sum() / (n_wps - 2)


def _wps_quotient(poses0, vis_wps_dist):
    """src/model.py:214: vis_wps_dist over the mean waypoint spacing of (W, 3) `poses0`, as a 0-d tensor of poses0's
    dtype (the reference divides by an fp32 tensor: when the spacing divides the distance, the rounded quotient can land
    on the integer that an fp64 division would miss, and the stride int(quotient) + 1 depends on it)."""
    mean_wps_dist = (poses0[1:, :] - poses0[:-1, :]).norm(dim=1).mean()
    return vis_wps_dist / mean_wps_dist


class _OrderedCloudModel(nn.Module):
    """What ModelTraj, ModelTrajBatch and ModelPoseBatch share: the Morton-ordered copy of `self.points` with its permutation and tile
    boxes (made once per state of the cloud), the kept workspace, and the release of the last autograd graph.
    Subclasses set `points`, `spatial_sort`, `_pts32`, `_perm`, `_boxes`, `_ws` and `_mean` in their constructor.
    ModelTraj and ModelTrajBatch also keep the prior log-odds (`_init_prior`) and the point weight (`_init_weight`)."""

    _prior_in_cloud_order = False   # the kernels read the prior and the weight in the cloud's (Morton) order, not in that of `points`

    def _init_prior(self, prior_logodds):
        # The kernels read the model's own copy of the prior (`_prior`, in the order they index it) and sum_j sigmoid(
        # prior_j) on the device (`_prior_sum`).  Like the cloud cache, both belong to ONE state of `prior_logodds`: keyed
        # on identity and torch's version counter, rebuilt on the next forward when either changes.
        self.prior_logodds = None if prior_logodds is None else torch.as_tensor(prior_logodds).to(self.device)
        self._prior = None
        self._prior_sum = None
        self._prior_key = None

    def _prior_state_key(self):
        p = self.prior_logodds
        return (id(p), p._version, id(self.points), self.points._version)

    @torch.no_grad()
    def _write_prior(self):
        # into the same buffers when the shape allows (captured CUDA graphs hold their addresses)
        pts = self._cloud()
        q = ops._check_prior(self.prior_logodds, pts.shape[0], pts.device)
        if not bool(torch.isfinite(q).all()):   # once per prior state (one host synchronisation)
            raise ValueError("prior_logodds must be finite (clamp it, OctoMap-style, before handing it to the model)")
        if self._prior_in_cloud_order and self._perm is not None:
            q = q.index_select(0, self._perm.long())
        if self._prior is None or self._prior.shape != q.shape or self._prior.device != q.device:
            self._prior = torch.empty_like(q)
            self._prior_sum = torch.empty(1, dtype=torch.float64, device=q.device)
        self._prior.copy_(q)
        self._prior_sum.copy_(ops._BACKEND.prior_sum(self._prior))
        self._prior_key = self._prior_state_key()

    def _prior_args(self):
        """(prior as the kernels index it, sum_j sigmoid(prior_j) (1,) fp64), or (None, None) without a prior."""
        if self.prior_logodds is None:
            return None, None
        if self._prior is None or self._prior_key != self._prior_state_key():
            self._write_prior()
        return self._prior, self._prior_sum

    def set_prior_logodds(self, prior_logodds):
        """Replace the prior log-odds (None: an empty map), (N,) fp32 in the order of `self.points`.  The model's copies
        are rewritten now, at the same addresses when the shape is unchanged, so a CUDA graph captured WITH a prior
        evaluates the new one on its next replay (a graph captured without a prior needs a new capture)."""
        self.prior_logodds = None if prior_logodds is None else prior_logodds.to(self.device)
        if self.prior_logodds is not None and self._prior is not None:
            self._write_prior()
        if getattr(self, "point_weight", None) is not None and self._weight is not None:
            self._write_weight()   # its reward-sum base is sum_j w_j sigmoid(prior_j)

    def _init_weight(self, point_weight):
        # Like the prior: the kernels read the model's copy (`_weight`, in the order they index it), this shard's
        # cov_weight_sums (`_weight_sums`, whose base depends on the prior) and sum_j w_j over every rank (`_weight_den`),
        # all belonging to ONE state of `point_weight`, of the cloud and of the prior.
        self.point_weight = None if point_weight is None else torch.as_tensor(point_weight).to(self.device)
        self._weight = None
        self._weight_sums = None
        self._weight_den = None
        self._weight_key = None

    def _weight_state_key(self):
        w, p = self.point_weight, self.prior_logodds
        return (id(w), w._version, id(self.points), self.points._version, None if p is None else (id(p), p._version))

    @torch.no_grad()
    def _write_weight(self):
        # into the same buffers when the shape allows (captured CUDA graphs hold their addresses)
        pts = self._cloud()
        w = ops._check_weight(self.point_weight, pts.shape[0], pts.device, what="point_weight")
        if bool((~torch.isfinite(w) | (w < 0)).any()):   # once per weight state (one host synchronisation)
            raise ValueError("point_weight must be finite and >= 0")
        if self._prior_in_cloud_order and self._perm is not None:
            w = w.index_select(0, self._perm.long())
        prior, _ = self._prior_args()
        if self._weight is None or self._weight.shape != w.shape or self._weight.device != w.device:
            self._weight = torch.empty_like(w)
            self._weight_sums = torch.empty(2, dtype=torch.float64, device=w.device)
            self._weight_den = torch.empty(1, dtype=torch.float64, device=w.device)
        self._weight.copy_(w)
        self._weight_sums.copy_(ops._BACKEND.weight_sums(self._weight, prior))
        self._weight_den.copy_(self._weight_sums[1:])
        ops._all_reduce(self._weight_den, ops._reduce_ops()[2], self.group)   # one double per weight state
        if not float(self._weight_den[0]) > 0.0:
            raise ValueError("point_weight must have a positive sum")
        self._weight_key = self._weight_state_key()

    def _weight_args(self):
        """(weight as the kernels index it, this shard's cov_weight_sums (2,), global sum_j w_j (1,)), or Nones."""
        if self.point_weight is None:
            return None, None, None
        if self._weight is None or self._weight_key != self._weight_state_key():
            self._write_weight()
        return self._weight, self._weight_sums, self._weight_den

    def set_point_weight(self, point_weight):
        """Replace the point weight (None: every point counts the same), (N,) fp32 in the order of `self.points`, finite,
        >= 0, with a positive sum.  The model's copies are rewritten now, at the same addresses when the shape is unchanged,
        so a CUDA graph captured WITH a weight evaluates the new one on its next replay (a graph captured without a weight
        needs a new capture)."""
        self.point_weight = None if point_weight is None else torch.as_tensor(point_weight).to(self.device)
        if self.point_weight is not None and self._weight is not None:
            self._write_weight()

    def _cloud(self):
        # The ordered copy, its permutation and the tile boxes belong to ONE state of `self.points`: the cache is keyed
        # on identity and on torch's version counter, so both `model.points = new` and an in-place `model.points.copy_()`
        # trigger a re-sort (the exact pruning relies on the boxes bounding the points the kernels read).
        key = (id(self.points), self.points._version)
        if self._pts32 is None or self._pts32_key != key:
            pts = ops._BACKEND.prepare(self.points, what="points")
            self._pts32, self._perm, self._boxes = ops._BACKEND.order_cloud(pts, self.spatial_sort)
            self._pts32_key = key
        return self._pts32

    def set_points(self, points):
        """Replace the cloud; the Morton-ordered copy, permutation and boxes are rebuilt on the next forward.  Inside a
        captured CUDA graph use `refresh_points_()` instead (same shapes, buffers rewritten in place)."""
        self.points = torch.as_tensor(points, dtype=torch.float32).to(self.device)
        self._pts32 = None

    def detach_state(self):
        """Drop the references this model keeps into the last autograd graph (`loss[...]`, `losses`, `_mean`, the
        per-point or per-candidate outputs) so that the graph — and the gradient-accumulation nodes bound to the stream it
        ran on — can be freed (graphs.GraphedStep calls this before it warms up on its capture stream)."""
        self._mean = None
        for name in ("loss", "losses", "rewards", "means", "totals"):
            v = getattr(self, name, None)
            if isinstance(v, torch.Tensor):
                setattr(self, name, v.detach())
            elif isinstance(v, dict):
                for k, t in list(v.items()):
                    if isinstance(t, torch.Tensor):
                        v[k] = t.detach()

    @torch.no_grad()
    def refresh_points_(self, points):
        """In-place cloud update for CUDA-graph replays (graphs.GraphedStep): `points` must have the shape of the
        current cloud; `self.points`, the ordered copy, the permutation and the boxes keep their addresses and are
        rewritten, so a graph captured earlier evaluates the NEW cloud on its next replay."""
        if self._pts32 is None:
            self._cloud()
        if tuple(points.shape) != tuple(self.points.shape):
            raise ValueError("refresh_points_ needs a cloud of the same shape; use set_points() and re-capture")
        self.points.copy_(points)
        pts = ops._BACKEND.prepare(self.points, what="points")
        new_pts, new_perm, new_boxes = ops._BACKEND.order_cloud(pts, self.spatial_sort)
        if self._pts32.data_ptr() != self.points.data_ptr():
            self._pts32.copy_(new_pts)
        if self._perm is not None:
            self._perm.copy_(new_perm)
        if self._boxes is not None and new_boxes is not None:
            self._boxes.copy_(new_boxes)
        self._pts32_key = (id(self.points), self.points._version)
        if getattr(self, "prior_logodds", None) is not None and self._prior is not None:
            self._write_prior()   # the prior copy follows the new permutation, in place
        if getattr(self, "point_weight", None) is not None and self._weight is not None:
            self._write_weight()   # so does the weight copy (and its sums)

    def _kept_workspace(self, cloud, need):
        # one workspace per (cloud, size), kept across steps: nothing in it outlives a call
        if not cloud.is_cuda:
            return None
        if self._ws is None or self._ws.numel() < need or self._ws.device != cloud.device:
            self._ws = torch.empty(need, dtype=torch.uint8, device=cloud.device)
        return self._ws


class ModelTraj(_OrderedCloudModel):
    def __init__(self, points, wps_poses, wps_quats, intrins, img_width, img_height, min_dist=1.0, max_dist=5.0,
                 smoothness_weight=14.0, traj_length_weight=0.02, device=torch.device("cuda"), group=None,
                 n_total=None, spatial_sort=True, fused_regularizers=False, prior_logodds=None, point_weight=None):
        super().__init__()
        assert wps_poses.dim() == wps_quats.dim()
        assert wps_poses.size()[1] == 3
        assert wps_quats.size()[1] == 4

        self.device = device
        self.points = torch.as_tensor(points, dtype=torch.float32).to(self.device)
        self.rewards = None
        self.observations = None
        self.lo_sum = 0.0
        self.poses0 = torch.as_tensor(wps_poses, dtype=torch.float32).to(self.device)
        self.quats0 = torch.as_tensor(wps_quats, dtype=torch.float32).to(self.device)
        self.poses = nn.Parameter(deepcopy(self.poses0))
        self.quats = nn.Parameter(deepcopy(self.quats0))
        self.K = torch.as_tensor(intrins, dtype=torch.float32).to(self.device)
        self.img_width, self.img_height = float(img_width), float(img_height)
        self.eps = 1e-6
        self.pc_clip_limits = [min_dist, max_dist]
        self.loss = {"vis": float("inf"), "length": float("inf"), "l2": float("inf"), "smooth": float("inf")}
        self.smoothness_weight = smoothness_weight
        self.traj_length_weight = traj_length_weight
        self.group = group        # torch.distributed group when `points` is this rank's shard
        self.n_total = n_total    # global point count in that case
        # The cloud is constant over the optimisation (src/trajectory_optimization.py:83-127), so a Morton-ordered
        # copy is made once; the kernels prune whole tiles of it per pose (bit-identical results) and write
        # `rewards` back in the order of `self.points`.
        self.spatial_sort = spatial_sort
        # The l2 / smooth / length terms default to the torch-op restatement, which repeats the reference's fp32
        # arithmetic operation by operation.  `fused_regularizers=True` computes them and their gradients in one launch
        # in fp64 (cov_traj_regularizers): ~40 % less step latency on small clouds, but on nearly straight paths the
        # smooth-term gradient then differs from the reference's by up to ~1e-4 relative — arccos' is ill-conditioned
        # near -1 and the reference evaluates it in fp32.
        self.fused_regularizers = fused_regularizers
        self._mean = None
        self._step_cache = {}
        self._pts32 = None
        self._perm = None
        self._boxes = None
        self._ws = None
        # Map memory: (N,) fp32 log-odds of what earlier paths observed, in the order of `self.points` (indexed like
        # `rewards`); rewards_j = sigmoid(prior_j + sum_w lo_jw).  Folding an executed path in: `observed_logodds()`.
        self._init_prior(prior_logodds)
        # What is worth seeing: (N,) fp32 importance per point, in the order of `self.points`; the visibility term then
        # uses the weighted mean sum_j w_j r_j / sum_j w_j (the rewards themselves do not change).
        self._init_weight(point_weight)
        self.to(self.device)

    def _workspace(self, cloud):
        if not cloud.is_cuda:
            return None
        return self._kept_workspace(cloud, ops._BACKEND.traj_workspace_bytes(cloud, max(1, self.poses.shape[0])))

    def _wps_step(self, vis_wps_dist):
        # src/model.py:214-215.  poses0 never changes, so the host sync happens once per distance
        key = float(vis_wps_dist)
        if key not in self._step_cache:
            self._step_cache[key] = int(_wps_quotient(self.poses0, vis_wps_dist)) + 1
        return self._step_cache[key]

    def forward(self, vis_wps_dist=0.5, debug=False):
        t0 = time()
        wps_step = self._wps_step(vis_wps_dist)
        # waypoints range(0, N_wps, wps_step) (src/model.py:217); the others get no visibility gradient
        cloud = self._cloud()
        prior, prior_sum = self._prior_args()
        weight, wsums, wden = self._weight_args()
        cam = ops._lib.camera(self.img_width, self.img_height, self.pc_clip_limits[0], self.pc_clip_limits[1], self.eps)
        rewards, mean = ops.CoverageTrajFn.apply(cloud, self.poses[::wps_step], self.quats[::wps_step], self.K, cam,
                                                 self.n_total, self.group, self._perm, self._boxes,
                                                 None if self.spatial_sort else True, self._workspace(cloud), prior,
                                                 prior_sum, weight, wsums, wden)
        self.rewards = rewards
        self._mean = mean
        if debug:
            if rewards.is_cuda:
                torch.cuda.synchronize(rewards.device)
            print(f"Trajectory evaluation took {1000 * (time() - t0)} msec")
        t1 = time()
        loss = self.criterion(self.rewards)
        if debug:
            print(f"Loss calculation took {1000 * (time() - t1)} msec")
        return loss

    @torch.no_grad()
    def observed_logodds(self, vis_wps_dist=0.5):
        """prior_j + sum_w lo_jw over the waypoints forward() evaluates at this `vis_wps_dist`, (N,) fp32 in the order of
        `self.points`, without gradients: sigmoid of it is `self.rewards`.  After executing the path,
        `model.set_prior_logodds(model.observed_logodds())` folds what it saw into the map; clamping is the caller's."""
        wps_step = self._wps_step(vis_wps_dist)
        cloud = self._cloud()
        prior, _ = self._prior_args()
        return ops.traj_logodds(cloud, self.poses[::wps_step], self.quats[::wps_step], self.K, self.img_width,
                                self.img_height, self.pc_clip_limits[0], self.pc_clip_limits[1], self.eps,
                                prior_logodds=prior, reward_index=self._perm, boxes=self._boxes, group=self.group,
                                dense=None if self.spatial_sort else True, workspace=self._workspace(cloud))

    def criterion(self, rewards):
        # src/model.py:244-260; with a point weight the weighted mean (fp64 sums), also for rewards from elsewhere
        if rewards is self.rewards and self._mean is not None:
            mean = self._mean
        elif self.point_weight is not None:
            w = self._weight_args()[0].to(torch.float64)
            mean = ((w * rewards.to(torch.float64)).sum() / w.sum()).to(rewards.dtype)
        else:
            mean = torch.mean(rewards)
        self.loss["vis"] = 1.0 / (mean + self.eps)
        if self.fused_regularizers and self.poses.is_cuda and self.poses.shape[0] >= 3:
            # the three O(W) regularisers and their gradients in one launch (same formulas, fp64 inside)
            reg = ops.traj_regularizers(self.poses, self.poses0, self.smoothness_weight, self.traj_length_weight, self.eps)
            self.loss["l2"], self.loss["smooth"], self.loss["length"] = reg[0], reg[1], reg[2]
            return self.loss["vis"] + reg.sum()
        return self._criterion_terms_torch()

    def _criterion_terms_torch(self):
        # the same terms as plain torch expressions (fewer than 3 waypoints keep the reference's corner cases; also
        # the restatement the fused kernel is tested against)
        self.loss["l2"] = torch.linalg.norm(self.poses[0] - self.poses0[0])
        self.loss["smooth"] = self.smoothness_weight / (mean_angle_calc(self.poses, self.eps) + self.eps)
        self.loss["length"] = self.traj_length_weight * torch.abs(length_calc(self.poses) - length_calc(self.poses0))
        return self.loss["vis"] + self.loss["l2"] + self.loss["length"] + self.loss["smooth"]


# ------------------------------------------------------------------------------------------
# T trajectories optimised at once (no reference counterpart: multi-start refinement of sweep candidates)
# ------------------------------------------------------------------------------------------
class ModelTrajBatch(_OrderedCloudModel):
    """T independent ModelTraj objectives on one cloud, evaluated together: the visibility terms of all trajectories
    and their gradients come from one differentiable sweep (ops.coverage_sweep) instead of T coverage_traj calls.
    Parameters `poses` (T, W, 3) and `quats` (T, W, 4); `forward()` returns sum_t loss_t, where loss_t is
    ModelTraj.criterion's loss of trajectory t.  The per-trajectory terms are kept as (T,) tensors in `self.losses`
    ("vis", "l2", "smooth", "length"), the (T,) mean rewards in `self.means`.  `prior_logodds` (N,) fp32, in the order
    of `points`: the map memory every trajectory is scored on top of (see ModelTraj).  `point_weight` (N,) fp32, in the
    order of `points`: per-point importance; the means are then weighted means (see ModelTraj)."""

    _prior_in_cloud_order = True    # the sweeps index the prior like the (Morton-ordered) cloud

    def __init__(self, points, wps_poses, wps_quats, intrins, img_width, img_height, min_dist=1.0, max_dist=5.0,
                 smoothness_weight=14.0, traj_length_weight=0.02, device=torch.device("cuda"), group=None,
                 n_total=None, spatial_sort=True, prior_logodds=None, point_weight=None):
        super().__init__()
        wps_poses = torch.as_tensor(wps_poses, dtype=torch.float32)
        wps_quats = torch.as_tensor(wps_quats, dtype=torch.float32)
        if (wps_poses.dim() != 3 or wps_quats.dim() != 3 or wps_poses.shape[2] != 3 or wps_quats.shape[2] != 4
                or wps_poses.shape[:2] != wps_quats.shape[:2]):
            raise ValueError("ModelTrajBatch: wps_poses must be (T, W, 3) and wps_quats (T, W, 4) with the same T and W")
        if wps_poses.shape[1] < 3:
            raise ValueError("ModelTrajBatch: the smoothness term needs W >= 3 waypoints per trajectory")
        self.device = device
        self.points = torch.as_tensor(points, dtype=torch.float32).to(self.device)
        self.poses0 = wps_poses.to(self.device)
        self.quats0 = wps_quats.to(self.device)
        self.poses = nn.Parameter(deepcopy(self.poses0))
        self.quats = nn.Parameter(deepcopy(self.quats0))
        self.K = torch.as_tensor(intrins, dtype=torch.float32).to(self.device)
        self.img_width, self.img_height = float(img_width), float(img_height)
        self.eps = 1e-6
        self.pc_clip_limits = [min_dist, max_dist]
        self.smoothness_weight = smoothness_weight
        self.traj_length_weight = traj_length_weight
        self.group = group        # torch.distributed group when `points` is this rank's shard
        self.n_total = n_total    # global point count in that case
        self.spatial_sort = spatial_sort
        self.losses = {}
        self.means = None
        self._mean = None
        self._step_cache = {}
        self._pts32 = None
        self._perm = None
        self._boxes = None
        self._ws = None
        self._init_prior(prior_logodds)
        self._init_weight(point_weight)
        self.to(self.device)

    def _wps_step(self, vis_wps_dist):
        # ModelTraj._wps_step for every trajectory's poses0, with the same arithmetic; one host sync per distance
        key = float(vis_wps_dist)
        if key not in self._step_cache:
            quot = torch.stack([_wps_quotient(p0, vis_wps_dist) for p0 in self.poses0]).cpu()
            steps = sorted({int(q) + 1 for q in quot})
            if len(steps) != 1:
                raise ValueError(f"ModelTrajBatch: the trajectories' visibility strides differ ({steps}) at "
                                 f"vis_wps_dist={vis_wps_dist}: every trajectory must be evaluated on the same waypoints")
            self._step_cache[key] = steps[0]
        return self._step_cache[key]

    def forward(self, vis_wps_dist=0.5):
        wps_step = self._wps_step(vis_wps_dist)
        cloud = self._cloud()
        prior, prior_sum = self._prior_args()
        weight, wsums, wden = self._weight_args()
        P, Q = self.poses[:, ::wps_step], self.quats[:, ::wps_step]
        with ops.evaluation(dense=None if self.spatial_sort else True):
            ws = self._kept_workspace(cloud, ops._BACKEND.sweep_fused_workspace_bytes(cloud, P.shape[0], P.shape[1]))
            if prior is None and weight is None:
                means = ops.coverage_sweep(cloud, P, Q, self.K, self.img_width, self.img_height, self.pc_clip_limits[0],
                                           self.pc_clip_limits[1], self.eps, n_total=self.n_total, group=self.group,
                                           boxes=self._boxes, presorted=True, workspace=ws)
            else:   # the kept sums of the prior and the weight: no reduction over them per step
                cam = ops._lib.camera(self.img_width, self.img_height, self.pc_clip_limits[0], self.pc_clip_limits[1],
                                      self.eps)
                means = ops.CoverageSweepFn.apply(cloud, P, Q, self.K, cam, int(self.n_total or cloud.shape[0]),
                                                  self.group, self._boxes, "points", ws, prior, prior_sum, weight, wsums,
                                                  wden)
        self.means = means
        return self.criterion(means)

    @torch.no_grad()
    def prefix_means(self, vis_wps_dist=0.5):
        """(T, P') fp64 mean rewards of every prefix of every trajectory over the waypoints `forward()` evaluates
        (`[:, ::wps_step]`): [t, i] is the mean of trajectory t cut after its i-th evaluated waypoint, and [:, -1] is
        `self.means` of a forward at the same poses (ops.sweep_prefix_rewards).  With the model's cloud, prior, weight
        and group; without gradients."""
        wps_step = self._wps_step(vis_wps_dist)
        cloud = self._cloud()
        prior, prior_sum = self._prior_args()
        weight, wsums, wden = self._weight_args()
        P, Q = self.poses[:, ::wps_step], self.quats[:, ::wps_step]
        cam = ops._lib.camera(self.img_width, self.img_height, self.pc_clip_limits[0], self.pc_clip_limits[1], self.eps)
        with ops.evaluation(dense=None if self.spatial_sort else True):
            out = ops._sweep_run(ops._prefix_sums, P.shape[1], cloud, P, Q, self.K, cam, self.n_total, self.group,
                                 self._boxes, "points", prior, prior_sum, weight, wsums, wden)
        return out.reshape(P.shape[0], P.shape[1])

    def criterion(self, means):
        # ModelTraj.criterion per trajectory; length_calc and mean_angle_calc restated over the batch dimension
        p, p0 = self.poses, self.poses0
        self.losses["vis"] = 1.0 / (means + self.eps)
        self.losses["l2"] = torch.linalg.norm(p[:, 0] - p0[:, 0], dim=-1)
        ab = p[:, :-2] - p[:, 1:-1]
        ac = p[:, 2:] - p[:, 1:-1]
        cosang = (ab * ac).sum(dim=2) / (torch.linalg.norm(ab, dim=2) * torch.linalg.norm(ac, dim=2) + self.eps)
        mean_angle = torch.arccos(cosang).sum(dim=1) / (p.shape[1] - 2)
        self.losses["smooth"] = self.smoothness_weight / (mean_angle + self.eps)
        length = torch.linalg.norm(p[:, 1:] - p[:, :-1], dim=-1).sum(dim=1)
        length0 = torch.linalg.norm(p0[:, 1:] - p0[:, :-1], dim=-1).sum(dim=1)
        self.losses["length"] = self.traj_length_weight * torch.abs(length - length0)
        loss = self.losses["vis"] + self.losses["l2"] + self.losses["length"] + self.losses["smooth"]
        return loss.sum()


# ------------------------------------------------------------------------------------------
# K camera poses optimised at once (no reference counterpart: multi-start ModelPose, scoring of candidate views)
# ------------------------------------------------------------------------------------------
class ModelPoseBatch(_OrderedCloudModel):
    """K independent ModelPose objectives on one cloud, evaluated together: the totals of all candidates and their
    gradients come from one pass over the cloud (ops.coverage_pose_batch) instead of K coverage_pose calls.
    Parameters `trans` (K, 3) and `quat` (K, 4); `forward()` returns sum_k 1/(total_k + eps), i.e. ModelPose.criterion
    per candidate, summed.  Adam is elementwise, so one Adam over both parameters is K independent ModelPose
    optimisations.  The (K,) totals are kept in `self.totals`, the (K,) per-candidate losses in `self.losses`."""

    def __init__(self, points, trans0, q0, intrins, img_width, img_height, min_dist=1.0, max_dist=5.0,
                 device=torch.device("cuda:0"), group=None, spatial_sort=True):
        super().__init__()
        trans0 = torch.as_tensor(trans0, dtype=torch.float32)
        q0 = torch.as_tensor(q0, dtype=torch.float32)
        if (trans0.dim() != 2 or q0.dim() != 2 or trans0.shape[1] != 3 or q0.shape[1] != 4
                or trans0.shape[0] != q0.shape[0] or trans0.shape[0] == 0):
            raise ValueError("ModelPoseBatch: trans0 must be (K, 3) and q0 (K, 4) with the same K >= 1; got "
                             f"{tuple(trans0.shape)} and {tuple(q0.shape)}")
        assert intrins.size() == torch.Size([3, 3])
        self.device = device
        self.points = torch.as_tensor(points, dtype=torch.float32).to(self.device)
        self.trans = nn.Parameter(trans0.to(self.device))
        self.quat = nn.Parameter(q0.to(self.device))
        self.K = torch.as_tensor(intrins, dtype=torch.float32).to(self.device)
        self.img_width, self.img_height = float(img_width), float(img_height)
        self.eps = 1e-6
        self.pc_clip_limits = [min_dist, max_dist]
        self.group = group            # torch.distributed group when `points` is this rank's shard
        # the objective is a sum over the points, so their order is free: the kernels read a Morton-ordered copy made
        # once per cloud, whose tile boxes let them skip (box, pose) pairs that are exactly zero
        self.spatial_sort = spatial_sort
        self.totals = None
        self.losses = None
        self._mean = None
        self._pts32 = None
        self._perm = None
        self._boxes = None
        self._ws = None
        self.to(self.device)

    def forward(self, debug=False, hpr=False):
        t0 = time()
        cloud = self._cloud()
        weight = None
        if hpr:  # ModelPose's mask: HPR of the untransformed cloud, in the caller's order, then into the cloud's order
            weight = hidden_pts_removal(self.points.detach(), device=self.device)[1]
            weight = ops._BACKEND.prepare(weight, cloud.device, "weight").reshape(-1)
            if self._perm is not None:
                weight = weight.index_select(0, self._perm.long())
        with ops.evaluation(dense=None if self.spatial_sort else True):
            ws = self._kept_workspace(cloud, ops._BACKEND.pose_batch_workspace_bytes(cloud, self.trans.shape[0]))
            totals = ops.coverage_pose_batch(cloud, self.trans, self.quat, self.K, self.img_width, self.img_height,
                                             self.pc_clip_limits[0], self.pc_clip_limits[1], self.eps, weight=weight,
                                             group=self.group, boxes=self._boxes, presorted=True, workspace=ws)
        self.totals = totals
        if debug:
            if totals.is_cuda:
                torch.cuda.synchronize(totals.device)
            print(f"\nBatched visibility estimation of {totals.shape[0]} poses took: {1000 * (time() - t0)} msec")
        return self.criterion(totals)

    def criterion(self, totals):
        self.losses = 1.0 / (totals + self.eps)
        return self.losses.sum()
