"""Cost of the long trajectory path (cov_traj_fused_long) on c4's 1e8-point cloud (bench.py's generator), Morton-ordered,
boxes given, one objective evaluation per step (pass A, pass B, epilogue), the paths alternated within one process.

    python scripts/long_traj_bench.py [--points 100000000] [--repeats 5] [--profile]

  (a) W = 2048: the single call (cov_traj_minmax + cov_traj_fused) against the long path (pass A per chunk +
      cov_traj_fused_long) with pose_chunk 2048 and 1024 on identical inputs: the pure cost of chunking.
  (b) W = 4096 and 8192 on the long path.

Poses: c4's 35 m body path (64 waypoints x 5 cameras = 320 poses) repeated at lateral offsets of 1.2 m, the first W
poses, so every W sees the cloud about as densely as c4's 320 poses do.  Prints one JSON line: per repetition and median
step time in ms (CUDA events, after a warm-up of every timed path), per-pose time in us, the ratios to the single call,
whether the long path's rewards equal the single call's bit for bit (a), and the card's name, power limit and max SM
clock read in the same run.  --profile adds, from a separate torch.profiler pass after the timing, the device time per
kernel name of one step of the single call and of the long path with pose_chunk 1024."""
import argparse
import collections
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402
from scripts.prior_bench import alternate, card  # noqa: E402


def offset_path(W, dev):
    """The first W camera poses of c4's body path repeated at lateral offsets of 1.2 m (centred on c4's path)."""
    from trajectory_optimization_b200 import multicam
    rig7 = multicam.rig_tensor(multicam.ring_rig(bench.N_CAMS), dev)
    per = bench.N_WAYPOINTS * bench.N_CAMS
    reps = (W + per - 1) // per
    ts, qs = [], []
    with torch.no_grad():
        for k in range(reps):
            body = bench.body_waypoints().to(dev) + torch.tensor([0.0, 1.2 * (k - reps // 2), 0.0, 0.0], device=dev)
            t, q = multicam.camera_poses_fused(body, rig7)
            ts.append(t)
            qs.append(q)
    return torch.cat(ts)[:W].contiguous(), torch.cat(qs)[:W].contiguous()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--points", type=int, default=bench.N_POINTS_C4)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--profile", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("long_traj_bench.py needs a CUDA device")
    from trajectory_optimization_b200 import _lib, ops, tools
    dev = torch.device("cuda:0")
    B, L = ops._BACKEND, _lib.lib()
    K, img_w, img_h = tools.load_intrinsics(dev)
    Kd = K.reshape(9).contiguous()
    cam = _lib.camera(img_w, img_h, 1.0, 5.0, 1e-6)
    out = {"card": card()}
    pts = bench.make_cloud_shard(args.points, 0, 1, dev)
    spts, perm = ops.spatial_sort(pts)
    del pts
    boxes = ops.tile_boxes(spts)
    n = spts.shape[0]
    poses = {W: offset_path(W, dev) for W in (2048, 4096, 8192)}
    ws = torch.empty(max(L.cov_traj_long_workspace_bytes(n, W, c) for W in poses for c in (1024, 2048)),
                     dtype=torch.uint8, device=dev)
    rewards = torch.empty(n, dtype=torch.float32, device=dev)

    def step(W, chunk):
        """One objective evaluation: chunk None = the single call."""
        P, Q = poses[W]
        if chunk is None:
            mm = B.traj_minmax(spts, P, Q, Kd, cam, boxes, ws, False, rewards)
            acc = B.traj_fused(spts, P, Q, Kd, cam, mm, None, rewards, perm, boxes, ws, False, True)
        else:
            mm = B.sweep_minmax(spts, P, Q, Kd, cam, boxes, ws, False, rewards)
            acc = B.traj_fused_long(spts, P, Q, Kd, cam, mm, None, rewards, perm, boxes, ws, True, pose_chunk=chunk)
        return B.traj_epilogue(acc, mm, Q, n, 0)

    paths = {"single_2048": lambda: step(2048, None), "long_2048_c2048": lambda: step(2048, 2048),
             "long_2048_c1024": lambda: step(2048, 1024), "long_4096": lambda: step(4096, 2048),
             "long_8192": lambda: step(8192, 2048)}
    res = alternate(paths, args.repeats)
    med = {k: statistics.median(v) for k, v in res.items()}
    W_of = {"single_2048": 2048, "long_2048_c2048": 2048, "long_2048_c1024": 2048, "long_4096": 4096, "long_8192": 8192}
    per_pose_us = {k: 1000.0 * med[k] / W_of[k] for k in med}
    ratios = {f"{k}_over_single": med[k] / med["single_2048"] for k in med if k != "single_2048"}
    ratios.update({f"{k}_per_pose_over_single": per_pose_us[k] / per_pose_us["single_2048"] for k in ("long_4096", "long_8192")})
    # identical outputs: rewards bit for bit, mean and gradients up to the fp64 addition order
    o_single = step(2048, None)
    r_single = rewards.clone()
    same = {}
    for c in (2048, 1024):
        o = step(2048, c)
        same[f"c{c}"] = dict(rewards_equal=bool(torch.equal(rewards, r_single)),
                             outputs_rel=float(((o - o_single).abs().max() / o_single.abs().max()).item()))
    out.update(config=f"c4 cloud: {n} points, Morton-ordered; c4's body path at lateral offsets", ms=res, median_ms=med,
               per_pose_us=per_pose_us, ratios=ratios, long_vs_single_2048=same)
    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        prof_out = {}
        for name, fn in (("single_2048", paths["single_2048"]), ("long_2048_c1024", paths["long_2048_c1024"])):
            fn()
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                fn()
                torch.cuda.synchronize()
            per = collections.defaultdict(lambda: [0, 0.0])
            for e in prof.events():
                if e.device_type.name == "CUDA":
                    key = e.name.replace("void ", "").replace("(anonymous namespace)::", "").split("(")[0][:90]
                    per[key][0] += 1
                    per[key][1] += e.device_time_total / 1000.0
            prof_out[name] = {k: {"launches": v[0], "ms": round(v[1], 4)} for k, v in sorted(per.items(), key=lambda kv: -kv[1][1])}
        out["profile"] = prof_out
    print(json.dumps(out))


if __name__ == "__main__":
    main()
