"""Cost of the differentiable candidate sweep on the c5 configuration (bench.py: 1024 trajectories x 32 poses, 5e7-point
synthetic cloud, Morton-ordered, boxes built once), against the forward-only sweep and a loop of single-trajectory calls.

    python scripts/sweep_grad_bench.py [--points 50000000] [--repeats 5] [--loop-traj 64]

Prints one JSON line: per repetition and median, in ms (CUDA events, after a warm-up of every timed path):
  forward     ops.sweep_rewards (no gradient)
  fused       ops.coverage_sweep forward + means.sum().backward()
  loop        coverage_traj + backward for each of the first `--loop-traj` trajectories, scaled linearly to all of them
plus the work counters of one fused call (cov_traj_opts.stats_dev: [0] pairs, [1] evaluated, [4] differentiated,
[6] listed) and the card's name and power limit read in the same run.  The 600 MB cloud is far larger than L2."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--points", type=int, default=bench.N_POINTS_C5)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--loop-traj", type=int, default=64, help="trajectories the coverage_traj loop runs (scaled to all)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sweep_grad_bench.py needs a CUDA device")
    from trajectory_optimization_b200 import ops, tools
    dev = torch.device("cuda:0")
    K, img_w, img_h = tools.load_intrinsics(dev)
    pts = bench.make_cloud_shard(args.points, 0, 1, dev)
    spts, _ = ops.spatial_sort(pts)
    del pts
    boxes = ops.tile_boxes(spts)
    poses, quats = bench.c5_trajectories()
    P, Q = poses.to(dev), quats.to(dev)
    T, Pn = P.shape[0], P.shape[1]
    n_loop = min(args.loop_traj, T)
    ws = torch.empty(ops._BACKEND.sweep_fused_workspace_bytes(spts, T, Pn), dtype=torch.uint8, device=dev)
    traj_ws = ops._BACKEND.traj_workspace(spts, Pn)

    def forward():
        return ops.sweep_rewards(spts, P, Q, K, img_w, img_h, boxes=boxes, presorted=True)

    def fused():
        Pg, Qg = P.detach().requires_grad_(True), Q.detach().requires_grad_(True)
        means = ops.coverage_sweep(spts, Pg, Qg, K, img_w, img_h, boxes=boxes, presorted=True, workspace=ws)
        means.sum().backward()
        return means

    def loop():
        for t in range(n_loop):
            Pg, Qg = P[t].detach().requires_grad_(True), Q[t].detach().requires_grad_(True)
            _, mean = ops.coverage_traj(spts, Pg, Qg, K, img_w, img_h, boxes=boxes, workspace=traj_ws)
            mean.backward()

    def timed(fn):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    for fn in (forward, fused, loop):   # warm-up: modules, occupancy queries, allocator
        fn()
    res = {"forward": [], "fused": [], "loop": []}
    for _ in range(args.repeats):       # alternate the three paths within each repetition
        res["forward"].append(timed(forward))
        res["fused"].append(timed(fused))
        res["loop"].append(timed(loop) * T / n_loop)
    stats = torch.zeros(8, dtype=torch.int64, device=dev)
    with ops.evaluation(stats=stats):
        fused()
    torch.cuda.synchronize()
    med = {k: statistics.median(v) for k, v in res.items()}
    print(json.dumps({
        "config": f"c5: {T} trajectories x {Pn} poses, {args.points} points (Morton-ordered, boxes given)",
        "card": card(), "ms": res, "median_ms": med,
        "loop_note": f"coverage_traj + backward on the first {n_loop} trajectories, scaled x{T / n_loop:g}",
        "fused_over_forward": med["fused"] / med["forward"], "loop_over_fused": med["loop"] / med["fused"],
        "stats_fused_call": {"pairs": int(stats[0]), "evaluated": int(stats[1]), "differentiated": int(stats[4]),
                             "listed": int(stats[6])}}))


if __name__ == "__main__":
    main()
