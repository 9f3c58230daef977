"""Cost of the batched ModelPose objective (ops.coverage_pose_batch: K candidate poses, one pass over the cloud) against
a loop of K single-pose calls (ops.coverage_pose), forward + backward of the totals in both.

    python scripts/pose_batch_bench.py [--repeats 5] [--skip-large]

Prints one JSON line with CUDA-event medians (ms), the card's name, power limit and max SM clock read in the same run,
and the work counters of the batch calls (cov_traj_opts.stats_dev: [0] (warp box, pose) pairs, [1] evaluated):
  c1     the c1 cloud of scripts/bench_extra.py (1e5 points in the 40 x 40 x 5 m bench box), K = 1, 16, 64, 256, 1024;
         the loop runs at most 64 poses per repetition and is scaled linearly to K.  Also one Adam step of
         ModelPoseBatch (K = 256) and of ModelPose, each captured as one CUDA graph (graphs.GraphedStep).
  bench  1e8 points in the same box (1.2 GB, far larger than L2), K = 64: batch against the loop.
  map    1e8 points on a 400 x 400 x 5 m map, K = 64 candidates spread over it: the pruned batch (boxes given) against
         the dense batch, with the fraction of (box, pose) pairs evaluated.
Every cloud is Morton-ordered and its boxes built once, outside the timed windows (what a caller that evaluates the
same cloud repeatedly does); the loop's coverage_pose calls read the same ordered cloud."""
import argparse
import json
import math
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


def box(n, seed, lo, hi, dev):
    g = torch.Generator(device=dev).manual_seed(seed)
    lo, hi = torch.tensor(lo, device=dev), torch.tensor(hi, device=dev)
    return torch.rand(n, 3, generator=g, device=dev) * (hi - lo) + lo


def candidates(K, lo, hi, seed, dev):
    g = torch.Generator().manual_seed(seed)
    lo, hi = torch.tensor(lo), torch.tensor(hi)
    trans = torch.rand(K, 3, generator=g) * (hi - lo) + lo
    yaw = (torch.rand(K, generator=g) * 2 - 1) * math.pi
    quats = torch.stack([torch.cos(yaw / 2), 0 * yaw, 0 * yaw, torch.sin(yaw / 2)], 1)
    return trans.to(dev), quats.to(dev)


def timed(fn, inner=1):
    """ms per call of fn, CUDA events around `inner` back-to-back calls."""
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(inner):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / inner


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--skip-large", action="store_true", help="only the c1-scale cases")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("pose_batch_bench.py needs a CUDA device")
    from trajectory_optimization_b200 import model, ops, tools
    from trajectory_optimization_b200.graphs import GraphedStep
    dev = torch.device("cuda:0")
    Kc, iw, ih = tools.load_intrinsics(dev)
    out = {"card": card()}

    def batch_fn(pts, boxes, T, Q, dense=False):
        def fn():
            Tg, Qg = T.detach().requires_grad_(True), Q.detach().requires_grad_(True)
            with ops.evaluation(dense=dense):
                totals = ops.coverage_pose_batch(pts, Tg, Qg, Kc, iw, ih, boxes=boxes, presorted=True)
            totals.sum().backward()
        return fn

    def loop_fn(pts, T, Q, n_loop):
        def fn():
            for k in range(n_loop):
                t, q = T[k:k + 1].detach().requires_grad_(True), Q[k:k + 1].detach().requires_grad_(True)
                _, total = ops.coverage_pose(pts, t, q, Kc, iw, ih)
                total.backward()
        return fn

    def counters(pts, boxes, T, Q, dense=False):
        stats = torch.zeros(8, dtype=torch.int64, device=dev)
        with ops.evaluation(stats=stats):
            batch_fn(pts, boxes, T, Q, dense)()
        torch.cuda.synchronize()
        return {"pairs": int(stats[0]), "evaluated": int(stats[1]), "evaluated_fraction": int(stats[1]) / max(int(stats[0]), 1)}

    def compare(pts, boxes, T, Q, inner, n_loop_max=64):
        K = T.shape[0]
        n_loop = min(K, n_loop_max)
        fb, fl = batch_fn(pts, boxes, T, Q), loop_fn(pts, T, Q, n_loop)
        fb(); fl()   # warm-up: modules, allocator
        rb, rl = [], []
        for _ in range(args.repeats):   # alternate the two paths within each repetition
            rb.append(timed(fb, inner))
            rl.append(timed(fl, max(1, inner // n_loop)) * K / n_loop)
        mb, ml = statistics.median(rb), statistics.median(rl)
        return {"K": K, "batch_ms": mb, "loop_ms": ml, "loop_over_batch": ml / mb, "batch_ms_reps": rb, "loop_ms_reps": rl,
                "loop_note": f"coverage_pose + backward on {n_loop} poses, scaled x{K / n_loop:g}",
                "counters": counters(pts, boxes, T, Q)}

    # ---- c1 scale ----
    pts, _ = ops.spatial_sort(box(100_000, 0, bench.BOX_LO, bench.BOX_HI, dev))
    boxes = ops.tile_boxes(pts)
    c1 = []
    for K in (1, 16, 64, 256, 1024):
        T, Q = candidates(K, (-5.0, -5.0, 0.0), (25.0, 25.0, 1.5), K, dev)
        c1.append(compare(pts, boxes, T, Q, inner=64))
    out["c1_1e5_points"] = c1
    T, Q = candidates(256, (-5.0, -5.0, 0.0), (25.0, 25.0, 1.5), 7, dev)
    mb = model.ModelPoseBatch(pts, T, Q, Kc, iw, ih, device=dev)
    ob = torch.optim.Adam([{"params": [mb.trans], "lr": 0.02}, {"params": [mb.quat], "lr": 0.02}], capturable=True)
    gb = GraphedStep(mb, ob)
    mp = model.ModelPose(pts, T[:1].clone(), Q[:1].clone(), Kc, iw, ih, device=dev)
    op = torch.optim.Adam([{"params": [mp.trans], "lr": 0.02}, {"params": [mp.quat], "lr": 0.02}], capturable=True)
    gp = GraphedStep(mp, op)
    rb, rp = [], []
    for _ in range(args.repeats):
        rb.append(timed(gb.step, 200))
        rp.append(timed(gp.step, 200))
    out["c1_graphed_adam_step"] = {"model_pose_batch_K256_ms": statistics.median(rb), "model_pose_ms": statistics.median(rp),
                                   "batch_reps": rb, "single_reps": rp}
    del mb, mp, gb, gp, pts, boxes
    if not args.skip_large:
        # ---- bench cloud: 1e8 points, 40 x 40 x 5 m, K = 64 ----
        pts, _ = ops.spatial_sort(box(100_000_000, 1, bench.BOX_LO, bench.BOX_HI, dev))
        boxes = ops.tile_boxes(pts)
        T, Q = candidates(64, (-5.0, -5.0, 0.0), (25.0, 25.0, 1.5), 11, dev)
        out["bench_1e8_points"] = compare(pts, boxes, T, Q, inner=1)
        del pts, boxes
        # ---- large map: 1e8 points, 400 x 400 x 5 m, K = 64 spread over it; pruned vs dense batch ----
        pts, _ = ops.spatial_sort(box(100_000_000, 2, (0.0, 0.0, 0.0), (400.0, 400.0, 5.0), dev))
        boxes = ops.tile_boxes(pts)
        T, Q = candidates(64, (10.0, 10.0, 0.5), (390.0, 390.0, 2.0), 13, dev)
        fp, fd = batch_fn(pts, boxes, T, Q), batch_fn(pts, boxes, T, Q, dense=True)
        fp(); fd()
        rp, rd = [], []
        for _ in range(args.repeats):
            rp.append(timed(fp))
            rd.append(timed(fd))
        mp_, md = statistics.median(rp), statistics.median(rd)
        out["map_1e8_points_400m"] = {"K": 64, "pruned_ms": mp_, "dense_ms": md, "dense_over_pruned": md / mp_,
                                      "pruned_ms_reps": rp, "dense_ms_reps": rd, "counters": counters(pts, boxes, T, Q)}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
