"""Thinned 99-threshold PR sweep (evaluate_boundaries' default protocol): composed ops against the fused op.

    python scripts/bench_thin_sweep.py --out profiles/thin_sweep.json [--images 102] [--warmup 1] [--iters 3]

Inputs: the predicted depth of bench.kitti_like_set(102, 7000) at the KITTI crop, 99 thresholds
(linspace(0.01, 0.99, 99)), max_dist 0.0075, with two strength maps per image:
  ridge  per-image normalised Sobel magnitude of the depth after non-maximum suppression (thin curves),
  blob   tests/synth.py::prob_map DEE maps (thick regions that thinning erodes over many iterations);
plus one uncropped 1216x1936 image of each kind (the thinning runs in global memory there).

Arms:
  composed  per image: binarise the window at every threshold, binary_thin_batch, correspond_pixels_batch against
            the GT window expanded T times -- what evaluate_boundaries ran before the fused op, kept on the device
            (no host synchronisation inside the timed loop);
  fused     one pr_counts(..., apply_thinning=True) over the batch.
The counts of both arms must be equal.  Times are CUDA events over --iters calls after --warmup calls, arms
alternating; Gpx/s counts (image x threshold) window pixels.  --profile adds, per case, the CUDA time and
launch count of every kernel per fused call (torch.profiler over two calls, after the timed loop).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def ridge_map(depth):
    """Sobel magnitude after 4-direction non-maximum suppression, normalised to [0, 1] per image."""
    import cv2
    gx = cv2.Sobel(depth, cv2.CV_32F, 1, 0, ksize=3)
    gy = cv2.Sobel(depth, cv2.CV_32F, 0, 1, ksize=3)
    mag = np.hypot(gx, gy)
    ang = (np.rad2deg(np.arctan2(gy, gx)) + 180.0) % 180.0
    sector = ((ang + 22.5) // 45).astype(np.int32) % 4          # 0: E-W, 1: NE-SW, 2: N-S, 3: NW-SE
    p = np.pad(mag, 1)
    H, W = mag.shape
    nb = {0: ((0, 1), (0, -1)), 1: ((-1, 1), (1, -1)), 2: ((1, 0), (-1, 0)), 3: ((1, 1), (-1, -1))}
    keep = np.zeros_like(mag, dtype=bool)
    for s, ((ay, ax), (by, bx)) in nb.items():
        a = p[1 + ay:1 + ay + H, 1 + ax:1 + ax + W]
        b = p[1 + by:1 + by + H, 1 + bx:1 + bx + W]
        keep |= (sector == s) & (mag >= a) & (mag >= b)
    out = np.where(keep, mag, 0.0)
    m = out.max()
    return (out / m if m > 0 else out).astype(np.float32)


def composed(pred, gt, thr_dev, max_dist, crop):
    """Per image: binarise, binary_thin_batch, correspond_pixels_batch against the expanded GT -> int64[T,4]."""
    import torch
    from mindtheedge_b200.bsds.thin import binary_thin_batch
    from mindtheedge_b200.eval_depth_edges import correspond_pixels_batch
    T = thr_dev.shape[0]
    out = torch.zeros((T, 4), dtype=torch.int64, device=pred.device)
    if crop is not None:
        pred = pred[:, crop[2]:crop[3], crop[0]:crop[1]]
        gt = gt[:, crop[2]:crop[3], crop[0]:crop[1]]
    for i in range(pred.shape[0]):
        bins = (pred[i].double()[None] >= thr_dev[:, None, None]).to(torch.uint8)
        bins = binary_thin_batch(bins)
        g = gt[i][None].expand_as(bins).contiguous()
        _, _, cnt = correspond_pixels_batch(bins, g, max_dist, want_maps=False)
        out[:, 0] += cnt
        out[:, 1] += g.flatten(1).sum(1)
        out[:, 2] += cnt
        out[:, 3] += bins.flatten(1).sum(1)
    return out


def fused(pred, gt, thr, max_dist, crop):
    from mindtheedge_b200.eval_depth_edges import pr_counts
    return pr_counts(pred, gt, thr, max_dist=max_dist, crop=crop, apply_thinning=True)


def time_arms(arms, warmup, iters):
    """CUDA-event ms per call of every arm; arms alternate within each round."""
    import torch
    for _ in range(warmup):
        for fn in arms.values():
            fn()
    torch.cuda.synchronize()
    ms = {k: [] for k in arms}
    for _ in range(iters):
        for k, fn in arms.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            ms[k].append(a.elapsed_time(b))
    return {k: float(np.median(v)) for k, v in ms.items()}, ms


def kernel_split(fn, calls=2):
    """Per kernel name: CUDA ms per call of fn and launches per call, from torch.profiler over `calls` calls (after
    one untraced call).  The sum over kernels is reported beside it, so a split with lost events shows as a sum well
    below the event-timed call."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA], acc_events=True) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if t > 0:
            k = ev.key[:80]
            ms, n = out.get(k, (0.0, 0.0))
            out[k] = (ms + t / 1e3 / calls, n + ev.count / calls)
    split = {k: {"ms": v[0], "launches": v[1]} for k, v in sorted(out.items(), key=lambda kv: -kv[1][0])}
    return split, sum(v["ms"] for v in split.values())


def gpu_facts():
    import torch
    facts = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                            "-i", "0"], capture_output=True, text=True, timeout=60).stdout.strip().split(",")
        facts["power_limit_w"] = float(q[0])
        facts["max_sm_clock_mhz"] = float(q[1])
    except Exception as exc:  # noqa: BLE001 -- the numbers are still reported, without the limit
        facts["power_limit_w"] = f"unknown ({exc})"
    return facts


def main():
    import torch
    import bench
    from synth import prob_map, scene_with_gt
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--images", type=int, default=102)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--profile", action="store_true")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs a GPU"
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    thr = np.linspace(0.01, 0.99, 99)
    thr_dev = torch.from_numpy(thr).to(dev)
    max_dist = 0.0075

    depths, gts = bench.kitti_like_set(args.images, 7000)
    H, W = depths.shape[1:]
    kitti = {"ridge": np.stack([ridge_map(d) for d in depths]),
             "blob": np.stack([prob_map(H, W, 7000 + i) for i in range(args.images)])}
    g_dd, d_dd = scene_with_gt(1216, 1936, 5, n_rect=120)
    ddad = {"ridge": ridge_map(d_dd)[None], "blob": prob_map(1216, 1936, 5)[None]}
    cases = [(f"kitti_crop_{k}", m, gts, bench.KITTI_CROP) for k, m in kitti.items()]
    cases += [(f"ddad_uncropped_{k}", m, (g_dd > 127).astype(np.uint8)[None], None) for k, m in ddad.items()]

    res = gpu_facts()
    res.update({"thresholds": "linspace(0.01, 0.99, 99)", "max_dist": max_dist, "warmup": args.warmup,
                "iters": args.iters, "cases": []})
    ok = True
    for name, m, g, crop in cases:
        p = torch.from_numpy(np.ascontiguousarray(m)).to(dev)
        gd = torch.from_numpy(np.ascontiguousarray(g)).to(dev)
        c_comp = composed(p, gd, thr_dev, max_dist, crop).cpu().numpy()
        c_fused = fused(p, gd, thr, max_dist, crop).cpu().numpy()
        equal = bool(np.array_equal(c_comp, c_fused))
        ok &= equal
        med, runs = time_arms({"composed": lambda: composed(p, gd, thr_dev, max_dist, crop),
                               "fused": lambda: fused(p, gd, thr, max_dist, crop)}, args.warmup, args.iters)
        N = p.shape[0]
        h, w = (crop[3] - crop[2], crop[1] - crop[0]) if crop is not None else tuple(p.shape[1:])
        px = N * len(thr) * h * w
        row = {"case": name, "images": N, "window": [h, w], "counts_equal": equal,
               "composed_ms": med["composed"], "fused_ms": med["fused"],
               "composed_runs_ms": runs["composed"], "fused_runs_ms": runs["fused"],
               "composed_gpx_s": px / med["composed"] / 1e6, "fused_gpx_s": px / med["fused"] / 1e6,
               "speedup": med["composed"] / med["fused"],
               "sum_p_t0_t98": [int(c_fused[0, 3]), int(c_fused[-1, 3])], "count_r_t0": int(c_fused[0, 0])}
        if args.profile:
            row["fused_kernels"], row["fused_kernels_sum_ms"] = kernel_split(lambda: fused(p, gd, thr, max_dist, crop))
        res["cases"].append(row)
        print(json.dumps(row), flush=True)
    res["all_counts_equal"] = ok
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    if not ok:
        sys.exit("counts of the composed and the fused arm differ")


if __name__ == "__main__":
    main()
