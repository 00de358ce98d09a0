"""Device resize of predicted depth (``mte_resize_linear``): what the kernel costs, and what the AUC sweep from
half-resolution predictions costs with the resize on the device against today's host ``cv2.resize``.

    python scripts/bench_resize_eval.py --out profiles/r06_resize_eval.json [--images 102] [--warmup 2] [--iters 7]

Parts:
  kernel   resize_linear alone on device-resident planes, 102 x 192x640 -> 384x1280 (KITTI 2x) and
           8 x 608x968 -> 1216x1936 (DDAD size, 2x): CUDA events around --launches back-to-back calls, ms per call;
           bytes = 4*N*h*w read + 4*N*H*W written (the model of the kernel, every source pixel read once), over the
           7.7 TB/s data-sheet HBM figure of one B200.  Both working sets exceed the 126 MB L2 (written output).
  sweep    the 12-setting AUC sweep (KITTI crop, max_dist 0.002) of bench.kitti_like_set(--images, 7000) with the
           predictions downsampled to 192x640 on the host BEFORE any timing:
             device_e2e    host arrays -> upload of the half-size planes -> resize + sweep on the device -> counts on
                           the host (pr_evaluation_arrays' new path);
             host_e2e      host cv2.resize of every plane to 384x1280 -> upload -> sweep -> counts on the host
                           (the path before the device resize);
             device_planes the half-size planes already on the device: resize + sweep;
             full_planes   the full-size planes already on the device: sweep only (no resize).
           e2e arms: host clock around the call, ending in the device-to-host copy of the counts (a synchronise);
           device arms: CUDA events.  Arms alternate within each of --iters rounds after --warmup rounds; medians and
           every run are reported.  The counts of all four arms must be equal.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "scripts"))

HBM_TBS = 7.7   # NVIDIA HGX B200 data sheet, one GPU


def kernel_ms(fn, launches, warmup, iters):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    runs = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(launches):
            fn()
        b.record()
        b.synchronize()
        runs.append(a.elapsed_time(b) / launches)
    return float(np.median(runs)), runs


def main():
    import cv2
    import torch
    import bench
    from bench_thin_sweep import gpu_facts
    from mindtheedge_b200.edge import resize_linear
    from mindtheedge_b200.eval_depth_edges import sweep_counts
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--images", type=int, default=102)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--iters", type=int, default=7)
    ap.add_argument("--launches", type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs a GPU"
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    res = gpu_facts()
    res.update({"images": args.images, "warmup": args.warmup, "iters": args.iters, "launches": args.launches,
                "hbm_datasheet_tb_s": HBM_TBS, "opencv": cv2.__version__, "opencv_threads": cv2.getNumThreads(),
                "kernel": [], "sweep": {}})

    # ---- the kernel alone
    g = np.random.default_rng(0)
    for N, (h, w), (H, W) in [(102, (192, 640), (384, 1280)), (8, (608, 968), (1216, 1936))]:
        src = torch.from_numpy(g.uniform(0, 80, (N, h, w)).astype(np.float32)).to(dev)
        ms, runs = kernel_ms(lambda: resize_linear(src, (H, W)), args.launches, args.warmup, args.iters)
        nbytes = 4 * N * (h * w + H * W)
        row = {"N": N, "src": [h, w], "dst": [H, W], "ms": ms, "runs_ms": runs, "bytes": nbytes,
               "tb_s": nbytes / ms / 1e9, "share_of_datasheet_hbm": nbytes / ms / 1e9 / HBM_TBS}
        res["kernel"].append(row)
        print(json.dumps(row), flush=True)
        del src

    # ---- the AUC sweep from half-resolution predictions
    depths, gts = bench.kitti_like_set(args.images, 7000)
    H, W = gts.shape[1:]
    half = np.stack([cv2.resize(d, (W // 2, H // 2), interpolation=cv2.INTER_LINEAR) for d in depths])
    crop, rng = bench.KITTI_CROP, list(range(20, 241, 20))
    g_dev = torch.from_numpy(gts).to(dev)
    half_dev = torch.from_numpy(half).to(dev)
    full_dev = torch.from_numpy(np.stack([cv2.resize(d, (W, H), interpolation=cv2.INTER_LINEAR) for d in half])).to(dev)

    def sweep(d):
        return sweep_counts(d, g_dev, rng, crop, 0.0, 80.0, max_dist=0.002)

    def device_e2e():
        return sweep(torch.from_numpy(half).to(dev)).cpu().numpy()

    def host_e2e():
        full = np.stack([cv2.resize(d, (W, H), interpolation=cv2.INTER_LINEAR) for d in half])
        return sweep(torch.from_numpy(full).to(dev)).cpu().numpy()

    e2e = {"device_e2e": device_e2e, "host_e2e": host_e2e}
    dev_arms = {"device_planes": lambda: sweep(half_dev), "full_planes": lambda: sweep(full_dev)}
    counts = {k: fn() for k, fn in e2e.items()}
    counts.update({k: fn().cpu().numpy() for k, fn in dev_arms.items()})
    equal = all(np.array_equal(c, counts["host_e2e"]) for c in counts.values())
    for _ in range(args.warmup):
        for fn in list(e2e.values()) + list(dev_arms.values()):
            fn()
    torch.cuda.synchronize()
    runs = {k: [] for k in list(e2e) + list(dev_arms)}
    for _ in range(args.iters):
        for k, fn in e2e.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            runs[k].append((time.perf_counter() - t0) * 1e3)
        for k, fn in dev_arms.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            runs[k].append(a.elapsed_time(b))
    med = {k: float(np.median(v)) for k, v in runs.items()}
    res["sweep"] = {"src": list(half.shape[1:]), "gt": [H, W], "counts_equal": bool(equal),
                    **{f"{k}_ms": v for k, v in med.items()}, **{f"{k}_runs_ms": v for k, v in runs.items()},
                    "host_over_device_e2e": med["host_e2e"] / med["device_e2e"],
                    "resize_in_sweep_ms": med["device_planes"] - med["full_planes"]}
    print(json.dumps({k: v for k, v in res["sweep"].items() if not k.endswith("runs_ms")}), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    if not equal:
        sys.exit("the counts of the arms differ")


if __name__ == "__main__":
    main()
