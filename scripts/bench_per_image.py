"""Per-image PR counts: what one batched per-image call costs against the summed call and against the only way to get
per-image counts without it (one call per image).

    python scripts/bench_per_image.py --out profiles/r05_per_image.json [--images 102] [--warmup 2] [--iters 5]

Workloads (max_dist, crop and thresholds as the shipped protocols use them):
  canny12  bench.kitti_like_set(102, 7000): 102 KITTI-DE GT maps at 384x1280, 12 Canny settings, KITTI crop,
           max_dist 0.002, through sweep_counts (Canny level plane + counts);
  thin99   the same depths' ridge maps (scripts/bench_thin_sweep.py::ridge_map), KITTI crop, 99 thresholds
           linspace(0.01, 0.99, 99), max_dist 0.0075, apply_thinning=True, through pr_counts.
Arms: summed (per_image=False, as today), per_image (one batched per_image=True call), single (N calls of one image).
The per-image rows of the per_image and single arms must be equal and sum to the summed arm.  Times are CUDA events per
call after --warmup calls of every arm, arms alternating within each of --iters rounds; the median is reported next to
every run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "scripts"))


def main():
    import torch
    import bench
    from bench_thin_sweep import gpu_facts, ridge_map, time_arms
    from mindtheedge_b200.eval_depth_edges import pr_counts, sweep_counts
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--images", type=int, default=102)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--iters", type=int, default=5)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs a GPU"
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    depths, gts = bench.kitti_like_set(args.images, 7000)
    d_dev, g_dev = torch.from_numpy(depths).to(dev), torch.from_numpy(gts).to(dev)
    crop, rng = bench.KITTI_CROP, list(range(20, 241, 20))
    ridge = torch.from_numpy(np.stack([ridge_map(d) for d in depths])).to(dev)
    thr = np.linspace(0.01, 0.99, 99)
    N = d_dev.shape[0]

    def canny(per_image, d=d_dev, g=g_dev):
        return sweep_counts(d, g, rng, crop, 0.0, 80.0, max_dist=0.002, per_image=per_image)

    def thin(per_image, p=ridge, g=g_dev):
        return pr_counts(p, g, thr, max_dist=0.0075, crop=crop, apply_thinning=True, per_image=per_image)

    workloads = {
        "canny12": (canny, lambda i: canny(False, d_dev[i:i + 1], g_dev[i:i + 1])),
        "thin99": (thin, lambda i: thin(False, ridge[i:i + 1], g_dev[i:i + 1])),
    }
    res = gpu_facts()
    res.update({"images": N, "warmup": args.warmup, "iters": args.iters, "workloads": []})
    ok = True
    for name, (batched, one) in workloads.items():
        arms = {"summed": lambda: batched(False), "per_image": lambda: batched(True),
                "single": lambda: torch.stack([one(i) for i in range(N)])}
        summed, rows, single = (arms[k]().cpu().numpy() for k in ("summed", "per_image", "single"))
        equal = bool(np.array_equal(rows, single) and np.array_equal(rows.sum(0), summed))
        ok &= equal
        med, runs = time_arms(arms, args.warmup, args.iters)
        row = {"workload": name, "rows_equal": equal, "T": int(rows.shape[1]),
               **{f"{k}_ms": v for k, v in med.items()}, **{f"{k}_runs_ms": v for k, v in runs.items()},
               "per_image_over_summed": med["per_image"] / med["summed"],
               "single_over_per_image": med["single"] / med["per_image"]}
        res["workloads"].append(row)
        print(json.dumps(row), flush=True)
    res["all_rows_equal"] = ok
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    if not ok:
        sys.exit("per-image rows of the arms differ")


if __name__ == "__main__":
    main()
