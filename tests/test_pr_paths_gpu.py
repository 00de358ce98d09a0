"""Every matcher path of the precision/recall counts (``pr_counts.cu``: ``launch``) against the C oracle, bit-exact.

``test_pr_gpu.py`` checks the shipped wiring.  Here each path is reached only through shapes, dtypes, alignment,
crops, radii, thresholds and pixel layout, on the release library:

* tables: offsets and thresholds in the kernel parameters (<= 256 offsets, <= 160 fp thresholds) or staged in the
  workspace (more offsets: radius above ~9 px; more fp thresholds);
* kernels: ``match_sweep_kernel`` (level planes, strength maps with ascending thresholds) with every problem resident,
  in compact mode (more predicted pixels than it holds) and overflowing an image to ``match_kernel`` (more GT pixels);
  ``match_smem_kernel`` (unsorted thresholds, binary maps, T = 1) with problems that fit and problems that overflow to
  ``match_kernel`` in the same call; ``match_kernel`` alone (more than 1024 offsets: radius 19-31 px), also with more
  problems than its 296 persistent arenas;
* the sweep kernel's hard cases: more than 2,048 augmenting roots finding a free GT pixel in one phase (``kEndsCap``),
  an augmenting path of thousands of hops, colliding trees behind a bottleneck, closed forests walled off as DEAD;
* the window scan: the word scan of level planes and the scalar scan (W % 4 != 0, a view one byte into its buffer),
  crops with x0 % 4 != 0; strength values at and around every threshold, NaN, +-Inf, -0.0, subnormals;
* crops with python slice semantics (negative bounds count from the end), and the refusal of a radius >= 32 px.

Every count is checked through the summed call and ``per_image=True`` (whose rows must sum to it) against
``oracle.pr_counts.match_count`` on the numpy-sliced window of every (image, threshold).  ``test_path_manifest``
restates the host planning of ``launch`` and checks that every path above is taken by some case, with every case at
least 10 % away from the boundary it sits next to; it needs no GPU.
"""
import math
import os
import re
import subprocess

import numpy as np
import pytest
import torch

# ---- the host's planning rules (pr_counts.cu: build_offsets / smem_layout / sweep_layout / layout / launch) --------
OPTIN = 232448          # cudaDevAttrMaxSharedMemoryPerBlockOptin of a B200 (227 KB)
NUM_SMS = 148           # B200
STATIC_SMEM = {"match_smem_kernel": 9248, "match_sweep_kernel": 11296}   # cuobjdump --dump-resource-usage, sm_100a
CTAS_PER_SM = 2         # kCtasPerSm: arenas of match_kernel = min(148 * 2, problems)
PARAM_OFF, PARAM_THR = 256, 160      # kParamOff, kParamThr
SMEM_TABLE_OFF = 1024                # kSmemTableOff
ENDS_CAP = 2048                      # kEndsCap
ARENAS = NUM_SMS * CTAS_PER_SM

KITTI_HW = (384, 1280)
KITTI_CROP = [44, 1197, 153, 371]    # window 218 x 1153
KITTI_MD = 0.002                     # radius 2.3469 px, 21 offsets


def radius_of(h, w, max_dist):
    return max_dist * math.sqrt(h * h + w * w)


def n_offsets(radius):
    """build_offsets: None when it refuses (int(radius) > 31)."""
    r = int(radius)
    if r > 31:
        return None
    return sum(1 for dy in range(-r, r + 1) for dx in range(-r, r + 1) if dy * dy + dx * dx <= radius * radius)


def _cap(budget, fixed, per):
    if budget - fixed < 512 * per:
        return 0
    return min((budget - fixed) // per, 0xFFF0) & ~7


def smem_cap(h, w):
    nW = (h * w + 31) // 32
    return _cap(OPTIN - STATIC_SMEM["match_smem_kernel"] - 1024, nW * 4 + (nW * 2 + 15) // 16 * 16 + 256, 20)


def sweep_cap(h, w):
    nW = (h * w + 31) // 32
    return _cap(OPTIN - STATIC_SMEM["match_sweep_kernel"] - 1024, nW * 4 + nW + 2 * ENDS_CAP + 512, 21)


def window(a, crop):
    return a if crop is None else a[crop[2]:crop[3], crop[0]:crop[1]]


def binarise(p, t, thr):
    return (p <= t) if thr is None else (p.astype(np.float64) >= thr[t])


class Case:
    """pred [N,H,W] (u8 level plane when thr is None, else f32/f64 strength map), gt [N,H,W] u8.  binary: the pair is
    handed to correspond_pixels_batch instead (pred = a, gt = b, one problem per plane)."""

    def __init__(self, pred, gt, thr=None, n_levels=None, max_dist=KITTI_MD, crop=None, binary=False, expect=None,
                 misalign=False, max_roots=None):
        self.pred, self.gt, self.thr, self.max_dist, self.crop = pred, gt, thr, max_dist, crop
        self.T = 1 if binary else (n_levels if thr is None else len(thr))
        self.binary, self.expect, self.misalign = binary, expect, misalign
        self.max_roots = max_roots   # hand-derived bound on the augmenting roots of one phase, where one is known

    def windows(self):
        for i in range(self.pred.shape[0]):
            yield window(self.pred[i], self.crop), window(self.gt[i], self.crop) != 0

    def bins(self, p):
        if self.binary:
            return [p != 0]
        return [binarise(p, t, self.thr) for t in range(self.T)]


def oracle_rows(case):
    from oracle import pr_counts as opr
    rows = np.zeros((case.pred.shape[0], case.T, 4), np.int64)
    for i, (p, g) in enumerate(case.windows()):
        if p.size == 0:
            continue
        for t, b in enumerate(case.bins(p)):
            m = opr.match_count(b, g, case.max_dist)
            rows[i, t] = (m, int(g.sum()), m, int(b.sum()))
    return rows


def plan(case):
    """-> (set of path tags, list of boundary problems) of launch() for this call."""
    tags, problems = set(), []
    h, w = window(case.pred[0], case.crop).shape
    noff = n_offsets(radius_of(h, w, case.max_dist))
    levels = case.thr is None and not case.binary
    in_param = noff <= PARAM_OFF and (case.thr is None or case.T <= PARAM_THR)
    tags.add("tables-param" if in_param else "tables-workspace")
    if noff > PARAM_OFF:
        tags.add("offsets-workspace")
    if case.thr is not None and case.T > PARAM_THR:
        tags.add("thresholds-workspace")
    for b in (PARAM_OFF, SMEM_TABLE_OFF):
        if 0.9 * b < noff < 1.1 * b:
            problems.append(("offsets", noff, b))
    scap = smem_cap(h, w)
    use_smem = scap > 0 and noff <= SMEM_TABLE_OFF
    ascending = case.thr is None or all(b > a for a, b in zip(case.thr[:-1], case.thr[1:]))
    sweep = use_smem and not case.binary and case.T > 1 and ascending and sweep_cap(h, w) > 0
    dense = 0
    if sweep:
        cap = sweep_cap(h, w)
        for p, g in case.windows():
            nQ = int(g.sum())
            nPall = int((p < case.T).sum()) if levels else int(binarise(p, 0, case.thr).sum())
            if nQ > cap or nQ >= 0xFFF0 or cap - nQ < 256:
                tags.add("sweep-overflow")
                dense += case.T
            else:
                tags.add("sweep-compact" if nPall > cap else "sweep-resident")
            for v, b in ((nQ, cap), (nQ, cap - 256), (nPall, cap)):
                if 0.9 * b < v < 1.1 * b:
                    problems.append(("sweep capacity", v, b))
    elif use_smem:
        for p, g in case.windows():
            nQ = int(g.sum())
            for b in case.bins(p):
                nP = int(b.sum())
                fits = nP <= scap and nQ <= scap
                tags.add("smem" if fits else "smem-overflow")
                dense += 0 if fits else 1
                for v in (nP, nQ):
                    if 0.9 * scap < v < 1.1 * scap:
                        problems.append(("smem capacity", v, scap))
    else:
        tags.add("dense-only")
        dense = case.pred.shape[0] * case.T
        if dense > ARENAS:
            tags.add("dense-persistent")
    if dense and 0.9 * ARENAS < dense < 1.1 * ARENAS:
        problems.append(("arenas", dense, ARENAS))
    return tags, problems


# ---- inputs ---------------------------------------------------------------------------------------------------------
def contours(H, W, r, n, steps=150):
    gt = np.zeros((H, W), np.uint8)
    for _ in range(n):
        y, x = int(r.integers(0, H)), int(r.integers(0, W))
        for _ in range(steps):
            gt[y, x] = 1
            y = int(np.clip(y + r.integers(-1, 2), 0, H - 1))
            x = int(np.clip(x + r.integers(0, 2), 0, W - 1))
    return gt


def strength_near(gt, r, near_density, salt):
    """A predicted strength map in [0, 1): values near the GT contours plus salt noise (0 elsewhere)."""
    import cv2
    H, W = gt.shape
    near = cv2.dilate(gt, np.ones((5, 5), np.uint8)) > 0
    s = np.where(near & (r.random((H, W)) < near_density), r.random((H, W)), 0.0)
    return np.maximum(s, (r.random((H, W)) < salt) * r.random((H, W)))


def levels_of(strength, T):
    """Level plane: a pixel of strength s > 0 is an edge from level floor((1 - s) * T) on; 255 = never."""
    lv = np.floor((1.0 - strength) * T).astype(np.int64)
    return np.where(strength > 0, np.clip(lv, 0, T - 1), 255).astype(np.uint8)


def kitti_images(seed, n, gt_contours=60, near=0.3, salt=0.003):
    r = np.random.default_rng(seed)
    gts = [contours(*KITTI_HW, r, gt_contours) for _ in range(n)]
    return np.stack([strength_near(g, r, near, salt) for g in gts]), np.stack(gts)


def _thr6():
    return np.array([0.15, 0.3, 0.45, 0.6, 0.75, 0.9])


def case_levels_sweep():
    s, g = kitti_images(1, 2)
    return Case(levels_of(s, 12), g, n_levels=12, crop=KITTI_CROP)


def case_f32_compact_and_resident():
    s, g = kitti_images(2, 2, gt_contours=60, near=0.3, salt=0.002)
    s[1] = np.maximum(s[1], (np.random.default_rng(3).random(KITTI_HW) < 0.06) * 0.95)   # image 1: many pred px
    return Case(s.astype(np.float32), g, thr=_thr6(), crop=KITTI_CROP)


def case_f64_overflow_and_resident():
    s, g = kitti_images(4, 2, gt_contours=60)
    r = np.random.default_rng(5)
    g[0] = np.maximum(g[0], contours(*KITTI_HW, r, 700))     # image 0: more GT px than the sweep kernel holds
    s[0] = np.maximum(s[0], strength_near(g[0], r, 0.2, 0.0))
    return Case(s.astype(np.float64), g, thr=_thr6(), crop=KITTI_CROP)


def case_unsorted_smem_and_overflow():
    s, g = kitti_images(6, 2, gt_contours=60, salt=0.002)
    s[0] = np.maximum(s[0], (np.random.default_rng(7).random(KITTI_HW) < 0.06) * 0.2)    # > capacity at 0.15 only
    return Case(s.astype(np.float32), g, thr=np.array([0.9, 0.15, 0.5]), crop=KITTI_CROP)


def case_levels_offsets_workspace():
    s, g = kitti_images(8, 2, gt_contours=25, near=0.3, salt=0.001)
    return Case(levels_of(s, 12), g, n_levels=12, max_dist=0.0075)          # uncropped 384 x 1280: radius 10.02 px


def small_images(seed, n, H=64, W=100, gt_density=0.25, pred_density=0.3):
    r = np.random.default_rng(seed)
    g = (r.random((n, H, W)) < gt_density).astype(np.uint8)
    s = np.where(r.random((n, H, W)) < pred_density, r.random((n, H, W)), 0.0)
    return s, g


def case_f64_t160_param():
    s, g = small_images(10, 3)
    return Case(s, g, thr=np.linspace(0.002, 0.998, 160), max_dist=0.02)


def case_f64_t161_workspace():
    s, g = small_images(11, 3)
    return Case(s, g, thr=np.linspace(0.002, 0.998, 161), max_dist=0.02)


def case_f32_t254_workspace():
    s, g = small_images(12, 3)
    return Case(s.astype(np.float32), g, thr=np.linspace(0.001, 0.999, 254), max_dist=0.02)


def case_unsorted_t161_workspace():
    s, g = small_images(13, 2)
    thr = np.random.default_rng(14).permutation(np.linspace(0.002, 0.998, 161))
    return Case(s.astype(np.float32), g, thr=thr, max_dist=0.0125)


def case_levels_t1_smem():
    s, g = kitti_images(15, 2)
    return Case(levels_of(s, 1), g, n_levels=1, crop=KITTI_CROP)


def case_binary_param():
    s, g = kitti_images(16, 3)
    return Case((window_stack(s, KITTI_CROP) > 0.3).astype(np.uint8), window_stack(g, KITTI_CROP), binary=True)


def case_binary_workspace_and_overflow():
    s, g = kitti_images(17, 2, gt_contours=25, salt=0.001)
    a = (s > 0.3).astype(np.uint8)
    a[1] |= (np.random.default_rng(18).random(KITTI_HW) < 0.04).astype(np.uint8)     # plane 1 overflows to match_kernel
    return Case(a, g, binary=True, max_dist=0.0075)


def case_binary_dense():
    s, g = small_images(19, 4, H=60, W=80, gt_density=0.1, pred_density=0.1)
    return Case((s > 0).astype(np.uint8), g, binary=True, max_dist=0.195)                     # radius 19.5 px


def window_stack(a, crop):
    return np.ascontiguousarray(a[:, crop[2]:crop[3], crop[0]:crop[1]])


def case_dense_r25_edge():
    s, g = small_images(20, 3, H=60, W=80, gt_density=0.08, pred_density=0.08)
    return Case(levels_of(s, 3), g, n_levels=3, max_dist=0.25)      # radius exactly 25: (7, 24), (15, 20) included


def case_dense_r31():
    s, g = small_images(21, 2, H=60, W=80, gt_density=0.06, pred_density=0.06)
    return Case(s.astype(np.float32), g, thr=np.array([0.2, 0.5, 0.8]), max_dist=0.31)


def case_dense_r31_9():
    s, g = small_images(22, 2, H=60, W=80, gt_density=0.06, pred_density=0.06)
    return Case(s, g, thr=np.array([0.7, 0.1, 0.4]), max_dist=0.319)


def case_dense_persistent():
    s, g = small_images(23, 28, H=60, W=80, gt_density=0.05, pred_density=0.05)
    return Case(levels_of(s, 12), g, n_levels=12, max_dist=0.2)     # 28 x 12 = 336 problems at radius 20 px


PATH_CASES = {f.__name__[5:]: f for f in [
    case_levels_sweep, case_f32_compact_and_resident, case_f64_overflow_and_resident, case_unsorted_smem_and_overflow,
    case_levels_offsets_workspace, case_f64_t160_param, case_f64_t161_workspace, case_f32_t254_workspace,
    case_unsorted_t161_workspace, case_levels_t1_smem, case_binary_param, case_binary_workspace_and_overflow,
    case_binary_dense, case_dense_r25_edge, case_dense_r31, case_dense_r31_9, case_dense_persistent]}


# ---- adversarial matchings for the sweep kernel (KITTI crop, radius 2.35 px: edges at distance 1, sqrt 2, 2, sqrt 5)
WIN_H, WIN_W = 218, 1153


def _plane_from_window(win_levels, win_gt):
    """Embed window planes into a 384 x 1280 plane at the KITTI crop, with salt outside the crop that must not count."""
    r = np.random.default_rng(99)
    lv = np.where(r.random(KITTI_HW) < 0.05, 0, 255).astype(np.uint8)
    g = (r.random(KITTI_HW) < 0.05).astype(np.uint8)
    x0, x1, y0, y1 = KITTI_CROP
    lv[y0:y1, x0:x1] = win_levels
    g[y0:y1, x0:x1] = win_gt
    return lv, g


def greedy_traps(n, split):
    """n gadgets, 8 px apart horizontally and 3 px vertically (no edge between two gadgets).  Gadget at (y, x):
    p2 at x, q1 and p1 at x + 2, q2 at x + 4.  Edges: p1-q1 (0), p1-q2 (2), p2-q1 (2); p2-q2 is 4 px > 2.35.

    Maximum: p1-q2, p2-q1 = 2 per gadget.  Greedy goes nearest first in distance rounds: p1 takes q1 at distance 0
    before p2's round (distance 2) comes, so every p2 is a free root whose only augmenting path is p2 -> q1 -> p1 -> q2,
    and all n roots reach a free GT pixel in the first phase.  split: p1 at level 0, p2 at level 1 (counts n, 2n);
    else both at level 0 (2n, 2n)."""
    lv = np.full((WIN_H, WIN_W), 255, np.uint8)
    g = np.zeros((WIN_H, WIN_W), np.uint8)
    k = 0
    for y in range(1, WIN_H - 1, 3):
        for x in range(1, WIN_W - 5, 8):
            if k == n:
                return lv, g
            lv[y, x] = 1 if split else 0
            lv[y, x + 2] = 0
            g[y, x + 2] = g[y, x + 4] = 1
            k += 1
    raise AssertionError("window too small")


def serpentine(n_points):
    """Lattice points of a path along the window rows 3 apart (right, down 3, left, ...), consecutive points 1 apart."""
    pts, y, x, d = [], 1, 1, 1
    while len(pts) < n_points:
        pts.append((y, x))
        if 1 <= x + d <= WIN_W - 2:
            x += d
        else:
            for _ in range(3):
                y += 1
                pts.append((y, x))
            d = -d
            x += d
    return pts[:n_points]


def long_chain(m):
    """Along a serpentine path, point k is a predicted pixel when k % 3 == 0, a GT pixel when k % 3 == 2, empty
    otherwise; the path ends on a GT pixel.  The head (k = 0) joins at level 1, every other predicted pixel at level 0.

    Every predicted pixel k = 3i (i >= 1) has GT k - 1 at distance 1 and GT k + 2 at distance 2 (or sqrt 2 on a turn);
    no other pair of a predicted and a GT pixel is within 2.35 px (checked in the test).  Level 0: greedy matches every
    predicted pixel to its distance-1 GT neighbour (nobody else is that close), leaving the tail free: m matches.  Level
    1: the head's only GT neighbour is taken, and its only augmenting path runs along the whole chain to the tail:
    m + 1 matches, m + 1 predicted pixels on the path."""
    pts = serpentine(3 * m + 3)
    lv = np.full((WIN_H, WIN_W), 255, np.uint8)
    g = np.zeros((WIN_H, WIN_W), np.uint8)
    for k, (y, x) in enumerate(pts):
        if k % 3 == 0:
            lv[y, x] = 1 if k == 0 else 0
        elif k % 3 == 2:
            g[y, x] = 1
    return lv, g, pts


def checker_block(lv, g, y0, x0, n, level):
    """n x n block, (y + x) even = predicted at `level`, odd = GT: a perfect matching of n * n / 2 pairs (n even)."""
    for y in range(y0, y0 + n):
        for x in range(x0, x0 + n):
            if (y + x) % 2 == 0:
                lv[y, x] = level
            else:
                g[y, x] = 1


def bottlenecks(n_blocks=6, n=20, lanes=3, lane_len=30, roots=16):
    """Blocks of colliding trees.  Each block: an n x n checkerboard (level 0), `lanes` single-file lanes leaving its
    right side (GT, pred, GT, ..., GT: lane_len predicted and lane_len + 1 GT pixels, level 0, rows 6 apart) and
    `roots` predicted pixels at level 1 along its left side.

    Level 0: every predicted pixel is matched (the block perfectly, each lane with one GT pixel to spare): n*n/2 +
    lanes * lane_len per block.  Level 1: every augmenting path ends on one of the `lanes` spare GT pixels at the far
    end of a lane, so the count can grow by at most `lanes` per block, and it does (all GT matched): n*n/2 + lanes *
    (lane_len + 1).  The roots' trees all run into the same block and collide; a lane lets one path through per
    phase, so most roots lose every phase they take part in."""
    lv = np.full((WIN_H, WIN_W), 255, np.uint8)
    g = np.zeros((WIN_H, WIN_W), np.uint8)
    per_row = 4
    for b in range(n_blocks):
        y0, x0 = 4 + (b // per_row) * (n + 12), 4 + (b % per_row) * (n + 2 * lane_len + 20)
        checker_block(lv, g, y0, x0 + 3, n, 0)
        for k in range(roots):               # left of the block, 2 px out: adjacent to GT at (y, x0 + 3) or (y, x0 + 4)
            lv[y0 + k * n // roots, x0 + 1] = 1
        for l in range(lanes):
            y = y0 + 2 + 6 * l
            for j in range(2 * lane_len + 1):
                if j % 2 == 0:
                    g[y, x0 + 3 + n + j] = 1
                else:
                    lv[y, x0 + 3 + n + j] = 0
    per_block0 = n * n // 2 + lanes * lane_len
    return lv, g, (n_blocks * per_block0, n_blocks * (per_block0 + lanes))


def dead_walls(n_blocks=10, n=16):
    """Level 0: checkerboard blocks (perfectly matched).  Level 1: predicted pixels along each block's left side, all
    of whose GT neighbours are matched block pixels: every search fails and the block's forest is walled off (DEAD).
    Level 2: greedy-trap gadgets (as greedy_traps) to the right of each block whose p2 also has a DEAD block GT pixel
    in range: p2 must augment around the wall (p2 -> q1 -> p1 -> q2).  Level 3: a second set of gadgets with p1 at
    level 2 and p2 at level 3.  Per block B = n*n/2 pairs and 2 gadgets of each set:
    counts B, B, B + 4 + 2 (second set's p1 takes its q1), B + 4 + 4 per block."""
    lv = np.full((WIN_H, WIN_W), 255, np.uint8)
    g = np.zeros((WIN_H, WIN_W), np.uint8)
    per_row = 10
    for b in range(n_blocks):
        y0, x0 = 4 + (b // per_row) * (n + 10), 4 + (b % per_row) * (n + 16)
        checker_block(lv, g, y0, x0 + 2, n, 0)
        for y in range(y0, y0 + n, 2):
            lv[y, x0] = 1
        xr = x0 + 2 + n - 1            # the block's last column
        for k, y in enumerate((y0 + 1, y0 + 5, y0 + 9, y0 + 13)):
            # p2 two px right of the block (the block pixel at (y, xr) is GT when (y + xr) is odd)
            if (y + xr) % 2 == 0:
                y += 1
            first = k < 2
            lv[y, xr + 2] = 2 if first else 3
            lv[y, xr + 4] = 2
            g[y, xr + 4] = g[y, xr + 6] = 1
    B = n * n // 2
    return lv, g, [n_blocks * c for c in (B, B, B + 6, B + 8)]


def adjacency(pred_mask, gt_mask, radius):
    """Edges (pred index, gt index) of the matching graph, by brute force over the offsets."""
    r = int(radius)
    py, px = np.nonzero(pred_mask)
    gi = -np.ones(gt_mask.shape, np.int64)
    gi[gt_mask] = np.arange(int(gt_mask.sum()))
    edges = []
    H, W = gt_mask.shape
    for dy in range(-r, r + 1):
        for dx in range(-r, r + 1):
            if dy * dy + dx * dx > radius * radius:
                continue
            y, x = py + dy, px + dx
            ok = (y >= 0) & (y < H) & (x >= 0) & (x < W)
            j = np.full(len(py), -1)
            j[ok] = gi[y[ok], x[ok]]
            for i in np.nonzero(j >= 0)[0]:
                edges.append((int(i), int(j[i])))
    return edges


def case_greedy_traps():
    a, ga = greedy_traps(3000, True)
    b, gb = greedy_traps(3000, False)
    (la, pa), (lb, pb) = _plane_from_window(a, ga), _plane_from_window(b, gb)
    return Case(np.stack([la, lb]), np.stack([pa, pb]), n_levels=2, crop=KITTI_CROP,
                expect=np.array([[3000, 6000], [6000, 6000]]), max_roots=3000)


def case_long_chain():
    lv, g, _ = long_chain(2400)
    lv, g = _plane_from_window(lv, g)
    # level 0 is matched by the greedy start alone (no root), level 1 has one root
    return Case(lv[None], g[None], n_levels=2, crop=KITTI_CROP, expect=np.array([[2400, 2401]]), max_roots=1)


def case_bottlenecks():
    win, g, counts = bottlenecks()
    lv, g = _plane_from_window(win, g)
    # at most every predicted pixel of a level is a root
    return Case(lv[None], g[None], n_levels=2, crop=KITTI_CROP, expect=np.array([counts]),
                max_roots=int(np.bincount(win[win < 2]).max()))


def case_dead_walls():
    lv, g, counts = dead_walls()
    lv, g = _plane_from_window(lv, g)
    return Case(lv[None], g[None], n_levels=4, crop=KITTI_CROP, expect=np.array([counts]))


def case_random_stress_levels():
    s, g = small_images(30, 4, gt_density=0.3, pred_density=0.35)
    return Case(levels_of(s, 254), g, n_levels=254, max_dist=0.02)


def case_random_stress_f64():
    s, g = small_images(31, 4, gt_density=0.3, pred_density=0.35)
    return Case(s, g, thr=np.linspace(0.001, 0.999, 254), max_dist=0.0125)


ADVERSARIAL = {f.__name__[5:]: f for f in [case_greedy_traps, case_long_chain, case_bottlenecks, case_dead_walls,
                                          case_random_stress_levels, case_random_stress_f64]}


# ---- scan and value edges -------------------------------------------------------------------------------------------
def case_scan_w_mod4(m):
    s, g = small_images(40 + m, 3, H=70, W=96 + m, gt_density=0.1, pred_density=0.12)
    return Case(levels_of(s, 9), g, n_levels=9, max_dist=0.02)


def case_scan_misaligned():
    s, g = small_images(44, 3, H=70, W=96, gt_density=0.1, pred_density=0.12)
    return Case(levels_of(s, 9), g, n_levels=9, max_dist=0.02, misalign=True)


def scan_crops():
    W = 124
    return [[1, 101, 3, 60], [2, W, 0, 70], [3, 97, 5, 66], [W - 1, W, 0, 70], [5, W, 7, 70]]


def case_scan_crop(k):
    s, g = small_images(50 + k, 2, H=70, W=124, gt_density=0.1, pred_density=0.12)
    return Case(levels_of(s, 9), g, n_levels=9, max_dist=0.02, crop=scan_crops()[k])


def value_planes(dtype, thr):
    """Every threshold, its fp64 neighbours (and, for fp32 maps, its fp32 neighbours), specials, subnormals."""
    r = np.random.default_rng(60)
    vals = [np.nan, np.inf, -np.inf, -0.0, 0.0, 5e-324, -5e-324, 2.2250738585072014e-308, 1e-45, 1.0, -1.0]
    for t in thr:
        vals += [t, np.nextafter(t, np.inf), np.nextafter(t, -np.inf)]
        f = np.float32(t)
        vals += [float(f), float(np.nextafter(f, np.float32(np.inf))), float(np.nextafter(f, np.float32(-np.inf)))]
    vals = np.array(vals, np.float64)
    p = r.choice(vals, size=(3, 60, 90))
    p = np.where(r.random(p.shape) < 0.6, p, np.nan)       # keep the predicted sets sparse (NaN is never set)
    g = (r.random((3, 60, 90)) < 0.15).astype(np.uint8)
    return p.astype(dtype), g


VALUE_THR = np.array([-1e-300, 0.0, 5e-324, 0.1, 1.0 / 3.0, 0.5, 0.7, 1.0])   # 0.1, 1/3, 0.7 are not fp32 values


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("order", ["ascending", "unsorted"])
@pytest.mark.gpu
def test_strength_values_on_and_around_thresholds(dtype, order):
    """pred >= thr[t] in fp64: -0.0 >= 0.0, subnormals, +-Inf, NaN never set, fp32 values against fp64 thresholds
    that fp32 cannot represent.  Ascending thresholds take the sweep kernel's bisection, unsorted ones the per-problem
    comparison."""
    thr = VALUE_THR if order == "ascending" else VALUE_THR[[3, 0, 7, 5, 1, 6, 2, 4]]
    p, g = value_planes(dtype, VALUE_THR)
    case = Case(p, g, thr=thr, max_dist=0.02)
    assert "sweep-resident" in plan(case)[0] if order == "ascending" else "smem" in plan(case)[0]
    _check(case)
    assert float(np.float32(0.1)) != 0.1 and (p == 0.0).any() and np.signbit(p[p == 0.0]).any()


# ---- running a case -------------------------------------------------------------------------------------------------
def _device(a, misalign):
    t = torch.from_numpy(np.ascontiguousarray(a))
    if not misalign:
        return t.cuda()
    buf = torch.empty(t.numel() * t.element_size() + 1, dtype=torch.uint8, device="cuda")
    v = buf[1:].view(t.dtype).view(t.shape) if t.element_size() == 1 else None
    assert v is not None
    v.copy_(t.cuda())
    assert v.data_ptr() % 4 != 0
    return v


def _device_counts(case, per_image, crop=None, thinning=False):
    from mindtheedge_b200.eval_depth_edges import pr_counts
    d = _device(case.pred, case.misalign)
    g = torch.from_numpy(case.gt).cuda()
    kw = dict(max_dist=case.max_dist, crop=case.crop if crop is None else crop, apply_thinning=thinning,
              per_image=per_image)
    if case.thr is None:
        return pr_counts(d, g, n_levels=case.T, **kw).cpu().numpy()
    return pr_counts(d, g, case.thr, **kw).cpu().numpy()


def _check(case):
    ref = oracle_rows(case)
    if case.binary:
        from mindtheedge_b200.eval_depth_edges import correspond_pixels_batch
        a, b = torch.from_numpy(case.pred).cuda(), torch.from_numpy(case.gt).cuda()
        ma, mb, cnt = (x.cpu().numpy() for x in correspond_pixels_batch(a, b, case.max_dist))
        assert np.array_equal(cnt, ref[:, 0, 0]), (cnt, ref[:, 0, 0])
        for k in range(len(cnt)):
            assert ma[k].sum() == cnt[k] and mb[k].sum() == cnt[k]
            assert not (ma[k] & ~(case.pred[k] != 0)).any() and not (mb[k] & ~(case.gt[k] != 0)).any()
        return ref
    rows = _device_counts(case, True)
    summed = _device_counts(case, False)
    assert np.array_equal(rows, ref), [(i, t, rows[i, t].tolist(), ref[i, t].tolist())
                                       for i, t in zip(*np.nonzero((rows != ref).any(2)))][:10]
    assert np.array_equal(rows.sum(0), summed)
    return ref


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(PATH_CASES))
def test_path_matrix(name):
    case = PATH_CASES[name]()
    tags, problems = plan(case)
    assert not problems, problems
    _check(case)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(ADVERSARIAL))
def test_adversarial_matchings(name):
    """Each gadget family's hand-derived count (see its builder) equals match_count, match_count_scipy and the
    kernel, at every level."""
    from oracle import pr_counts as opr
    case = ADVERSARIAL[name]()
    assert plan(case)[0] & {"sweep-resident"}, plan(case)
    _adversarial_preconditions(name, case)
    ref = _check(case)
    if case.expect is not None:
        assert np.array_equal(ref[:, :, 0], case.expect), (ref[:, :, 0], case.expect)
        for i, (p, g) in enumerate(case.windows()):
            for t, b in enumerate(case.bins(p)):
                assert opr.match_count_scipy(b, g, case.max_dist) == case.expect[i, t], (i, t)


def _adversarial_preconditions(name, case):
    """The property each family exists for, asserted on its input."""
    h, w = window(case.pred[0], case.crop).shape
    radius = radius_of(h, w, case.max_dist)
    if name == "greedy_traps":
        # split image: level 1 brings 3000 free roots, each with its own free GT pixel at the end of a 3-hop path
        p, g = next(case.windows())
        roots = int((p == 1).sum())
        assert roots >= 1.1 * ENDS_CAP and n_offsets(radius) == 21
        assert len(adjacency(p <= 1, g, radius)) == 3 * roots          # exactly the three edges of every gadget
    elif name == "long_chain":
        p, g = next(case.windows())
        e = adjacency(p <= 1, g, radius)
        n_p, n_q = int((p <= 1).sum()), int(g.sum())
        # a simple path: head of degree 1, every other predicted pixel of degree 2, connected without cycles
        assert len(e) == 2 * n_p - 1 and n_q == n_p and n_p - 1 >= 1000
        deg = np.bincount([i for i, _ in e], minlength=n_p)
        assert (deg == 1).sum() == 1 and (deg == 2).sum() == n_p - 1
        parent = list(range(n_p + n_q))

        def find(x):
            while parent[x] != x:
                parent[x] = parent[parent[x]]
                x = parent[x]
            return x
        for i, j in e:
            a, b = find(i), find(n_p + j)
            assert a != b          # a tree with n_p + n_q - 1 edges is a path here
            parent[a] = b
    elif name == "bottlenecks":
        p, g = next(case.windows())
        assert int((p == 1).sum()) >= 4 * 3 * 6       # roots per block well beyond its lanes
    elif name == "dead_walls":
        p, g = next(case.windows())
        # every level-1 pixel has GT neighbours, all inside a block
        e = adjacency(p == 1, g, radius)
        assert len({i for i, _ in e}) == int((p == 1).sum())
    elif name.startswith("random_stress"):
        assert case.T == 254 and h * w == 6400


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 2, 3])
def test_scan_width_not_multiple_of_4(k):
    """W % 4 != 0: level planes are read pixel by pixel instead of as 32-bit words."""
    _check(case_scan_w_mod4(k))


@pytest.mark.gpu
def test_scan_view_one_byte_into_buffer():
    """A 4-aligned width through a view whose base is not 4-byte aligned: the scalar scan."""
    _check(case_scan_misaligned())


@pytest.mark.gpu
@pytest.mark.parametrize("k", range(len(scan_crops())))
def test_scan_crop_offsets(k):
    """Word scan with x0 % 4 in {1, 2, 3}, x1 = W, and a one-column window x0 = W - 1."""
    _check(case_scan_crop(k))


@pytest.mark.gpu
@pytest.mark.parametrize("max_dist,noff", [(0.005, 1), (0.01, 5)])
def test_radius_below_and_at_one(max_dist, noff):
    """Radius 0.5 px: only coincident pixels match; radius exactly 1 px: the four neighbours at distance 1 too."""
    assert n_offsets(radius_of(60, 80, max_dist)) == noff
    s, g = small_images(70, 3, H=60, W=80, gt_density=0.3, pred_density=0.3)
    _check(Case(levels_of(s, 5), g, n_levels=5, max_dist=max_dist))
    _check(Case(s, g, thr=np.array([0.6, 0.2]), max_dist=max_dist))


@pytest.mark.gpu
def test_radius_32_is_refused():
    """build_offsets refuses radius >= 32 px (int(radius) > 31): the call raises instead of returning counts."""
    from mindtheedge_b200.eval_depth_edges import correspond_pixels_batch, pr_counts
    assert n_offsets(radius_of(60, 80, 0.32)) is None and n_offsets(radius_of(60, 80, 0.319)) is not None
    s, g = small_images(71, 1, H=60, W=80)
    d, gg = torch.from_numpy(levels_of(s, 3)).cuda(), torch.from_numpy(g).cuda()
    with pytest.raises(RuntimeError, match=r"code -4"):
        pr_counts(d, gg, n_levels=3, max_dist=0.32)
    with pytest.raises(RuntimeError, match=r"code -4"):
        correspond_pixels_batch((d < 3).to(torch.uint8), gg, 0.32)
    torch.cuda.synchronize()


# ---- crop semantics -------------------------------------------------------------------------------------------------
CROPS = [[4, -3, 6, -4], [-120, -3, -60, 50], [-500, 90, 2, 500], [10, 140, -1000, -5], [90, 30, 5, 60],
         [0, 0, 0, 70], [-5, 200, 3, 3], [130, 200, 0, 70]]


@pytest.mark.gpu
@pytest.mark.parametrize("thinning", [False, True])
def test_crop_python_slice_semantics(thinning):
    """Negative bounds count from the end of the axis, bounds beyond the plane clamp, x0 > x1 is an empty window:
    exactly numpy's plane[y0:y1, x0:x1], as the reference crops.  Unthinned and thinned, summed and per image."""
    from oracle import pr_counts as opr
    from oracle import thin as othin
    s, g = small_images(80, 2, H=70, W=124, gt_density=0.1, pred_density=0.12)
    lv = levels_of(s, 4)
    gt_seen = 0
    for crop in CROPS:
        case = Case(lv, g, n_levels=4, max_dist=0.02, crop=crop)
        ref = np.zeros((2, 4, 4), np.int64)
        for i, (p, q) in enumerate(case.windows()):
            if p.size == 0:
                continue
            for t, b in enumerate(case.bins(p)):
                if thinning:
                    b = othin.binary_thin(b)
                m = opr.match_count(b, q, case.max_dist)
                ref[i, t] = (m, int(q.sum()), m, int(b.sum()))
        rows = _device_counts(case, True, thinning=thinning)
        assert np.array_equal(rows, ref), (crop, rows.tolist(), ref.tolist())
        assert np.array_equal(_device_counts(case, False, thinning=thinning), ref.sum(0)), crop
        gt_seen += int(ref[:, :, 1].sum())
    assert gt_seen > 0


@pytest.mark.gpu
def test_crop_negative_bounds_sweep_counts_and_pr_evaluation(tmp_path):
    """The reference's negative-bound crop through sweep_counts (level planes of the Canny sweep) against the oracle's
    pr_evaluation, and through pr_evaluation(per_image=True) against _pred_eval on the same list crop."""
    import cv2
    from synth import scene_with_gt
    from mindtheedge_b200.edge import canny_from_depth
    from mindtheedge_b200.eval_depth_edges import _pred_eval, pr_evaluation, sweep_counts
    from oracle import pr_counts as opr
    crop = [44, -83, 153, -4]
    gts, depths = zip(*[scene_with_gt(384, 1280, 300 + k) for k in range(2)])
    rng = [40, 120, 200]
    c = sweep_counts(torch.from_numpy(np.stack(depths)).cuda(), torch.from_numpy(np.stack(gts) > 127).to(
        torch.uint8).cuda(), rng, crop, 0.0, 80.0, max_dist=0.002).cpu().numpy()
    ref = opr.pr_sweep_counts(depths, gts, rng, crop)
    assert np.array_equal(c, ref), (c.tolist(), ref.tolist())
    assert ref[:, 0].min() > 100
    gp, dp = str(tmp_path / "gt.png"), str(tmp_path / "pred.npy")
    cv2.imwrite(gp, gts[0])
    np.save(dp, depths[0])
    _, _, results = pr_evaluation([gp], [dp], edge_thresh_range=rng, gt_crop=crop, per_image=True)
    for k, t in enumerate(rng):
        e = canny_from_depth(torch.from_numpy(depths[0]).cuda(), [(int(t / 2), int(t))])[0].cpu().numpy()
        pe = str(tmp_path / f"pe{k}.png")
        cv2.imwrite(pe, e)
        want = _pred_eval(pe, gp, str(crop))
        got = results[0][k]
        for f in ("count_r_overall", "sum_r_overall", "count_p_overall", "sum_p_overall", "recall", "precision"):
            assert np.array_equal(getattr(got, f), getattr(want, f)), (t, f, getattr(got, f), getattr(want, f))
        assert want.sum_p_overall[0] > 0


# ---- coverage manifest (no GPU work) --------------------------------------------------------------------------------
def _margin_ok(value, boundary):
    return value <= 0.9 * boundary or value >= 1.1 * boundary


def test_static_shared_memory_pins():
    """The pinned static shared memory of the matcher kernels equals what the built library declares."""
    from mindtheedge_b200 import _lib
    out = subprocess.run(["cuobjdump", "--dump-resource-usage", _lib.LIB_PATH], capture_output=True,
                         text=True).stdout
    for name, pinned in STATIC_SMEM.items():
        m = re.search(r"Function _ZN3mte2pr\d+" + name + r"E\S*:\s*\n\s*REG:\d+ STACK:\d+ SHARED:(\d+)", out)
        assert m, name
        assert int(m.group(1)) == pinned, (name, int(m.group(1)), pinned)


def test_path_manifest():
    """Every path of launch() is taken by some case, every case is at least 10 % away from the boundaries it sits next
    to (256 / 1024 offsets, the sweep and shared-memory capacities, capP - nQ >= 256, the 296 arenas, 2,048 ends),
    and the numbers the boundaries come from are the ones derived by hand.  The 160-threshold boundary is straddled on
    purpose (T = 160 in the parameters, T = 161 in the workspace)."""
    from oracle import pr_counts as opr
    assert sweep_cap(WIN_H, WIN_W) == 8392 and smem_cap(WIN_H, WIN_W) == 8736 and sweep_cap(384, 1280) == 6600
    assert n_offsets(radius_of(WIN_H, WIN_W, KITTI_MD)) == 21 and n_offsets(radius_of(384, 1280, 0.0075)) == 317
    assert n_offsets(18.0) == 1009 and n_offsets(19.5) > 1.1 * SMEM_TABLE_OFF and n_offsets(25.0) == 1961
    seen, problems = set(), []
    cases = {**{("path", k): f for k, f in PATH_CASES.items()}, **{("adv", k): f for k, f in ADVERSARIAL.items()}}
    cases.update({("scan", k): (lambda k=k: case_scan_w_mod4(k)) for k in (1, 2, 3)})
    cases.update({("crop", k): (lambda k=k: case_scan_crop(k)) for k in range(len(scan_crops()))})
    cases[("scan", "misaligned")] = case_scan_misaligned
    for key, build in cases.items():
        case = build()
        tags, probs = plan(case)
        seen |= tags
        problems += [(key,) + p for p in probs]
        if "sweep-resident" in tags or "sweep-compact" in tags:
            # ends recorded in one phase <= matches gained in one stage (one augmenting path per recorded end)
            # (the images the sweep kernel keeps), unless the family states a tighter bound on its roots
            gain = case.max_roots
            if gain is None:
                ref = oracle_rows(case)
                cap = sweep_cap(*window(case.pred[0], case.crop).shape)
                kept = [i for i, (p, g) in enumerate(case.windows()) if int(g.sum()) <= cap - 256]
                c = ref[kept, :, 0] if case.thr is None else ref[kept, ::-1, 0]
                gain = int(np.diff(c, axis=1, prepend=0).max())
            if gain > 0.9 * ENDS_CAP:
                seen.add("ends-cap")
                if key != ("adv", "greedy_traps"):
                    problems.append((key, "ends", gain))
        if tags & {"sweep-resident", "sweep-compact", "sweep-overflow"} and case.thr is None:
            # level planes are scanned as 32-bit words when the plane width and the base allow it
            W = case.pred.shape[2]
            words = W % 4 == 0 and not case.misalign
            seen.add("scan-words" if words else "scan-scalar")
            if words and case.crop is not None and slice(*case.crop[:2]).indices(W)[0] % 4:
                seen.add("scan-crop-x0%4")
    assert not problems, problems
    want = {"tables-param", "tables-workspace", "offsets-workspace", "thresholds-workspace", "sweep-resident",
            "sweep-compact", "sweep-overflow", "smem", "smem-overflow", "dense-only", "dense-persistent", "ends-cap",
            "scan-words", "scan-scalar", "scan-crop-x0%4"}
    assert want <= seen, sorted(want - seen)
    assert opr.match_radius((60, 80), 0.25) == 25.0 and opr.match_radius((60, 80), 0.31) == 31.0


@pytest.mark.gpu
def test_manifest_constants_match_device():
    p = torch.cuda.get_device_properties(0)
    assert p.shared_memory_per_block_optin == OPTIN and p.multi_processor_count == NUM_SMS
