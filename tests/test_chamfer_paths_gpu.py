"""Every kernel path of the light edge metric (``chamfer.cu``: ``mte_chamfer_counts``) against ``oracle.chamfer``
(scipy's exact EDT) and a brute-force integer d^2 oracle, counts and the int8 map bit for bit.

``test_chamfer_gpu.py`` checks the goldens and one KITTI batch.  Here:

* shapes: W = 1, 31, 256, 257 (``row_eval_kernel`` walks a row in strides of 256 threads), 1280, 1936; H = 1;
  batches of up to 8 images with mixed content;
* per image in one batch: no GT (scipy measures from row -1, column 0), no pred, both empty, GT everywhere,
  pred == GT;
* long searches: a single GT pixel in a corner under a dense pred (the column search runs the whole width), GT in
  one row only, H = 65,533 (the largest accepted) with distances up to 65,532;
* the H and W limits: W = 24,481 .. 24,576 needs more than the 48 KB of shared memory a launch gets without the
  opt-in; H = 65,534 and W = 24,577 are refused;
* thresholds that fall exactly on a distance (5 with 3-4-5 offsets, sqrt 2, sqrt 8), 0, 0.5, 1, large, inf;
* binarisation at 127 / 128 (u8), 127.49 / 127.5 / 127.51 (float64 ``chamfer_distance``), GT at and next to 0.5
  (float32 and float64 ``compute_edge_metrics``);
* the distance sum against ``math.fsum`` within the bound of the kernel's summation order, and bit-identical
  repeats;
* ``compute_edge_metrics`` at KITTI and DDAD size with and without a crop, and its ``edge_model`` branch.

``test_path_manifest`` restates the launch of ``mte_chamfer_counts`` and checks that every path is taken by some
case; ``test_brute_force_oracle_vs_scipy`` pins the brute-force oracle.  Neither needs a GPU.
"""
import math

import numpy as np
import pytest
import torch
from scipy import ndimage

THREADS = 256            # kThreads of row_eval_kernel: one CTA per row, columns x, x + 256, ...
STATIC_SMEM = 192        # row_eval_kernel's static shared memory (ptxas --resource-usage, sm_100a)
DEFAULT_SMEM = 48 * 1024
MAX_H, MAX_W = 65533, 24 * 1024
U = 2.0 ** -53


# ---- oracles --------------------------------------------------------------------------------------------------------
def brute_d2(gt):
    """Integer squared distance of every pixel to the nearest set pixel of gt [H,W] bool; without any, scipy's
    convention: (y + 1)^2 + x^2."""
    H, W = gt.shape
    y, x = np.mgrid[0:H, 0:W]
    gy, gx = np.nonzero(gt)
    if len(gy) == 0:
        return (y + 1) ** 2 + x ** 2
    d = (y[..., None] - gy) ** 2 + (x[..., None] - gx) ** 2
    return d.min(-1)


def is_set(a):
    return (np.asarray(a) / 255) > 0.5


def reference(pred, gt, thresh):
    """pred, gt: [N,H,W] -> per image (exact distance sum, n, close), int8 map, and the distances themselves."""
    rows, cond, dists = [], np.full(pred.shape, -1, np.int8), []
    for i in range(pred.shape[0]):
        p, g = is_set(pred[i]), is_set(gt[i])
        dist = ndimage.distance_transform_edt(~g)
        d = dist[p]
        dists.append(d)
        rows.append((math.fsum(d.tolist()), int(p.sum()), int((d < thresh).sum())))
        cond[i][p] = (d < thresh).astype(np.int8)
    return rows, cond, dists


def sum_bound(H, W):
    """Relative error bound of the kernel's distance sum: u times the longest chain of additions a term goes
    through (per thread W / 256 columns, the warp butterfly, the 8 warps of the CTA in order, H / 32 rows per lane
    in finish_kernel, its warp butterfly), plus one u for the rounding of the exact sum."""
    chain = math.ceil(W / THREADS) + 5 + THREADS // 32 + math.ceil(H / 32) + 5
    return (chain + 1) * U


# ---- cases ----------------------------------------------------------------------------------------------------------
class Case:
    def __init__(self, pred, gt, thresh=5.0, brute=None):
        self.pred, self.gt, self.thresh = pred.astype(np.uint8), gt.astype(np.uint8), thresh
        self.brute = pred.shape[1] * pred.shape[2] <= 4096 if brute is None else brute


def rand_planes(r, N, H, W, pd, gd):
    p = (r.random((N, H, W)) < pd).astype(np.uint8) * 255
    g = (r.random((N, H, W)) < gd).astype(np.uint8) * 255
    return p, g


def case_width(W, N=3, H=24):
    r = np.random.default_rng(W)
    p, g = rand_planes(r, N, H, W, 0.2, 0.02)
    return Case(p, g)


def case_h1():
    r = np.random.default_rng(1)
    p, g = rand_planes(r, 4, 1, 300, 0.3, 0.02)
    g[1] = 0
    return Case(p, g)


def case_mixed_empty():
    """One batch: normal, no GT, no pred, both empty, GT everywhere, pred == GT, a single pred pixel, normal."""
    r = np.random.default_rng(2)
    p, g = rand_planes(r, 8, 40, 300, 0.1, 0.03)
    g[1] = 0
    p[2] = 0
    p[3] = g[3] = 0
    g[4] = 255
    p[5] = g[5]
    p[6] = 0
    p[6, 39, 299] = 255
    return Case(p, g)


def case_corner_gt():
    """Dense pred, one GT pixel at (0, 0): every pixel's column search runs out to column 0."""
    p = np.full((2, 64, 1936), 255, np.uint8)
    g = np.zeros_like(p)
    g[0, 0, 0] = 255
    g[1, 63, 1935] = 255
    return Case(p, g)


def case_gt_one_row():
    r = np.random.default_rng(3)
    p, _ = rand_planes(r, 2, 200, 700, 0.2, 0.0)
    g = np.zeros_like(p)
    g[0, 150, r.integers(0, 700, 5)] = 255
    g[1, 0, :] = 255
    return Case(p, g)


def case_tall():
    """H = 65,533: GT in row 0 only (distances up to 65,532), and an image without GT (up to 65,533 from row -1)."""
    H, W = MAX_H, 5
    p = np.zeros((2, H, W), np.uint8)
    p[:, ::97] = 255
    p[:, -1] = 255
    g = np.zeros_like(p)
    g[0, 0, 2] = 255
    return Case(p, g, thresh=60000.0)


def case_wide(W):
    r = np.random.default_rng(W)
    p, g = rand_planes(r, 2, 3, W, 0.05, 0.001)
    g[1] = 0
    g[1, 2, W - 1] = 255       # one GT pixel at the far end of image 1: searches across the whole row
    return Case(p, g)


def exact_distance_planes():
    """Two images of isolated GT pixels, each with pred pixels at offsets (3, 4), (1, 1), (2, 2), (0, 0), (0, 1),
    (1, 2), far apart from the other groups, so every distance is exactly one of 5, sqrt 2, sqrt 8, 0, 1, sqrt 5."""
    p = np.zeros((2, 60, 200), np.uint8)
    g = np.zeros_like(p)
    offsets = [(3, 4), (1, 1), (2, 2), (0, 0), (0, 1), (1, 2), (-4, 3), (4, -3)]
    for i in range(2):
        for k, (dy, dx) in enumerate(offsets):
            y, x = 20 + 20 * (k // 6) + 5 * i, 15 + 30 * (k % 6)
            g[i, y, x] = 255
            p[i, y + dy, x + dx] = 255
    return p, g


THRESHOLDS = [5.0, math.sqrt(2), math.sqrt(8), 0.0, 0.5, 1.0, 1e9, math.inf]


CASES = {
    **{f"w{W}": (lambda W=W: case_width(W)) for W in (1, 31, 256, 257, 1280, 1936)},
    "h1": case_h1, "mixed_empty": case_mixed_empty, "corner_gt": case_corner_gt, "gt_one_row": case_gt_one_row,
    "tall": case_tall, **{f"wide{W}": (lambda W=W: case_wide(W)) for W in (24480, 24481, 24576)},
}


# ---- the launch of mte_chamfer_counts, restated ---------------------------------------------------------------------
def plan(case):
    N, H, W = case.pred.shape
    if H > MAX_H or W > MAX_W:
        return {"refused"}
    tags = {"row-one-stride" if W <= THREADS else "row-strides", "finish-one-row" if H <= 32 else "finish-rows"}
    if 2 * W + STATIC_SMEM > DEFAULT_SMEM:
        tags.add("smem-opt-in")
    for i in range(N):
        g, p = is_set(case.gt[i]), is_set(case.pred[i])
        tags.add("gt" if g.any() else "no-gt")
        tags.add("pred" if p.any() else "no-pred")
        if g.all():
            tags.add("gt-everywhere")
        if p.any() and (p == g).all():
            tags.add("pred-is-gt")
        if g.any() and p.any():
            # longest column search: the farthest nearest-GT column of a pred pixel in its row
            cols = np.nonzero(g.any(0))[0]
            px = np.nonzero(p.any(0))[0]
            if np.abs(px[:, None] - cols[None]).min(1).max() >= W - 1 and W > 1000:
                tags.add("search-full-width")
    if H == MAX_H:
        tags.add("h-max")
    return tags


# ---- running --------------------------------------------------------------------------------------------------------
def _counts(pred, gt, thresh):
    from mindtheedge_b200.edge import chamfer_counts
    out, cond = chamfer_counts(torch.from_numpy(pred).cuda(), torch.from_numpy(gt).cuda(), thresh, want_map=True)
    return out.cpu().numpy(), cond.cpu().numpy()


def _check(case, thresh=None):
    t = case.thresh if thresh is None else thresh
    N, H, W = case.pred.shape
    rows, cond_ref, dists = reference(case.pred, case.gt, t)
    out, cond = _counts(case.pred, case.gt, t)
    assert np.array_equal(cond, cond_ref), np.argwhere(cond != cond_ref)[:5].tolist()
    bound = sum_bound(H, W)
    for i, (s, n, close) in enumerate(rows):
        assert out[i, 1] == n and out[i, 2] == close and out[i, 3] == 0, (i, out[i].tolist(), (n, close))
        assert abs(out[i, 0] - s) <= bound * s, (i, out[i, 0], s, bound)
        if case.brute:
            d2 = brute_d2(is_set(case.gt[i]))[is_set(case.pred[i])]
            assert np.array_equal(np.sqrt(d2.astype(np.float64)), dists[i]), i
    again, cond2 = _counts(case.pred, case.gt, t)
    assert np.array_equal(again, out) and np.array_equal(cond2, cond)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_path_matrix(name):
    case = CASES[name]()
    assert "refused" not in plan(case)
    out = _check(case)
    if name == "tall":
        assert out[0, 1] > 0 and out[0, 2] < out[0, 1]      # some distances beyond 60,000
    if name == "mixed_empty":
        assert out[2, 1] == 0 and out[3, 1] == 0 and out[2, 0] == 0 and out[4, 0] == 0 and out[5, 0] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("N,H,W", [(1, MAX_H + 1, 4), (1, 3, MAX_W + 1), (2, 70000, 2)])
def test_limits_refused(N, H, W):
    from mindtheedge_b200.edge import chamfer_counts
    z = torch.zeros((N, H, W), dtype=torch.uint8, device="cuda")
    with pytest.raises(RuntimeError, match=r"code -2"):
        chamfer_counts(z, z)
    torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("thresh", THRESHOLDS)
def test_thresholds_on_exact_distances(thresh):
    p, g = exact_distance_planes()
    _, _, dists = reference(p, g, thresh)
    assert sorted(set(np.round(dists[0] ** 2).astype(int).tolist())) == [0, 1, 2, 5, 8, 25]
    out = _check(Case(p, g, thresh=thresh, brute=True))
    want_close = {5.0: 5, math.sqrt(2): 2, math.sqrt(8): 4, 0.0: 0, 0.5: 1, 1.0: 1, 1e9: 8, math.inf: 8}[thresh]
    assert out[:, 2].tolist() == [want_close, want_close], (thresh, out[:, 2])


@pytest.mark.gpu
def test_binarisation_u8_127_128():
    r = np.random.default_rng(4)
    vals = np.array([0, 127, 128, 255], np.uint8)
    p = r.choice(vals, (3, 50, 270), p=[0.6, 0.15, 0.15, 0.1])
    g = r.choice(vals, (3, 50, 270), p=[0.9, 0.04, 0.04, 0.02])
    assert is_set(128) and not is_set(127)
    _check(Case(p, g))


@pytest.mark.gpu
def test_chamfer_distance_float64_binarisation():
    """chamfer_distance on float64 maps: 127.5 / 255 is exactly 0.5 (not set), 127.51 is set, 127.49 is not."""
    from mindtheedge_b200.edge import chamfer_distance
    from oracle import chamfer as och
    r = np.random.default_rng(5)
    vals = np.array([0.0, 127.49, 127.5, 127.51, 255.0])
    p = r.choice(vals, (60, 300), p=[0.6, 0.1, 0.1, 0.1, 0.1])
    g = r.choice(vals, (60, 300), p=[0.88, 0.03, 0.03, 0.03, 0.03])
    c, pc, cond = chamfer_distance(p, g)
    _, rpc, close, n = och.chamfer_distance(p, g)
    (s, _, _), = reference(p[None], g[None], 5)[0]
    assert pc == rpc and abs(c - s / n) <= (sum_bound(60, 300) + 2 * U) * (s / n)
    _, cond_ref, _ = reference(p[None], g[None], 5)
    assert np.array_equal(cond, cond_ref[0].astype(np.float64))
    assert int((cond >= 0).sum()) == n == int(((p == 127.51) | (p == 255)).sum())
    # no pred pixel: NaN mean and share, as the reference divides by zero
    c0, pc0, cond0 = chamfer_distance(np.where(p == 127.5, p, 0.0), g)
    assert np.isnan(c0) and np.isnan(pc0) and (cond0 == -1).all()


def _metrics_eq(got, want):
    assert np.array_equal(np.array(got, np.float64), np.array(want, np.float64), equal_nan=True), (got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("size,crop", [((384, 1280), None), ((384, 1280), []), ((384, 1280), [44, 1197, 153, 371]),
                                       ((1216, 1936), None), ((1216, 1936), [0, 1936, 300, 1100])])
def test_compute_edge_metrics_depth(size, crop):
    from synth import scene_with_gt
    from mindtheedge_b200.edge import compute_edge_metrics
    from oracle import chamfer as och
    gt, depth = scene_with_gt(*size, 60 + size[0])
    g01 = (gt / 255).astype(np.float32)
    got = compute_edge_metrics(torch.from_numpy(depth).cuda()[None, None], torch.from_numpy(g01).cuda()[None, None],
                               crop)
    _metrics_eq(got, och.compute_edge_metrics(depth, g01, crop))
    assert np.isfinite(got).all()


def _on_and_next_to(ts, dtype):
    v = []
    for t in ts:
        f = dtype(t)
        v += [f, np.nextafter(f, dtype(np.inf)), np.nextafter(f, dtype(-np.inf))]
    return np.array(v, dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_compute_edge_metrics_edge_model_and_gt_values(dtype):
    """edge_model: the prediction is binarised as p > t for t = 0.5, 0.75, 0.9 in its own dtype, with values on and
    next to every t; the GT is binarised as (g * 255) / 255 > 0.5 in its own dtype, with values on and next to 0.5
    (a float64 GT just above 0.5 is set although its float32 value is 0.5)."""
    from mindtheedge_b200.edge import compute_edge_metrics
    from oracle import chamfer as och
    r = np.random.default_rng(6)
    H, W = 96, 320
    pv = np.concatenate([_on_and_next_to([0.5, 0.75, 0.9], dtype), np.array([0, 0.3, 1], dtype)])
    pm = np.where(r.random((H, W)) < 0.3, r.choice(pv, (H, W)), 0).astype(dtype)
    gv = _on_and_next_to([0.5], dtype)
    if dtype is np.float64:
        gv = np.concatenate([gv, [0.5 + 2.0 ** -30]])
        assert np.float32(gv[-1]) == 0.5
    gm = np.where(r.random((H, W)) < 0.05, r.choice(np.concatenate([gv, [1.0]]), (H, W)), 0).astype(dtype)
    dp, dg = torch.from_numpy(pm).cuda(), torch.from_numpy(gm).cuda()
    for crop in (None, [10, 300, 5, 90]):
        _metrics_eq(compute_edge_metrics(dp, dg, crop, edge_model=True), och.compute_edge_metrics(pm, gm, crop, True))
    # the binarisation decides: some pred and GT pixels sit on the threshold itself
    assert (pm == dtype(0.9)).any() and (gm == dtype(0.5)).any()
    # the same GT under the depth branch
    from synth import scene_with_gt
    d = scene_with_gt(H, W, 7)[1]
    _metrics_eq(compute_edge_metrics(torch.from_numpy(d).cuda(), dg), och.compute_edge_metrics(d, gm))


# ---- CPU: the brute-force oracle and the manifest -------------------------------------------------------------------
def test_brute_force_oracle_vs_scipy():
    """brute_d2 equals the square of scipy's EDT (the oracle's distances) bit for bit after sqrt, also without GT
    (scipy's row -1 convention), with GT everywhere and with a single GT pixel."""
    r = np.random.default_rng(8)
    planes = [r.random((17, 23)) < 0.05, np.zeros((9, 31), bool), np.ones((5, 7), bool), np.zeros((1, 40), bool),
              np.zeros((30, 1), bool)]
    planes[3][0, 39] = True
    for g in planes:
        want = ndimage.distance_transform_edt(~g)
        assert np.array_equal(np.sqrt(brute_d2(g).astype(np.float64)), want)
    y, x = np.mgrid[0:9, 0:31]
    assert np.array_equal(brute_d2(planes[1]), (y + 1) ** 2 + x ** 2)
    p, g = exact_distance_planes()
    for i in range(2):
        d2 = brute_d2(is_set(g[i]))[is_set(p[i])]
        assert sorted(d2.tolist()) == [0, 1, 2, 5, 8, 25, 25, 25]


def test_path_manifest():
    """Every path of the launch is taken by some case, and the numbers the boundaries come from hold."""
    # 2 * W + the static reduction buffers against the 48 KB default: the first W past it is 24,481
    assert 2 * 24480 + STATIC_SMEM <= DEFAULT_SMEM < 2 * 24481 + STATIC_SMEM
    seen = set()
    for name, build in CASES.items():
        seen |= plan(build())
    seen |= plan(Case(np.zeros((1, MAX_H + 1, 1)), np.zeros((1, MAX_H + 1, 1))))
    seen |= plan(Case(np.zeros((1, 1, MAX_W + 1)), np.zeros((1, 1, MAX_W + 1))))
    want = {"row-one-stride", "row-strides", "finish-one-row", "finish-rows", "smem-opt-in", "gt", "no-gt", "pred",
            "no-pred", "gt-everywhere", "pred-is-gt", "search-full-width", "h-max", "refused"}
    assert want <= seen, sorted(want - seen)
    assert plan(case_wide(24480)) & {"smem-opt-in"} == set()
    assert "smem-opt-in" in plan(case_wide(24481)) and "smem-opt-in" in plan(case_wide(24576))
    assert sum_bound(MAX_H, 5) < 3000 * U
