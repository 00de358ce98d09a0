"""Per-image PR counts (mte_pr_counts_per_image, pr_counts(per_image=True) and the layers above it): every row
(image, threshold) bit-exact against the oracle run on that image alone, and the rows summed equal to the summed
counts of the same batch."""
import os

import cv2
import numpy as np
import pytest
import torch

from conftest import GOLDEN
from synth import prob_map, random_boundary_maps, scene_with_gt

pytestmark = pytest.mark.gpu

KITTI_CROP = [44, 1197, 153, 371]
CANNY_RANGE = list(range(20, 241, 20))


def _window(a, crop):
    return a if crop is None else a[crop[2]:crop[3], crop[0]:crop[1]]


def _oracle_rows(preds, gts, thr, max_dist, crop=None, thin=False):
    """oracle.pr_counts.evaluate_boundaries(pred[win], [gt[win]], thr, max_dist, apply_thinning) for every image."""
    from oracle import pr_counts as opr
    return np.stack([opr.evaluate_boundaries(np.ascontiguousarray(_window(p, crop), dtype=np.float64),
                                             [np.ascontiguousarray(_window(g, crop))], np.asarray(thr, np.float64),
                                             max_dist, apply_thinning=thin)[0] for p, g in zip(preds, gts)])


def _dev(arrays, device="cuda"):
    return torch.from_numpy(np.ascontiguousarray(np.stack(arrays))).to(device)


def _both(preds, gts, thr, max_dist, crop=None, thin=False):
    """(per-image rows, summed counts) of one batch, both from the device."""
    from mindtheedge_b200.eval_depth_edges import pr_counts
    p, g = _dev(preds), _dev(gts)
    kw = dict(max_dist=max_dist, crop=crop, apply_thinning=thin)
    return (pr_counts(p, g, thr, per_image=True, **kw).cpu().numpy(), pr_counts(p, g, thr, **kw).cpu().numpy())


def _check(rows, summed, ref):
    assert rows.shape == ref.shape and rows.dtype == np.int64
    for i in range(ref.shape[0]):
        assert np.array_equal(rows[i], ref[i]), (i, rows[i].tolist(), ref[i].tolist())
    assert np.array_equal(rows.sum(0), summed)


def _soft(h, w, seed, dtype=np.float32):
    pb, _ = random_boundary_maps(h, w, seed)
    ridge = (cv2.GaussianBlur((pb != 0).astype(np.float32), (5, 5), 1.2) * 2.5).clip(0, 1)
    return np.maximum(prob_map(h, w, seed), ridge).astype(dtype)


def _ridge(h, w, seed, dtype=np.float32):
    """Thin curves with values along them: thinning keeps most of them, the matcher has real work."""
    r = np.random.default_rng(seed)
    pb, _ = random_boundary_maps(h, w, seed)
    ridge = (cv2.GaussianBlur((pb != 0).astype(np.float32), (3, 3), 0.6) * 1.6).clip(0, 1)
    return (ridge * (0.5 + 0.5 * r.random((h, w)))).astype(dtype)


def _gt(h, w, seed):
    return (random_boundary_maps(h, w, seed)[1] != 0).astype(np.uint8)


# ---------------------------------------------------------------------------------------------- Canny level planes
def test_canny_level_rows_vs_oracle():
    """12 Canny settings, KITTI crop, max_dist 0.002: bundled KITTI-DE GT maps (incl. the heavy #19 and #29) next to
    synthetic scenes in one batch.  Row i = oracle.pr_sweep_counts of image i alone; the rows sum to sweep_counts."""
    import bench
    from mindtheedge_b200.eval_depth_edges import sweep_counts
    from oracle import pr_counts as opr
    depths, gts = bench.kitti_like_set(102, 7000)
    idx = [19, 29, 3, 60]
    ds = [depths[i] for i in idx]
    gs = [gts[i] for i in idx]
    for k in range(2):
        g, d = scene_with_gt(384, 1280, 120 + k)
        ds.append(d.astype(np.float32))
        gs.append((g > 127).astype(np.uint8))
    d_dev, g_dev = _dev(ds), _dev(gs)
    rng = CANNY_RANGE[::-1][:5] + CANNY_RANGE[:7]        # the caller's order is not the sweep order
    rows = sweep_counts(d_dev, g_dev, rng, KITTI_CROP, 0.0, 80.0, max_dist=0.002, per_image=True).cpu().numpy()
    summed = sweep_counts(d_dev, g_dev, rng, KITTI_CROP, 0.0, 80.0, max_dist=0.002).cpu().numpy()
    ref = np.stack([opr.pr_sweep_counts([d], [g * 255], rng, tuple(KITTI_CROP)) for d, g in zip(ds, gs)])
    _check(rows, summed, ref)
    assert ref[:2, :, 0].min() > 1000
    # chunks on side streams: each chunk's rows land at its images' offsets
    chunked = sweep_counts(d_dev, g_dev, rng, KITTI_CROP, 0.0, 80.0, max_dist=0.002, per_image=True,
                           pipeline_chunks=3).cpu().numpy()
    assert np.array_equal(chunked, rows)
    out = torch.ones((len(ds), len(rng), 4), dtype=torch.int64, device="cuda")
    sweep_counts(d_dev, g_dev, rng, KITTI_CROP, 0.0, 80.0, max_dist=0.002, per_image=True, out=out)
    assert np.array_equal(out.cpu().numpy(), rows + 1)


# ---------------------------------------------------------------------------------------------- strength maps
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_strength_map_rows_vs_oracle(dtype):
    """99 ascending thresholds (sweep matcher) and unsorted, repeated thresholds (per-problem matchers), with a crop,
    NaN and values on a threshold."""
    h, w, crop = 120, 300, [7, 290, 3, 111]
    r = np.random.default_rng(11)
    preds, gts = [], []
    for k in range(3):
        pb, gb = random_boundary_maps(h, w, 700 + k)
        soft = (cv2.GaussianBlur((pb != 0).astype(np.float32), (5, 5), 1.2) * 2.5).clip(0, 1)
        soft = (soft * (0.4 + 0.6 * r.random((h, w)))).astype(dtype)
        soft[5, 9] = 0.5
        soft[9, 11] = np.nan
        preds.append(soft)
        gts.append((gb != 0).astype(np.uint8))
    for thr in (np.linspace(0.01, 0.99, 99), np.array([0.5, 0.2, 0.5, 0.9, 0.05, 0.2, 0.7])):
        rows, summed = _both(preds, gts, thr, 0.0075, crop)
        _check(rows, summed, _oracle_rows(preds, gts, thr, 0.0075, crop))
        assert rows[:, :, 0].max() > 0


# ---------------------------------------------------------------------------------------------- thinned sweep
def test_thinned_kitti_crop_99_thresholds():
    from mindtheedge_b200 import _lib
    preds = [_ridge(384, 1280, 800 + k) for k in range(2)]
    gts = [_gt(384, 1280, 810 + k) for k in range(2)]
    thr = np.linspace(0.01, 0.99, 99)
    rows, summed = _both(preds, gts, thr, 0.002, KITTI_CROP, thin=True)
    _check(rows, summed, _oracle_rows(preds, gts, thr, 0.002, KITTI_CROP, thin=True))
    assert rows[:, 0, 0].min() > 500
    assert _lib.MTE_MAX_THRESHOLDS >= 99


def test_thinned_ddad_size_uncropped_spanning_two_chunks():
    """Two uncropped 1216x1936 planes: their bit planes do not fit shared memory (global-memory thinning), and the
    slab holds fewer problems than the batch has, so the chunk boundary falls inside the second image."""
    from mindtheedge_b200 import _lib
    N, H, W, T = 2, 1216, 1936, 64
    per = 2 * H * ((W + 31) // 32) * 4
    region = _lib.lib.mte_pr_thin_workspace_bytes(N, H, W, T, 0.002) - _lib.lib.mte_pr_workspace_bytes(N, H, W, T, 0.002)
    assert T < region // per < N * T
    preds = [_ridge(H, W, 900 + k) for k in range(N)]
    gts = [_gt(H, W, 910 + k) for k in range(N)]
    thr = np.linspace(0.2, 0.95, T)
    rows, summed = _both(preds, gts, thr, 0.002, thin=True)
    _check(rows, summed, _oracle_rows(preds, gts, thr, 0.002, thin=True))
    assert rows[:, 0, 0].min() > 5000


# ---------------------------------------------------------------------------------------------- overflow paths
def test_rows_of_images_that_overflow_the_sweep_matcher():
    """A window with more GT pixels than the sweep matcher keeps resident (its problems go to the per-problem kernels
    through the overflow list) between two that fit."""
    H, W = 384, 1280
    r = np.random.default_rng(int(1000 * 0.02 + 100000 * 0.08))
    gt = np.zeros((H, W), np.uint8)
    for _ in range(int(0.08 * H * W / 150)):
        y, x = int(r.integers(0, H)), int(r.integers(0, W))
        for _ in range(150):
            gt[y, x] = 1
            y = int(np.clip(y + r.integers(-1, 2), 0, H - 1)); x = int(np.clip(x + r.integers(0, 2), 0, W - 1))
    near = cv2.dilate(gt, np.ones((5, 5), np.uint8)) > 0
    dense = np.where(near, r.random((H, W)), 0.0) * (r.random((H, W)) < 0.02 / max(near.mean(), 1e-6) * 0.7)
    dense = np.maximum(dense, (r.random((H, W)) < 0.006) * r.random((H, W))).astype(np.float32)
    assert int(_window(gt, KITTI_CROP).sum()) > 9500
    preds = [_ridge(H, W, 1001), dense, _ridge(H, W, 1002)]
    gts = [_gt(H, W, 1011), gt, _gt(H, W, 1012)]
    thr = np.array([0.15, 0.3, 0.45, 0.6, 0.75, 0.9])
    rows, summed = _both(preds, gts, thr, 0.002, KITTI_CROP)
    _check(rows, summed, _oracle_rows(preds, gts, thr, 0.002, KITTI_CROP))


def test_thinned_rows_with_a_window_beyond_the_shared_memory_matcher():
    """A lattice of isolated pixels survives thinning with more than 0xFFF0 pixels: that problem runs in match_kernel,
    the other image's in the shared-memory matcher."""
    H, W = 384, 1280
    r = np.random.default_rng(5)
    lattice = np.zeros((H, W), np.float32)
    lattice[::2, ::2] = r.random((H // 2, W // 2))
    preds = [_ridge(H, W, 1101), lattice]
    gts = [_gt(H, W, 1111), (r.random((H, W)) < 0.03).astype(np.uint8)]
    thr = np.array([0.05, 0.5])
    rows, summed = _both(preds, gts, thr, 0.002, thin=True)
    _check(rows, summed, _oracle_rows(preds, gts, thr, 0.002, thin=True))
    assert rows[1, 0, 3] > 0xFFF0


# ---------------------------------------------------------------------------------------------- edge cases
def test_empty_crop_leaves_the_rows_untouched():
    from mindtheedge_b200.eval_depth_edges import pr_counts
    p = _dev([_soft(40, 60, 1), _soft(40, 60, 2)])
    g = _dev([_gt(40, 60, 3), _gt(40, 60, 4)])
    for thin in (False, True):
        out = torch.full((2, 3, 4), 7, dtype=torch.int64, device="cuda")
        pr_counts(p, g, [0.1, 0.5, 0.9], crop=[10, 10, 0, 40], apply_thinning=thin, per_image=True, out=out)
        assert (out.cpu() == 7).all()
        assert not pr_counts(p, g, [0.1, 0.5, 0.9], crop=[0, 60, 30, 30], apply_thinning=thin,
                             per_image=True).cpu().any()


def test_single_image_and_accumulation_through_the_c_abi():
    """N = 1 equals mte_pr_counts; two calls into one buffer give twice the rows; the level-plane mode too."""
    import ctypes as C
    from mindtheedge_b200 import _lib, runtime
    L = _lib.lib
    H, W, T = 90, 200, 9
    thr_np = np.linspace(0.1, 0.9, T)
    thr = thr_np.ctypes.data_as(C.POINTER(C.c_double))
    crop = (C.c_int32 * 4)(5, 190, 4, 80)
    for thin in (0, 1):
        for N in (1, 3):
            p = _dev([_soft(H, W, 20 + k) for k in range(N)])
            g = _dev([_gt(H, W, 30 + k) for k in range(N)])
            q = L.mte_pr_thin_workspace_bytes if thin else L.mte_pr_workspace_bytes
            ws = torch.zeros(q(N, H, W, T, 0.0075), dtype=torch.uint8, device="cuda")
            summed = torch.zeros((T, 4), dtype=torch.int64, device="cuda")
            rows = torch.zeros((N, T, 4), dtype=torch.int64, device="cuda")
            args = (p.data_ptr(), _lib.MTE_F32, g.data_ptr(), N, H, W, crop, thr, T, 0.0075, thin)
            tail = (ws.data_ptr(), ws.numel(), runtime.current_stream_ptr(p.device))
            assert L.mte_pr_counts(*args, summed.data_ptr(), *tail) == 0
            for _ in range(2):
                assert L.mte_pr_counts_per_image(*args, rows.data_ptr(), *tail) == 0
            torch.cuda.synchronize()
            s, r = summed.cpu().numpy(), rows.cpu().numpy()
            assert np.array_equal(r.sum(0), 2 * s)
            assert r[:, :, 0].max() > 0 and np.all(r % 2 == 0)
            if N == 1:
                assert np.array_equal(r[0], 2 * s)
            ref = _oracle_rows([p_.cpu().numpy() for p_ in p], [g_.cpu().numpy() for g_ in g], thr_np, 0.0075,
                               [5, 190, 4, 80], bool(thin))
            assert np.array_equal(r, 2 * ref)


def test_level_plane_rows():
    """uint8 level planes (edge at t iff level <= t), thinned and not."""
    from mindtheedge_b200.eval_depth_edges import pr_counts
    from oracle import pr_counts as opr
    from oracle import thin as othin
    T, crop = 6, [3, 95, 2, 58]
    levels = [np.clip((1.0 - _soft(64, 100, 40 + k)) * 9, 0, 255).astype(np.uint8) for k in range(3)]
    gts = [_gt(64, 100, 50 + k) for k in range(3)]
    for thin in (False, True):
        rows = pr_counts(_dev(levels), _dev(gts), n_levels=T, max_dist=0.0075, crop=crop, apply_thinning=thin,
                         per_image=True).cpu().numpy()
        for i, (lv, g) in enumerate(zip(levels, gts)):
            lw, gw = _window(lv, crop), np.ascontiguousarray(_window(g, crop))
            for t in range(T):
                b = lw <= t
                b = (othin.binary_thin(b) if thin else b).astype(np.uint8)
                m = opr.match_count(b, gw, 0.0075)
                assert tuple(rows[i, t]) == (m, int(gw.sum()), m, int(b.sum())), (thin, i, t)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_per_image_rows_on_second_gpu():
    from mindtheedge_b200.eval_depth_edges import pr_counts
    preds = [_soft(218, 400, 500 + k) for k in range(2)]
    gts = [_gt(218, 400, 510 + k) for k in range(2)]
    thr = np.linspace(0.05, 0.95, 19)
    torch.cuda.set_device(0)
    for thin in (False, True):
        c1 = pr_counts(_dev(preds, "cuda:1"), _dev(gts, "cuda:1"), thr, apply_thinning=thin, per_image=True)
        assert c1.device == torch.device("cuda:1")
        assert np.array_equal(c1.cpu().numpy(), _oracle_rows(preds, gts, thr, 0.0075, thin=thin))


# ---------------------------------------------------------------------------------------------- pr_evaluation
def _write_edges(tmp, i, depth, gt_shape, rng):
    """The predicted edge image of every Canny setting as pr_evaluation's worker would save it (lossless here)."""
    from mindtheedge_b200.edge import _edges_of_array
    H, W = gt_shape
    paths = []
    for t in rng:
        e = _edges_of_array(depth, None if depth.shape == (H, W) else (W, H), 0.0, 80.0, int(t / 2), int(t))
        pe = os.path.join(tmp, f"edge{i}_{t}.png")
        cv2.imwrite(pe, e)
        paths.append(pe)
    return paths


def _assert_same_result(a, b):
    for name, x, y in zip(a._fields, a, b):
        assert type(x) is type(y), name
        assert np.asarray(x).dtype == np.asarray(y).dtype, name
        assert np.array_equal(x, y), (name, x, y)


def test_pr_evaluation_per_image_golden_files(tmp_path):
    from mindtheedge_b200.eval_depth_edges import _pred_eval, pr_evaluation
    z = np.load(os.path.join(GOLDEN, "pr.npz"))
    H, W = (int(v) for v in z["pr_shape"])
    rng = [int(v) for v in z["pr_range"]]
    crop = [int(v) for v in z["pr_crop"]]
    gts, preds = [], []
    for i in range(3):
        g = np.unpackbits(z[f"pr_gt{i}"])[: H * W].reshape(H, W)
        gp, dp = str(tmp_path / f"gt{i}.png"), str(tmp_path / f"pred{i}.npy")
        cv2.imwrite(gp, g.astype(np.uint8) * 255)
        np.save(dp, (z[f"pr_depth_u16_{i}"] / 256).astype(np.float32))
        gts.append(gp)
        preds.append(dp)
    pv, rv, results = pr_evaluation(gts, preds, edge_thresh_range=rng, gt_crop=crop, per_image=True)
    assert np.array_equal(np.array(pv), z["pr_precision"])
    assert np.array_equal(np.array(rv), z["pr_recall"])
    assert len(results) == 3 and all(len(r) == len(rng) for r in results)
    for i in range(3):
        edges = _write_edges(str(tmp_path), i, np.load(preds[i]), (H, W), rng)
        for k, pe in enumerate(edges):
            _assert_same_result(results[i][k], _pred_eval(pe, gts[i], str(crop)))
    assert sum(r.count_r_overall[0] for r in results[0]) > 0


def test_pr_evaluation_per_image_mask_image(tmp_path):
    """Mask-image branch: per-image rows with the fractional sum_r of (gt * mask) per image."""
    from mindtheedge_b200.eval_depth_edges import _pred_eval, pr_evaluation
    z = np.load(os.path.join(GOLDEN, "pr_mask.npz"))
    H, W = (int(v) for v in z["shape"])
    mp = str(tmp_path / "mask.png")
    cv2.imwrite(mp, z["mask"])
    rng = [int(v) for v in z["range"]]
    gts, preds = [], []
    for i in range(2):
        g = np.unpackbits(z[f"gt{i}"])[:H * W].reshape(H, W)
        gp, dp = str(tmp_path / f"gt{i}.png"), str(tmp_path / f"pred{i}.npy")
        cv2.imwrite(gp, g.astype(np.uint8) * 255)
        np.save(dp, (z[f"depth_u16_{i}"] / 256).astype(np.float32))
        gts.append(gp)
        preds.append(dp)
    pv, rv, results = pr_evaluation(gts, preds, edge_thresh_range=rng, gt_crop=mp, per_image=True)
    assert np.array_equal(np.array(pv), z["precision"])
    assert np.array_equal(np.array(rv), z["recall"])
    for i in range(2):
        edges = _write_edges(str(tmp_path), i, np.load(preds[i]), (H, W), rng)
        for k, pe in enumerate(edges):
            _assert_same_result(results[i][k], _pred_eval(pe, gts[i], mp))
        assert results[i][0].sum_r_overall[0] != np.round(results[i][0].sum_r_overall[0])   # fractional


# ---------------------------------------------------------------------------------------------- evaluate_boundaries_batch
def test_evaluate_boundaries_batch_equals_the_per_image_loop():
    from mindtheedge_b200.eval_depth_edges import evaluate_boundaries, evaluate_boundaries_batch
    preds = [_soft(60, 90, 1).astype(np.float64), _soft(60, 90, 2), _soft(45, 70, 3), _soft(60, 90, 4),
             (_soft(45, 70, 5) > 0.5).astype(np.uint8)]
    gts = [_gt(60, 90, 11).astype(np.float64) * 0.5, _gt(60, 90, 12), _gt(45, 70, 13) * 255, _gt(60, 90, 14),
           _gt(45, 70, 15).astype(bool)]
    soft = np.random.default_rng(0).random((60, 90)) * _gt(60, 90, 16)      # soft GT: sum_r is the sum of the values
    preds.append(_soft(60, 90, 6).astype(np.float64))
    gts.append(soft)
    for kw in (dict(thresholds=25), dict(thresholds=25, apply_thinning=False), dict(),
               dict(thresholds=np.array([0.6, 0.1, 0.6, 0.3]), max_dist=0.02),
               dict(thresholds=300, apply_thinning=True)):
        got = evaluate_boundaries_batch(preds, gts, **kw)
        ref = [evaluate_boundaries(p, [g], **kw) for p, g in zip(preds, gts)]
        assert len(got) == len(ref)
        for a, b in zip(got, ref):
            assert len(a) == len(b) == 5
            for x, y in zip(a, b):
                assert x.dtype == y.dtype and np.array_equal(x, y), kw
    assert got[5][1][0] == soft.sum() and got[5][1][0] != np.round(got[5][1][0])
