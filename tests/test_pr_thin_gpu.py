"""Thinned threshold sweep: the bit-parallel thinning (mte_binary_thin and the thinning stage of
mte_pr_counts(apply_thinning=1)) and the thinned PR counts against oracle/thin.py + oracle/csrc/match.c."""
import ctypes as C

import cv2
import numpy as np
import pytest
import torch

from synth import prob_map, random_boundary_maps

KITTI_CROP = [44, 1197, 153, 371]


def _window(a, crop):
    return a if crop is None else a[crop[2]:crop[3], crop[0]:crop[1]]


def _oracle(preds, gts, thr, max_dist, crop=None):
    """oracle.pr_counts.evaluate_boundaries(pred[win], [gt[win]], thr, max_dist, apply_thinning=True) summed over
    the images."""
    from oracle import pr_counts as opr
    out = np.zeros((len(thr), 4), np.int64)
    for p, g in zip(preds, gts):
        c, _ = opr.evaluate_boundaries(np.ascontiguousarray(_window(p, crop), dtype=np.float64),
                                       [np.ascontiguousarray(_window(g, crop))], np.asarray(thr, np.float64), max_dist,
                                       apply_thinning=True)
        out += c
    return out


def _gpu(preds, gts, thr, max_dist, crop=None, **kw):
    from mindtheedge_b200.eval_depth_edges import pr_counts
    return pr_counts(torch.from_numpy(np.stack(preds)).cuda(), torch.from_numpy(np.stack(gts)).cuda(), thr,
                     max_dist=max_dist, crop=crop, apply_thinning=True, **kw).cpu().numpy()


def _soft(h, w, seed, dtype=np.float32):
    """A DEE-like map plus an edge-like ridge map: thick blobs at low thresholds, thin curves at high ones."""
    pb, _ = random_boundary_maps(h, w, seed)
    ridge = (cv2.GaussianBlur((pb != 0).astype(np.float32), (5, 5), 1.2) * 2.5).clip(0, 1)
    return np.maximum(prob_map(h, w, seed), ridge).astype(dtype)


def _gt(h, w, seed):
    return (random_boundary_maps(h, w, seed)[1] != 0).astype(np.uint8)


# ---------------------------------------------------------------------------------------------- host-only checks
def test_thin_workspace_queries_and_argument_checks_without_a_gpu():
    from mindtheedge_b200 import _lib
    L = _lib.lib
    for n, h, w, t, d in [(1, 8, 8, 1, 0.0075), (102, 384, 1280, 99, 0.0075), (1, 1216, 1936, 4, 0.0075),
                          (3, 2000, 1, 5, 0.1)]:
        assert L.mte_pr_thin_workspace_bytes(n, h, w, t, d) >= L.mte_pr_workspace_bytes(n, h, w, t, d) > 0
    assert L.mte_pr_thin_workspace_bytes(0, 8, 8, 1, 0.0075) == 0
    # binary_thin's global-memory bit planes: 2 planes of ceil(w/32) words per row, also for tall, narrow planes
    for n, h, w in [(1, 4000, 1), (2, 1216, 1936), (5, 3, 33)]:
        assert L.mte_thin_workspace_bytes(n, h, w) >= _lib.MTE_WS_HEADER_BYTES + n * 2 * h * ((w + 31) // 32) * 4
    thr = (C.c_double * 1)(0.5)
    small = L.mte_pr_workspace_bytes(1, 8, 8, 1, 0.0075)
    assert L.mte_pr_counts(256, 0, 256, 1, 8, 8, None, thr, 1, 0.0075, 1, 256, 256, small, None) == -3
    assert L.mte_pr_counts(256, 0, 256, 1, 8, 8, None, thr, 1, 0.0075, 2, 256, 256, 1 << 30, None) == -4
    assert L.mte_pr_counts(256, 0, 256, 1, 8, 8, None, thr, 1, 0.0075, -1, 256, 256, 1 << 30, None) == -4
    assert L.mte_pr_counts(256, 2, 256, 1, 8, 8, None, None, 300, 0.002, 1, 256, 256, 1 << 30, None) == -4


# ---------------------------------------------------------------------------------------------- thinning
@pytest.mark.gpu
def test_all_256_neighbourhood_codes_at_every_word_phase():
    """Every 3x3 neighbourhood code as an isolated patch, centred at every x mod 32 (patches cross word boundaries):
    binary_thin with max_iter=1 and to convergence equals oracle/thin.py."""
    from mindtheedge_b200.bsds.thin import binary_thin_batch
    from oracle import thin as othin
    cols = 64
    H, W = 4 * (256 // cols) + 1, 32 + 4 * cols + 2
    planes = np.zeros((32, H, W), np.uint8)
    phases = set()
    for n in range(32):
        for c in range(256):
            y, x = 2 + 4 * (c // cols), n + 1 + 4 * (c % cols)
            planes[n, y, x] = 1
            for k, (dy, dx) in enumerate(othin.NEIGH):
                planes[n, y + dy, x + dx] = (c >> k) & 1
            phases.add((c, x % 32))
    assert len(phases) == 256 * 32
    d = torch.from_numpy(planes).cuda()
    for it in (1, None):
        got = binary_thin_batch(d, it).cpu().numpy()
        for n in range(32):
            assert np.array_equal(got[n].astype(bool), othin.binary_thin(planes[n], it)), (n, it)


@pytest.mark.gpu
def test_binary_thin_shapes_and_global_memory_planes():
    """Shapes around the word size, a single row, and a plane whose bit planes do not fit shared memory."""
    from mindtheedge_b200.bsds.thin import binary_thin_batch
    from oracle import thin as othin
    r = np.random.default_rng(3)
    for shape, dens in [((9, 5), 0.6), ((40, 31), 0.5), ((33, 65), 0.5), ((1, 70), 0.9), ((300, 1), 1.0),
                        ((1216, 1936), 0.05)]:
        x = r.random((2,) + shape) < dens
        x[:, : shape[0] // 2, : shape[1] // 2] = True
        got = binary_thin_batch(torch.from_numpy(x.astype(np.uint8)).cuda()).cpu().numpy()
        for k in range(2):
            assert np.array_equal(got[k].astype(bool), othin.binary_thin(x[k])), shape


# ---------------------------------------------------------------------------------------------- thinned counts
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_thinned_99_threshold_sweep_vs_oracle(dtype):
    """99 thresholds, NaN values and values exactly on a threshold, fp32 and fp64 maps."""
    thr = np.linspace(0.01, 0.99, 99)
    preds, gts = [], []
    for k in range(3):
        p = _soft(60, 100, 30 + k, dtype)
        p[5, 7] = thr[40]
        p[20:23, 30:33] = thr[70]
        p[9, 11] = np.nan
        p[40:44, 50:60] = np.nan
        preds.append(p)
        gts.append(_gt(60, 100, 60 + k))
    c = _gpu(preds, gts, thr, 0.0075)
    ref = _oracle(preds, gts, thr, 0.0075)
    assert np.array_equal(c, ref), (c.tolist(), ref.tolist())
    assert (np.diff(ref[:, 3]) != 0).any() and ref[:, 0].max() > 0


@pytest.mark.gpu
def test_thinned_unsorted_and_repeated_thresholds():
    thr = np.array([0.5, 0.2, 0.5, 0.9, 0.05, 0.2, 0.7])
    preds = [_soft(50, 90, 5), _soft(50, 90, 6)]
    gts = [_gt(50, 90, 7), _gt(50, 90, 8)]
    c = _gpu(preds, gts, thr, 0.0075)
    assert np.array_equal(c, _oracle(preds, gts, thr, 0.0075))
    assert np.array_equal(c[0], c[2]) and np.array_equal(c[1], c[5])


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(20, 5), (30, 31), (37, 70), (17, 96), (1, 50), (1, 1), (200, 1)])
def test_thinned_counts_narrow_and_unaligned_windows(shape):
    h, w = shape
    thr = np.array([0.05, 0.2, 0.4, 0.6])
    r = np.random.default_rng(h * 1000 + w)
    preds = [np.maximum(r.random((h, w)) * 0.5, (r.random((h, w)) < 0.3) * 0.9).astype(np.float32) for _ in range(2)]
    gts = [(r.random((h, w)) < 0.1).astype(np.uint8) for _ in range(2)]
    c = _gpu(preds, gts, thr, 0.05)
    assert np.array_equal(c, _oracle(preds, gts, thr, 0.05))


@pytest.mark.gpu
def test_crop_through_thick_blobs_pads_at_the_window_border():
    """The crop cuts through solid blobs: thinning must zero-pad at the crop border (the reference crops, then thins).
    Thinning the whole plane and cropping afterwards gives different counts, so the test sees the difference."""
    from oracle import thin as othin
    H, W = 96, 160
    crop = [30, 130, 20, 70]
    preds, gts = [], []
    for k in range(2):
        p = _soft(H, W, 80 + k) * 0.5
        p[10:60, 20:60] = 0.9          # blobs cut by the crop's left and top edges
        p[50:90, 100:140] = 0.8        # ... and by its bottom and right edges
        preds.append(p)
        gts.append((np.random.default_rng(90 + k).random((H, W)) < 0.05).astype(np.uint8))
    thr = np.array([0.3, 0.6, 0.85])
    c = _gpu(preds, gts, thr, 0.0075, crop=crop)
    ref = _oracle(preds, gts, thr, 0.0075, crop=crop)
    assert np.array_equal(c, ref), (c.tolist(), ref.tolist())
    thin_then_crop = sum(int(_window(othin.binary_thin(p >= thr[1]), crop).sum()) for p in preds)
    assert thin_then_crop != ref[1, 3]


@pytest.mark.gpu
def test_empty_crop_counts_nothing():
    from mindtheedge_b200.eval_depth_edges import pr_counts
    p = torch.from_numpy(_soft(40, 60, 1)).cuda()[None]
    g = torch.from_numpy(_gt(40, 60, 2)).cuda()[None]
    out = torch.full((3, 4), 7, dtype=torch.int64, device="cuda")
    pr_counts(p, g, [0.1, 0.5, 0.9], crop=[10, 10, 0, 40], apply_thinning=True, out=out)
    assert (out.cpu() == 7).all()


@pytest.mark.gpu
def test_thinned_level_plane():
    """uint8 level plane (edge at t iff level <= t), thinned per level."""
    from mindtheedge_b200.eval_depth_edges import pr_counts
    from oracle import pr_counts as opr
    from oracle import thin as othin
    T, crop = 5, [3, 95, 2, 58]
    levels, gts = [], []
    for k in range(2):
        s = _soft(64, 100, 40 + k)
        levels.append(np.clip((1.0 - s) * 8, 0, 255).astype(np.uint8))
        gts.append(_gt(64, 100, 50 + k))
    c = pr_counts(torch.from_numpy(np.stack(levels)).cuda(), torch.from_numpy(np.stack(gts)).cuda(), n_levels=T,
                  max_dist=0.0075, crop=crop, apply_thinning=True).cpu().numpy()
    ref = np.zeros((T, 4), np.int64)
    for lv, g in zip(levels, gts):
        lw, gw = _window(lv, crop), np.ascontiguousarray(_window(g, crop))
        for t in range(T):
            b = othin.binary_thin(lw <= t).astype(np.uint8)
            m = opr.match_count(b, gw, 0.0075)
            ref[t] += (m, int(gw.sum()), m, int(b.sum()))
    assert np.array_equal(c, ref), (c.tolist(), ref.tolist())


@pytest.mark.gpu
def test_evaluate_boundaries_thinned_vs_oracle():
    """The public evaluate_boundaries (default apply_thinning=True) with one GT map, soft GT values for sum_r."""
    from mindtheedge_b200.eval_depth_edges import evaluate_boundaries
    from oracle import pr_counts as opr
    p = _soft(70, 110, 11).astype(np.float64)
    g = _gt(70, 110, 12).astype(np.float64) * 0.5
    c_r, s_r, c_p, s_p, thr = evaluate_boundaries(p, [g], thresholds=25, max_dist=0.0075)
    ref, rthr = opr.evaluate_boundaries(p, [g != 0], thresholds=25, max_dist=0.0075, apply_thinning=True)
    assert np.array_equal(thr, rthr)
    assert np.array_equal(np.stack([c_r, c_p, s_p], 1).astype(np.int64), ref[:, [0, 2, 3]])
    assert (s_r == g.sum()).all()


# ---------------------------------------------------------------------------------------------- sizes
@pytest.mark.gpu
def test_kitti_size_cropped_and_uncropped():
    """384x1280: KITTI crop at max_dist 0.002, and the whole plane at 0.0075 (radius 10 px: the offset table is
    staged through the workspace)."""
    H, W = 384, 1280
    preds = [_soft(H, W, 200 + k) for k in range(2)]
    gts = [_gt(H, W, 210 + k) for k in range(2)]
    thr = np.array([0.15, 0.5, 0.8])
    c = _gpu(preds, gts, thr, 0.002, crop=KITTI_CROP)
    assert np.array_equal(c, _oracle(preds, gts, thr, 0.002, crop=KITTI_CROP))
    thr = np.array([0.3, 0.7])
    c = _gpu(preds, gts, thr, 0.0075)
    ref = _oracle(preds, gts, thr, 0.0075)
    assert np.array_equal(c, ref)
    assert ref[:, 0].min() > 1000


@pytest.mark.gpu
def test_thinned_sets_overflow_the_shared_memory_matcher():
    """Isolated pixels survive thinning.  A lattice of them leaves more than 0xFFF0 predicted pixels in the window at
    the low threshold: the shared-memory matcher numbers vertices with 16 bits and hands every such problem to the
    dense matcher (match_kernel), whatever its shared-memory capacity."""
    from oracle import thin as othin
    H, W = 384, 1280
    r = np.random.default_rng(5)
    pred = np.zeros((H, W), np.float32)
    pred[::2, ::2] = r.random((H // 2, W // 2))
    gt = (r.random((H, W)) < 0.03).astype(np.uint8)
    thr = np.array([0.05, 0.5])
    assert othin.binary_thin(pred >= thr[0]).sum() > 0xFFF0
    c = _gpu([pred], [gt], thr, 0.002)
    assert np.array_equal(c, _oracle([pred], [gt], thr, 0.002))
    assert c[0, 3] > 0xFFF0


@pytest.mark.gpu
def test_ddad_size_uncropped_global_memory_thinning():
    """1216x1936 without crop: the window's two bit planes (2 x 297 KB) do not fit shared memory."""
    H, W = 1216, 1936
    pred = _soft(H, W, 300)
    gt = _gt(H, W, 301)
    thr = np.array([0.3, 0.6, 0.9])
    c = _gpu([pred], [gt], thr, 0.002)
    ref = _oracle([pred], [gt], thr, 0.002)
    assert np.array_equal(c, ref), (c.tolist(), ref.tolist())
    assert ref[:, 0].max() > 10000


@pytest.mark.gpu
def test_batch_spanning_several_chunks_equals_per_image_calls():
    """1024x1024 planes thin in global memory, so the slab takes 256 problems per chunk: 3 images x 99 thresholds are
    two chunks with the boundary inside the third image; the counts must equal the sum of the per-image calls."""
    from mindtheedge_b200 import _lib
    N, H, W, T = 3, 1024, 1024, 99
    per = 2 * H * ((W + 31) // 32) * 4
    region = _lib.lib.mte_pr_thin_workspace_bytes(N, H, W, T, 0.0075) - _lib.lib.mte_pr_workspace_bytes(N, H, W, T, 0.0075)
    assert region // per < N * T
    preds = [_soft(H, W, 400 + k) for k in range(N)]
    gts = [_gt(H, W, 410 + k) for k in range(N)]
    thr = np.linspace(0.01, 0.99, T)
    c = _gpu(preds, gts, thr, 0.0075)
    parts = sum(_gpu([p], [g], thr, 0.0075) for p, g in zip(preds, gts))
    assert np.array_equal(c, parts)


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_thinned_counts_on_second_gpu():
    from mindtheedge_b200.eval_depth_edges import pr_counts
    preds = np.stack([_soft(218, 400, 500 + k) for k in range(2)])
    gts = np.stack([_gt(218, 400, 510 + k) for k in range(2)])
    thr = np.linspace(0.05, 0.95, 19)
    torch.cuda.set_device(0)
    c1 = pr_counts(torch.from_numpy(preds).to("cuda:1"), torch.from_numpy(gts).to("cuda:1"), thr,
                   apply_thinning=True)
    assert c1.device == torch.device("cuda:1")
    assert np.array_equal(c1.cpu().numpy(), _oracle(list(preds), list(gts), thr, 0.0075))
