"""Bit-exact parity of the sm_100a Canny path against goldens produced by the reference
``edge_from_depth`` (edge.py:73-93), against cv2.Canny itself and against the NumPy oracle."""
import os
import tempfile

import cv2
import numpy as np
import pytest
import torch

from conftest import GOLDEN

pytestmark = pytest.mark.gpu


def scene(H, W, seed, noise=0.3):
    r = np.random.default_rng(seed)
    d = np.full((H, W), 40.0, np.float32)
    for _ in range(30):
        y0, x0 = r.integers(0, H), r.integers(0, W)
        h, w = r.integers(1, max(2, H // 2)), r.integers(1, max(2, W // 2))
        d[y0:y0 + h, x0:x0 + w] = r.uniform(1, 80)
    return d + r.normal(0, noise, (H, W)).astype(np.float32)


def test_golden_edge_from_depth():
    from mindtheedge_b200.edge import edge_from_depth
    z = np.load(os.path.join(GOLDEN, "canny.npz"))
    with tempfile.TemporaryDirectory() as tmp:
        for i in range(6):
            d = z[f"depth{i}"]
            path = os.path.join(tmp, f"d{i}.npy")
            np.save(path, d)
            for t in (20, 60, 120, 240):
                got = edge_from_depth(path, None, os.path.join(tmp, "e.jpeg"), thresh_1=int(t / 2), thresh_2=int(t),
                                      is_write_edge=False)
                ref = np.unpackbits(z[f"edges{i}_t{t}"])[: d.size].reshape(d.shape) * 255
                assert got.dtype == np.uint8 and got.shape == d.shape
                assert np.array_equal(got, ref), (i, t, int((got != ref).sum()))
        d = z["depth_resize"]
        path = os.path.join(tmp, "dr.npy")
        np.save(path, d)
        out = os.path.join(tmp, "e.png")
        got = edge_from_depth(path, (160, 96), out, thresh_1=20, thresh_2=40, is_write_edge=True)
        ref = np.unpackbits(z["edges_resize"])[: 96 * 160].reshape(96, 160) * 255
        assert np.array_equal(got, ref)
        assert np.array_equal(cv2.imread(out)[:, :, 0], ref)


@pytest.mark.parametrize("shape", [(384, 1280), (1216, 1936), (33, 130), (1, 1), (2, 300), (129, 129)])
def test_vs_cv2_sweep_and_levels(shape):
    """The reference's 12 Canny settings (eval_depth_edges.py:243-244, 281-282) in one call."""
    from mindtheedge_b200.edge import canny_from_depth
    from oracle.canny import quantise_depth
    H, W = shape
    depths = np.stack([scene(H, W, 7 + k) for k in range(2)])
    depths[1] = np.random.default_rng(3).uniform(-5, 95, (H, W)).astype(np.float32)
    pairs = [(int(t / 2), int(t)) for t in range(240, 19, -20)]
    edges, levels = canny_from_depth(torch.from_numpy(depths).cuda(), pairs, want_edges=True, want_levels=True)
    edges, levels = edges.cpu().numpy(), levels.cpu().numpy()
    for n in range(2):
        q = quantise_depth(depths[n])
        for k, (lo, hi) in enumerate(pairs):
            ref = cv2.Canny(q, lo, hi)
            assert np.array_equal(edges[k, n], ref), (n, k, int((edges[k, n] != ref).sum()))
            assert np.array_equal((levels[n] <= k) * 255, ref)


def test_unordered_pairs_u8_and_f64():
    from mindtheedge_b200.edge import Canny, canny_from_depth
    from oracle.canny import canny_np, quantise_depth
    d = scene(200, 333, 11).astype(np.float64)
    q = quantise_depth(d)
    pairs = [(10, 20), (100, 200), (30, 60), (90, 40)]  # not nested; the last has low > high (cv2 swaps)
    e = canny_from_depth(torch.from_numpy(d).cuda(), pairs).cpu().numpy()
    for k, (lo, hi) in enumerate(pairs):
        assert np.array_equal(e[k], cv2.Canny(q, lo, hi))
        assert np.array_equal(e[k], canny_np(q, min(lo, hi), max(lo, hi)))
    assert np.array_equal(Canny(q, 20, 40), cv2.Canny(q, 20, 40))
    with pytest.raises(Exception):
        canny_from_depth(torch.from_numpy(d).cuda(), pairs, want_edges=False, want_levels=True)


def test_long_weak_chain_crosses_many_tiles():
    """A one-pixel-wide weak ramp that is strong only at one end must light up entirely
    (worst case for the tile-iterated hysteresis)."""
    from mindtheedge_b200.edge import canny_from_depth
    H, W = 96, 1300
    d = np.full((H, W), 10.0, np.float32)
    d[48:, :] = 10.0 + 80.0 / 255 * 12       # weak horizontal step along the whole width
    d[48:, :6] = 10.0 + 80.0 / 255 * 120     # strong only at the far left
    from oracle.canny import quantise_depth
    q = quantise_depth(d)
    ref = cv2.Canny(q, 20, 100)
    got = canny_from_depth(torch.from_numpy(d).cuda(), [(20, 100)]).cpu().numpy()[0]
    assert ref[47:49, 600:].any()
    assert np.array_equal(got, ref)


def test_hysteresis_fallback_when_reachable_set_exceeds_shared_memory():
    """White-noise u8 plane at KITTI size with very low thresholds: > 100 k candidates connected to strong pixels, far
    beyond what the shared-memory union-find holds (~25 k) -> the image is handed to the L2 kernel.  Bit-exact with
    cv2.Canny for every pair, alongside an ordinary image in the same batch (which stays on the fast path)."""
    import cv2
    from mindtheedge_b200.edge import canny_from_depth
    r = np.random.default_rng(5)
    noise = r.integers(0, 256, (384, 1280)).astype(np.uint8)
    smooth = cv2.GaussianBlur(r.integers(0, 256, (384, 1280)).astype(np.uint8), (9, 9), 3)
    batch = torch.from_numpy(np.stack([noise, smooth])).cuda()
    pairs = [(40, 80), (10, 20), (1, 2)]
    edges = canny_from_depth(batch, pairs).cpu().numpy()
    for t, (lo, hi) in enumerate(pairs):
        for k, img in enumerate((noise, smooth)):
            assert np.array_equal(edges[t, k], cv2.Canny(img, lo, hi)), (t, k)
    assert int((edges[2, 0] > 0).sum()) > 60000


@pytest.mark.parametrize("shape", [(96, 1296), (64, 48), (200, 16), (384, 1280),
                                   (640, 1280), (600, 1296), (720, 1600), (1216, 1936)])
def test_hysteresis_padded_rows_and_global_bitmap_mode(shape):
    """Shared-memory hysteresis on widths that are multiples of 16 but not of 32 (bitmap rows padded to whole words,
    the DDAD width 1936 is one), and on planes whose bitmaps do not fit in shared memory, so they live in the image's
    global scratch (BIG: more than 576 rows at W = 1280, padded rows at 600 x 1296, DDAD size): bit-exact with
    cv2.Canny for every nested pair."""
    from mindtheedge_b200.edge import canny_from_depth
    from oracle.canny import quantise_depth
    H, W = shape
    depths = np.stack([scene(H, W, 21 + k) for k in range(3)])
    depths[2] = np.random.default_rng(9).uniform(0, 90, (H, W)).astype(np.float32)
    pairs = [(int(t / 2), int(t)) for t in range(240, 19, -20)]
    levels = canny_from_depth(torch.from_numpy(depths).cuda(), pairs, want_edges=False, want_levels=True).cpu().numpy()
    for n in range(3):
        q = quantise_depth(depths[n])
        for k, (lo, hi) in enumerate(pairs):
            assert np.array_equal((levels[n] <= k) * 255, cv2.Canny(q, lo, hi)), (n, k)
