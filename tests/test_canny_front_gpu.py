"""The Canny front (``canny_nms_kernel``: quantise, Sobel, NMS) and the threshold handling of ``canny_from_depth``
against ``cv2.Canny`` on ``oracle.canny.quantise_depth``, bit-exact, and the level plane against
``canny_birth_levels``.

``test_canny_gpu.py`` checks smooth and noisy depth scenes at the shipped settings.  Here the paths are reached through
shapes, dtypes, alignment, values and thresholds: the fp32 ``float4`` load (W % 4 == 0, 16-byte aligned base) and the
scalar load (a view one element into its buffer), fp64 and u8 input, the vector and the byte stores of the candidate
and edge planes (W % 4 == 0 or not) at several tile seams; quantisation at every value boundary with NaN, +-Inf and
out-of-range depth and non-default depth ranges; the NMS tie rules; 254 nested pairs, degenerate pairs, and lists
that are not nested (one pass per pair).
"""
import cv2
import numpy as np
import pytest
import torch

from oracle.canny import canny_birth_levels, quantise_depth

pytestmark = pytest.mark.gpu

NESTED = [(int(t / 2), int(t)) for t in range(240, 19, -20)]


def scene(H, W, seed):
    r = np.random.default_rng(seed)
    d = np.full((H, W), 40.0)
    for _ in range(20):
        y0, x0 = r.integers(0, H), r.integers(0, W)
        d[y0:y0 + r.integers(1, max(2, H // 2)), x0:x0 + r.integers(1, max(2, W // 2))] = r.uniform(1, 80)
    return d + r.normal(0, 0.4, (H, W))


def _run(depth_dev, pairs, min_depth=0.0, max_depth=80.0, levels=True):
    from mindtheedge_b200.edge import canny_from_depth
    out = canny_from_depth(depth_dev, pairs, min_depth, max_depth, want_edges=True, want_levels=levels)
    if levels:
        return out[0].cpu().numpy(), out[1].cpu().numpy()
    return out.cpu().numpy(), None


def _check(depth, pairs, min_depth=0.0, max_depth=80.0, dev=None, levels=True):
    """depth [N,H,W] numpy; -> edges as computed (checked against cv2 per image and pair, levels against the
    oracle when the pairs are nested)."""
    d = torch.from_numpy(depth).cuda() if dev is None else dev
    edges, lv = _run(d, pairs, min_depth, max_depth, levels)
    for n in range(depth.shape[0]):
        q = depth[n] if depth.dtype == np.uint8 else quantise_depth(depth[n], min_depth, max_depth)
        for k, (lo, hi) in enumerate(pairs):
            ref = cv2.Canny(q, lo, hi)
            assert np.array_equal(edges[k, n], ref), (n, k, lo, hi, int((edges[k, n] != ref).sum()))
        if levels:
            assert np.array_equal(lv[n], canny_birth_levels(q, pairs)), n
    return edges


def _f32_view_one_element_in(a):
    buf = torch.empty(a.size + 1, dtype=torch.float32, device="cuda")
    v = buf[1:].view(a.shape)
    v.copy_(torch.from_numpy(a).cuda())
    assert v.data_ptr() % 16 != 0
    return v


SHAPES = [(h, w) for w in (127, 128, 129, 257, 1242) for h in (31, 32, 33, 65)]


@pytest.mark.parametrize("shape", SHAPES, ids=[f"{h}x{w}" for h, w in SHAPES])
def test_shapes_and_dtypes(shape):
    """fp32 aligned (float4 front) and one element into its buffer (scalar front) agree bit for bit and with cv2;
    fp64 and u8 too.  W % 4 != 0 selects the byte stores."""
    H, W = shape
    d = np.stack([scene(H, W, 3 + H + W), np.random.default_rng(W).uniform(-5, 95, (H, W))])
    f32 = d.astype(np.float32)
    e_al = _check(f32, NESTED)
    e_mis = _check(f32, NESTED, dev=_f32_view_one_element_in(f32))
    assert np.array_equal(e_al, e_mis)
    _check(d, NESTED)
    _check(quantise_depth(f32), NESTED)
    assert e_al[-1].any()


def boundary_values(max_depth, dtype):
    """k * max / 255 for every k and its neighbours in the array's own type, plus specials."""
    k = np.arange(256, dtype=np.float64)
    base = (k * max_depth / 255).astype(dtype)
    up = np.nextafter(base, dtype(np.inf))
    dn = np.nextafter(base, dtype(-np.inf))
    specials = np.array([np.nan, np.inf, -np.inf, -1.0, -0.0, 0.0, 2.9, 3.0, max_depth * 1.5, 1e30], dtype)
    return np.concatenate([base, up, dn, specials])


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("min_depth,max_depth", [(0.0, 80.0), (3.0, 50.0), (3.0, 100.7)])
def test_quantisation_boundaries(dtype, min_depth, max_depth):
    """Every value boundary of the u8 quantisation, NaN (-> 0), +-Inf, negative and out-of-range depth, scattered
    over a plane so that a one-level difference changes the edges at low thresholds."""
    vals = boundary_values(max_depth, dtype)
    r = np.random.default_rng(int(max_depth * 10) + 7 * (dtype == np.float32))
    H, W = 66, 260
    d = r.choice(vals, size=(2, H, W)).astype(dtype)
    d[1, :, : W // 2] = np.sort(r.choice(vals, size=H * (W // 2))).reshape(H, W // 2)  # ramps of neighbours
    with np.errstate(invalid="ignore"):
        assert quantise_depth(np.array([np.nan], dtype), min_depth, max_depth)[0] == 0
    _check(d, [(1, 2), (0, 1), (0, 0)], min_depth, max_depth, levels=False)
    _check(d, NESTED, min_depth, max_depth)


def test_nms_ties_on_low_contrast_planes():
    """u8 planes of 0/1/2: many equal magnitudes, so the asymmetric > / >= rule decides in every sector."""
    r = np.random.default_rng(11)
    planes = [r.integers(0, 3, (65, 257)).astype(np.uint8), r.integers(0, 2, (33, 129)).astype(np.uint8)]
    blocky = np.kron(r.integers(0, 3, (17, 33)), np.ones((2, 4), np.int64))[:33, :129].astype(np.uint8)
    planes.append(blocky)
    for p in planes:
        _check(p[None], [(0, 1), (1, 2), (2, 4), (0, 0)], levels=False)
        _check(p[None], [(4, 8), (2, 4), (1, 2), (0, 1)])


@pytest.mark.parametrize("angle", [22.5, 67.5])
def test_nms_ramps_around_sector_edges(angle):
    """Linear ramps whose gradient direction lies just either side of tan 22.5 deg / tan 67.5 deg, in all four
    quadrants."""
    H, W = 65, 257
    y, x = np.mgrid[0:H, 0:W].astype(np.float64)
    planes = []
    for da in (-2.0, -0.5, -0.1, 0.1, 0.5, 2.0):
        a = np.deg2rad(angle + da)
        for sx, sy in ((1, 1), (1, -1), (-1, 1), (-1, -1)):
            v = 3.7 * (sx * np.cos(a) * x + sy * np.sin(a) * y)
            planes.append(np.mod(np.floor(v), 256).astype(np.uint8))
    _check(np.stack(planes), [(1, 2), (8, 16), (20, 40)], levels=False)


def test_254_nested_pairs():
    """MTE_MAX_THRESHOLDS nested pairs, strictest first, edges and levels."""
    pairs = [(max(0, (2 + 8 * (253 - k)) // 2), 2 + 8 * (253 - k)) for k in range(254)]
    assert len(pairs) == 254 and pairs[0][1] >= 2024
    d = np.stack([scene(65, 257, 1), np.random.default_rng(2).uniform(0, 90, (65, 257))]).astype(np.float32)
    _check(d, pairs)


def test_degenerate_pairs():
    """low = 0, low = high, low > high (cv2 swaps), and high >= 2040, above any L1 Sobel magnitude of a u8 plane:
    no strong pixel, no edge."""
    d = np.stack([scene(65, 257, 5), np.random.default_rng(6).uniform(0, 90, (65, 257))]).astype(np.float32)
    e = _check(d, [(0, 50), (30, 30), (60, 20), (1000, 2040), (2040, 3000), (0, 0)], levels=False)
    assert not e[3].any() and not e[4].any() and e[0].any() and e[2].any()


def test_pairs_not_nested_next_to_nested_reordering():
    """A list that is not nested takes one pass per pair; its nested reordering takes the single multi-pair pass.
    Both give cv2's edges, pair for pair."""
    d = np.stack([scene(65, 257, 9), scene(65, 257, 10)]).astype(np.float32)
    loose = [(10, 20), (60, 120), (30, 60), (30, 90)]
    nested = [(60, 120), (30, 90), (30, 60), (10, 20)]
    e_loose = _check(d, loose, levels=False)
    e_nested = _check(d, nested)
    for i, j in ((0, 3), (1, 0), (2, 2), (3, 1)):
        assert np.array_equal(e_loose[i], e_nested[j]), (i, j)
