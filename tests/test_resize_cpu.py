"""The bilinear resize of predicted depth (``cv2.resize`` INTER_LINEAR, edge.py:76-78) without a GPU: the C oracle
against ``cv2.resize`` of the opencv-python wheel bit for bit, and the host-side argument checks of
``mte_resize_linear``.  No kernel is launched here."""
import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")

# named cases: KITTI 2x up, DDAD-size up, 12x down, 60x up, 2x2 source, near-identity
NAMED = [((192, 640), (384, 1280)), ((384, 1280), (1216, 1936)), ((1216, 1936), (96, 160)), ((20, 31), (1216, 1936)),
         ((2, 2), (384, 1280)), ((383, 1279), (384, 1280))]
# integer factors 2, 4, 1/2, 1/4, identity, W % 4 != 0
FACTORS = [((48, 80), (96, 160)), ((48, 80), (192, 320)), ((96, 160), (48, 80)), ((192, 320), (48, 80)),
           ((37, 53), (37, 53)), ((2, 3), (2, 3)), ((37, 53), (75, 107)), ((30, 41), (13, 7)), ((50, 60), (50, 97)),
           ((50, 60), (93, 60))]


def random_shapes(n=40, seed=2024):
    r = np.random.default_rng(seed)
    return [((int(r.integers(2, 701)), int(r.integers(2, 701))), (int(r.integers(2, 1401)), int(r.integers(2, 1401))))
            for _ in range(n)]


SHAPES = NAMED + FACTORS + random_shapes()
VALUES = ["u0_80", "x1e6", "minus1", "nonfinite", "dense_nonfinite"]


def plane(hw, values, seed):
    r = np.random.default_rng(seed)
    h, w = hw
    s = r.uniform(0, 80, (h, w)).astype(np.float32)
    if values == "x1e6":
        s *= np.float32(1e6)
    elif values == "minus1":
        s[r.random((h, w)) < 0.2] = -1
    elif values in ("nonfinite", "dense_nonfinite"):
        p = 0.02 if values == "nonfinite" else 0.15
        m = r.random((h, w))
        s[m < p] = np.nan
        s[(m >= p) & (m < 2 * p)] = np.inf
        s[(m >= 2 * p) & (m < 3 * p)] = -np.inf
    return s


def bits_equal(a, b):
    """Bit for bit, except that any NaN equals any NaN (their payloads are not part of the rule)."""
    nan = np.isnan(a)
    return a.shape == b.shape and np.array_equal(nan, np.isnan(b)) and \
        np.array_equal(a.view(np.uint32)[~nan], b.view(np.uint32)[~nan])


def test_reference_opencv_build():
    """The rule is pinned against this OpenCV build with its IPP HAL on (DESIGN.md section 2)."""
    assert cv2.__version__ == "4.13.0"
    assert cv2.ipp.useIPP()


@pytest.mark.parametrize("k", range(len(SHAPES)))
def test_oracle_equals_cv2_resize(k):
    from oracle.resize import resize_linear
    hw, HW = SHAPES[k]
    for v, values in enumerate(VALUES):
        s = plane(hw, values, 100 * k + v)
        ref = cv2.resize(s, (HW[1], HW[0]), interpolation=cv2.INTER_LINEAR)
        got = resize_linear(s, HW)
        assert bits_equal(got, ref), (hw, HW, values, int((got != ref).sum()))


def test_oracle_single_non_finite_pixel_everywhere():
    """One Inf, -Inf or NaN at every source position of small planes: the border taps copy, the corner blocks turn an
    Inf into NaN, interior taps propagate through the fma."""
    from oracle.resize import resize_linear
    r = np.random.default_rng(5)
    for val in (np.inf, -np.inf, np.nan):
        for hw, HW in [((5, 5), (9, 9)), ((5, 5), (3, 3)), ((6, 7), (11, 9)), ((7, 6), (3, 14))]:
            for y in range(hw[0]):
                for x in range(hw[1]):
                    s = r.uniform(0, 80, hw).astype(np.float32)
                    s[y, x] = val
                    ref = cv2.resize(s, (HW[1], HW[0]), interpolation=cv2.INTER_LINEAR)
                    assert bits_equal(resize_linear(s, HW), ref), (val, hw, HW, y, x)


def test_oracle_batch_equals_planes():
    from oracle.resize import resize_linear
    s = np.stack([plane((23, 41), "u0_80", k) for k in range(3)])
    out = resize_linear(s, (50, 17))
    for k in range(3):
        assert bits_equal(out[k], cv2.resize(s[k], (17, 50), interpolation=cv2.INTER_LINEAR))


def test_oracle_refuses_unpinned_shapes():
    from oracle.resize import resize_linear
    for hw in [(1, 50), (50, 1), (1, 1)]:
        with pytest.raises(ValueError):
            resize_linear(np.zeros(hw, np.float32), (4, 60))


def test_resize_supported_classes():
    import torch
    from mindtheedge_b200.edge import resize_supported
    assert resize_supported(np.float32, (2, 2)) and resize_supported(torch.float32, (3, 192, 640))
    assert not resize_supported(np.float64, (192, 640)) and not resize_supported(torch.float64, (192, 640))
    assert not resize_supported(np.float32, (1, 640)) and not resize_supported(np.float32, (192, 1))
    assert not resize_supported(np.uint16, (192, 640)) and not resize_supported(torch.uint8, (192, 640))


def test_resize_argument_checks_without_a_gpu():
    """mte_resize_linear validates every argument before it touches the device."""
    from mindtheedge_b200 import _lib
    L = _lib.lib
    F32, F64, U8 = _lib.MTE_F32, _lib.MTE_F64, _lib.MTE_U8
    assert L.mte_resize_linear(None, F32, 1, 8, 8, 256, 16, 16, None) == -1          # NULL src
    assert L.mte_resize_linear(256, F32, 1, 8, 8, None, 16, 16, None) == -1          # NULL dst
    for n, h, w, H, W in [(0, 8, 8, 16, 16), (1, 0, 8, 16, 16), (1, 8, -1, 16, 16), (1, 8, 8, 0, 16),
                          (1, 8, 8, 16, 0)]:
        assert L.mte_resize_linear(256, F32, n, h, w, 512, H, W, None) == -2         # shapes < 1
    assert L.mte_resize_linear(256, 7, 1, 8, 8, 512, 16, 16, None) == -4             # bad dtype
    assert L.mte_resize_linear(256, U8, 1, 8, 8, 512, 16, 16, None) == -4            # u8: not a depth plane
    assert L.mte_resize_linear(256, F64, 1, 8, 8, 512, 16, 16, None) == -4           # fp64: refused class
    assert L.mte_resize_linear(256, F32, 1, 1, 50, 512, 4, 60, None) == -2           # one-row source: refused
    assert L.mte_resize_linear(256, F32, 1, 50, 1, 512, 60, 4, None) == -2           # one-column source: refused
    assert L.mte_resize_linear(258, F32, 1, 8, 8, 512, 16, 16, None) == -5           # misaligned src
    assert L.mte_resize_linear(256, F32, 1, 8, 8, 514, 16, 16, None) == -5           # misaligned dst
