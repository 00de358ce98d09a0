"""Every kernel path of the on-device target preparation (``targets.cu``) against ``oracle.targets``, bit for bit.

``test_targets_gpu.py`` checks the goldens and the shipped identity shapes.  Here:

* the edge resize at identity shapes (``edge_max_kernel`` + ``edge_resize_preserve_kernel``: the input max is the
  output max) and at every other shape (``edge_gather_kernel`` + ``edge_scale_kernel``: the ``/255 if max > 1`` rule
  on the max of the resized map): 1 x 1, single rows and columns, odd sizes, integer and non-integer down- and
  upsampling, mixed axes, extreme ratios; each batch mixes value regimes, since the rule is per image;
* the float64 rounding of ``int(s * (H / h))``, at shape pairs where it differs from exact ``s * H // h``;
* the max rule after downsampling: maps whose input max is > 1 while the resized map's max is <= 1;
* ``[B,1,h,w]`` and non-contiguous inputs, large batches;
* ``decode_normals`` at sizes below, at and far above one pass of its grid, non-contiguous and 4-D inputs, empty;
* ``prepare_targets(shapes=...)`` with non-identity shapes per scale.

``test_path_manifest`` restates the path selection of ``mte_edge_resize_preserve`` / ``mte_decode_normals`` and
checks that every path is taken by some case; it needs no GPU.
"""
import numpy as np
import pytest
import torch

from oracle import targets as ot

NUM_SMS = 148          # B200: decode_normals_kernel runs min(blocks, 8 * SMs) blocks of 256 threads
DECODE_PASS = NUM_SMS * 8 * 256

REGIMES = ("0/255", "0/1", "1..255", "zero", "single")


def edge_plane(regime, h, w, r):
    """One u8 edge map of a value regime."""
    if regime == "zero":
        return np.zeros((h, w), np.uint8)
    if regime == "single":
        a = np.zeros((h, w), np.uint8)
        a[r.integers(0, h), r.integers(0, w)] = r.integers(2, 256)
        return a
    on = r.random((h, w)) < 0.3
    if regime == "0/255":
        return (on * 255).astype(np.uint8)
    if regime == "0/1":
        return on.astype(np.uint8)
    return np.where(on, r.integers(1, 256, (h, w)), 0).astype(np.uint8)


# (h, w) -> (H, W)
SHAPES = [
    ((1, 1), (1, 1)), ((1, 37), (1, 37)), ((41, 1), (41, 1)), ((33, 57), (33, 57)),          # identity
    ((64, 96), (32, 48)), ((64, 96), (16, 24)), ((64, 96), (8, 12)),                         # integer down
    ((37, 53), (20, 31)), ((1216, 1936), (384, 640)),                                        # non-integer down
    ((24, 32), (48, 64)), ((7, 7), (10, 10)),                                                # up
    ((60, 20), (25, 47)), ((20, 60), (47, 25)), ((33, 57), (33, 20)), ((1, 37), (1, 80)),    # mixed axes
    ((1, 1), (5, 7)), ((384, 1280), (1, 1)), ((1, 1280), (384, 1)),                          # extremes
]


def rounding_pairs(limit=100):
    """(h, H, s): source index s of an axis of h resized to H where NumPy's int(s * (H / h)) is not s * H // h."""
    return [(h, H, s) for h in range(1, limit) for H in range(1, limit) for s in range(h)
            if int(s * (H / h)) != s * H // h]


def rounding_shapes():
    pairs = rounding_pairs()
    picked = {(88, 48), (94, 48), (22, 30)} | {(h, H) for h, H, _ in pairs[::9]}
    return sorted(picked)


def max_flip(e, shape):
    """The input's max is > 1 and the resized map's max is not."""
    return e.max() > 1 and ot.resize_depth_preserve(e, shape).max() <= 1


def flip_batch(hw, shape, seed, n=300):
    """Random {0,1,255} maps resized hw -> shape; returns the batch and how many maps flip."""
    r = np.random.default_rng(seed)
    e = r.choice(np.array([0, 1, 255], np.uint8), size=(n,) + hw, p=[0.5, 0.35, 0.15])
    return e, sum(max_flip(a, shape) for a in e)


# ---- the host's path selection (targets.cu: mte_edge_resize_preserve, mte_decode_normals) --------------------------
def resize_path(hw, shape):
    return "identity" if tuple(hw) == tuple(shape) else "gather"


def resize_tags(hw, shape):
    (h, w), (H, W) = hw, shape
    tags = {resize_path(hw, shape)} | ({"identity-1x1"} if (h, w) == (H, W) == (1, 1) else set())
    if tags == {"gather"}:
        for a, b, ax in ((h, H, "y"), (w, W, "x")):
            tags.add(f"{'down' if b < a else 'up' if b > a else 'same'}-{ax}")
            if b < a and a % b:
                tags.add("non-integer-down")
    return tags


def decode_path(n):
    return "empty" if n == 0 else "one-pass" if n <= DECODE_PASS else "grid-stride"


# ---- running -------------------------------------------------------------------------------------------------------
def _check_resize(e, shape, src=None):
    """e: u8 [B,h,w] numpy; src: the device tensor handed to the op (default: e on the device)."""
    from mindtheedge_b200.targets import resize_edge_preserve
    got = resize_edge_preserve(torch.from_numpy(e).cuda() if src is None else src, shape)
    assert got.shape == (e.shape[0], 1) + tuple(shape) and got.dtype == torch.float32
    got = got.cpu().numpy()
    for b in range(e.shape[0]):
        want = ot.edge_target(e[b], shape)
        assert np.array_equal(got[b, 0], want), (b, np.argwhere(got[b, 0] != want)[:5].tolist())


@pytest.mark.gpu
@pytest.mark.parametrize("k", range(len(SHAPES)))
def test_resize_shape_matrix(k):
    hw, shape = SHAPES[k]
    r = np.random.default_rng(100 + k)
    regimes = [REGIMES[(k + j) % len(REGIMES)] for j in range(3)]
    e = np.stack([edge_plane(g, *hw, r) for g in regimes])
    _check_resize(e, shape)


@pytest.mark.gpu
def test_resize_float64_rounding_pairs():
    """Each axis resized between sizes whose scale H / h rounds so that int(s * (H / h)) differs from s * H // h for
    some s: source_range's +-2 window and __dmul_rn must follow NumPy's float64 product, not exact arithmetic."""
    pairs = rounding_pairs()
    assert (88, 48, 55) in pairs and (94, 48, 47) in pairs and (22, 30, 11) in pairs
    r = np.random.default_rng(7)
    for h, H in rounding_shapes():
        # every source pixel valid and distinct along the axis, so a misplaced one shows
        ramp = np.arange(1, h + 1, dtype=np.uint8)
        along_y = np.stack([np.repeat(ramp[:, None], 3, 1), np.repeat(ramp[::-1, None], 3, 1)])
        _check_resize(along_y, (H, 3))
        _check_resize(np.ascontiguousarray(along_y.transpose(0, 2, 1)), (3, H))
        _check_resize(edge_plane("1..255", h, h, r)[None], (H, H))


@pytest.mark.gpu
def test_max_rule_on_the_resized_map():
    """200 at (2, 3) and 1 at (7, 7) of an 8x8 map resized to 1x1: the last valid pixel (value 1) wins, the output's
    max is 1, so it is not divided by 255: 1.0, not 1/255."""
    from mindtheedge_b200.targets import resize_edge_preserve
    e = np.zeros((8, 8), np.uint8)
    e[2, 3], e[7, 7] = 200, 1
    assert ot.edge_target(e, (1, 1))[0, 0] == 1.0
    got = resize_edge_preserve(torch.from_numpy(e)[None].cuda(), (1, 1))
    assert got.item() == 1.0
    _check_resize(e[None], (1, 1))


@pytest.mark.gpu
@pytest.mark.parametrize("hw,shape", [((12, 10), (3, 2)), ((8, 8), (1, 1)), ((16, 24), (2, 3)), ((31, 29), (2, 3))])
def test_max_rule_random_downsamples(hw, shape):
    e, flips = flip_batch(hw, shape, 11 + hw[0])
    assert flips >= 5, flips
    _check_resize(e, shape)


@pytest.mark.gpu
def test_max_rule_one_image_flips():
    """Only the middle image of three has an input max > 1 and an output max <= 1."""
    r = np.random.default_rng(12)
    e = np.stack([edge_plane("0/255", 12, 10, r), np.zeros((12, 10), np.uint8), edge_plane("1..255", 12, 10, r)])
    e[1, 0, 0], e[1, 3, 4] = 255, 1
    assert [max_flip(a, (3, 2)) for a in e] == [False, True, False]
    _check_resize(e, (3, 2))


@pytest.mark.gpu
def test_resize_input_layouts():
    from mindtheedge_b200.targets import resize_edge_preserve
    r = np.random.default_rng(13)
    e = np.stack([edge_plane(REGIMES[b % 5], 37, 53, r) for b in range(4)])
    # [B,1,h,w]
    _check_resize(e, (20, 31), torch.from_numpy(e)[:, None].cuda())
    # non-contiguous: every other image of a batch, transposed planes
    big = np.stack([edge_plane(REGIMES[b % 5], 53, 37, r) for b in range(8)])
    view = torch.from_numpy(big).cuda()[::2].transpose(1, 2)
    assert not view.is_contiguous()
    _check_resize(np.ascontiguousarray(big[::2].transpose(0, 2, 1)), (20, 31), view)
    _check_resize(np.ascontiguousarray(big[::2].transpose(0, 2, 1)), (37, 53), view)
    # B = 70 at identity and downsampled shapes
    e70 = np.stack([edge_plane(REGIMES[b % 5], 24, 40, r) for b in range(70)])
    _check_resize(e70, (24, 40))
    _check_resize(e70, (7, 13))
    assert resize_edge_preserve(torch.from_numpy(e70).cuda(), (7, 13)).shape == (70, 1, 7, 13)


def _normal_values(n, r):
    """n u8 values holding every value 0..255 at random places when n >= 256."""
    v = r.integers(0, 256, n).astype(np.uint8)
    if n >= 256:
        v[r.choice(n, 256, replace=False)] = np.arange(256, dtype=np.uint8)
    return v


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(1,), (255,), (256,), (257,), (8, 1216, 1936)])
def test_decode_normals_sizes(shape):
    from mindtheedge_b200.targets import decode_normals
    r = np.random.default_rng(int(np.prod(shape)) % 1000)
    v = _normal_values(int(np.prod(shape)), r).reshape(shape)
    got = decode_normals(torch.from_numpy(v).cuda())
    assert got.shape == shape and got.dtype == torch.float32
    assert np.array_equal(got.cpu().numpy(), ot.decode_normals(v))


@pytest.mark.gpu
def test_decode_normals_layouts_and_empty():
    from mindtheedge_b200.targets import decode_normals
    r = np.random.default_rng(14)
    v = _normal_values(3 * 2 * 50 * 70, r).reshape(3, 2, 50, 70)
    got = decode_normals(torch.from_numpy(v).cuda())
    assert got.shape == v.shape and np.array_equal(got.cpu().numpy(), ot.decode_normals(v))
    view = torch.from_numpy(v).cuda()[:, 1].transpose(1, 2)[..., ::3]
    assert not view.is_contiguous()
    want = ot.decode_normals(v[:, 1].transpose(0, 2, 1)[..., ::3])
    assert np.array_equal(decode_normals(view).cpu().numpy(), want)
    empty = decode_normals(torch.empty((0, 5), dtype=torch.uint8, device="cuda"))
    assert empty.shape == (0, 5) and empty.dtype == torch.float32


@pytest.mark.gpu
def test_prepare_targets_with_shapes():
    """Per-scale planes resized to other shapes than their own (down, up, mixed, identity), batch of 3 with mixed
    value regimes; the normals are decoded at their own shape."""
    from mindtheedge_b200.targets import prepare_targets
    r = np.random.default_rng(15)
    planes = [(96, 320), (48, 160), (24, 80), (12, 40)]
    shapes = [(48, 160), (24, 80), (36, 50), (12, 40)]
    e8 = [np.stack([edge_plane(REGIMES[(s + b) % 5], *hw, r) for b in range(3)]) for s, hw in enumerate(planes)]
    n8 = [r.integers(0, 256, (3,) + hw).astype(np.uint8) for hw in planes]
    edges, normals = prepare_targets([torch.from_numpy(a).cuda() for a in e8],
                                     [torch.from_numpy(a).cuda() for a in n8], shapes=shapes)
    for s in range(4):
        assert edges[s].shape == (3, 1) + shapes[s] and normals[s].shape == (3, 1) + planes[s]
        for b in range(3):
            assert np.array_equal(edges[s][b, 0].cpu().numpy(), ot.edge_target(e8[s][b], shapes[s])), (s, b)
            assert np.array_equal(normals[s][b, 0].cpu().numpy(), ot.decode_normals(n8[s][b])), (s, b)


# ---- coverage manifest (no GPU work) --------------------------------------------------------------------------------
def test_path_manifest():
    """Every path of the resize and the decode is taken by some case above, the rounding search finds the pairs the
    rounding test needs, and the max-rule cases do flip."""
    seen = set()
    for hw, shape in SHAPES:
        seen |= resize_tags(hw, shape)
    for h, H in rounding_shapes():
        seen |= resize_tags((h, 3), (H, 3))
    seen |= resize_tags((37, 53), (20, 31)) | resize_tags((24, 40), (7, 13))
    for shape in [(1,), (255,), (256,), (257,), (8, 1216, 1936), (0, 5)]:
        seen.add("decode-" + decode_path(int(np.prod(shape))))
    want = {"identity", "identity-1x1", "gather", "down-y", "down-x", "up-y", "up-x", "same-y", "same-x",
            "non-integer-down", "decode-empty", "decode-one-pass", "decode-grid-stride"}
    assert want <= seen, sorted(want - seen)
    # every downsampled gather that can flip the max rule does so in some case
    assert sum(max_flip(a, (3, 2)) for a in flip_batch((12, 10), (3, 2), 23)[0]) > 0
    assert 8 * 1216 * 1936 > 50 * DECODE_PASS
    # rounding: the search finds pairs, among them the ones named in the rounding test
    pairs = rounding_pairs()
    assert len(pairs) > 10 and all(int(s * (H / h)) != s * H // h for h, H, s in pairs)
    assert {(88, 48, 55), (94, 48, 47), (22, 30, 11)} <= set(pairs)
    # every regime appears in some batch of the shape matrix
    assert {REGIMES[(k + j) % 5] for k in range(len(SHAPES)) for j in range(3)} == set(REGIMES)
