"""The device resize of predicted depth (``mte_resize_linear``) against the oracle, which equals ``cv2.resize``
INTER_LINEAR bit for bit (test_resize_cpu.py), and the evaluation paths that now resize on the device against the
same calls on host-resized arrays."""
import os
import tempfile

import cv2
import numpy as np
import pytest
import torch

from test_resize_cpu import SHAPES, VALUES, bits_equal, plane

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("k", range(len(SHAPES)))
def test_op_equals_oracle(k):
    """Every value set of one shape in ONE batched call (N = 5) against the oracle per plane."""
    from mindtheedge_b200.edge import resize_linear
    from oracle.resize import resize_linear as ref_resize
    hw, HW = SHAPES[k]
    src = np.stack([plane(hw, values, 100 * k + v) for v, values in enumerate(VALUES)])
    got = resize_linear(torch.from_numpy(src).cuda(), HW).cpu().numpy()
    assert got.dtype == np.float32 and got.shape == (len(VALUES),) + tuple(HW)
    ref = ref_resize(src, HW)
    for v in range(len(VALUES)):
        assert bits_equal(got[v], ref[v]), (hw, HW, VALUES[v])


def test_scalar_store_path_and_2d_input():
    """A 16-byte misaligned output (W % 4 == 0 but an odd offset in a larger buffer) takes the scalar stores; a 2-D
    input gives a 2-D output."""
    from mindtheedge_b200 import _lib
    from mindtheedge_b200.edge import resize_linear
    from oracle.resize import resize_linear as ref_resize
    s = plane((61, 90), "x1e6", 1)
    d = torch.from_numpy(s).cuda()
    out2d = resize_linear(d, (130, 200))
    assert out2d.shape == (130, 200) and bits_equal(out2d.cpu().numpy(), ref_resize(s, (130, 200)))
    buf = torch.full((130 * 200 + 1,), -7.0, device="cuda")
    rc = _lib.lib.mte_resize_linear(d.data_ptr(), _lib.MTE_F32, 1, 61, 90, buf.data_ptr() + 4, 130, 200,
                                    torch.cuda.current_stream().cuda_stream)
    assert rc == 0
    torch.cuda.synchronize()
    assert bits_equal(buf[1:].view(130, 200).cpu().numpy(), ref_resize(s, (130, 200)))
    assert buf[0].item() == -7.0


def test_non_contiguous_input():
    from mindtheedge_b200.edge import resize_linear
    from oracle.resize import resize_linear as ref_resize
    big = np.stack([plane((80, 120), "minus1", k) for k in range(4)])
    view = torch.from_numpy(big).cuda()[::2, :, ::3]            # [2, 80, 40], strided
    assert not view.is_contiguous()
    got = resize_linear(view, (160, 81)).cpu().numpy()
    ref = ref_resize(np.ascontiguousarray(big[::2, :, ::3]), (160, 81))
    assert bits_equal(got, ref)


def test_second_device_while_first_is_current():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from mindtheedge_b200.edge import resize_linear
    from oracle.resize import resize_linear as ref_resize
    s = np.stack([plane((96, 320), "u0_80", k) for k in range(3)])
    torch.cuda.set_device(0)
    got = resize_linear(torch.from_numpy(s).to("cuda:1"), (192, 640))
    assert got.device == torch.device("cuda:1") and torch.cuda.current_device() == 0
    assert bits_equal(got.cpu().numpy(), ref_resize(s, (192, 640)))


def test_refused_inputs_raise():
    from mindtheedge_b200 import _lib
    from mindtheedge_b200.edge import resize_linear
    with pytest.raises(_lib.MteError):
        resize_linear(torch.zeros(4, 8, dtype=torch.float64, device="cuda"), (8, 16))
    with pytest.raises(_lib.MteError):
        resize_linear(torch.zeros(1, 50, device="cuda"), (4, 60))
    with pytest.raises(_lib.MteError):
        resize_linear(torch.zeros(4, 8), (8, 16))                 # CPU tensor: no fallback


def test_edge_from_depth_new_shape():
    """edge_from_depth(new_shape) of a float32 .npy (device resize) equals Canny of the host-resized plane; a float64
    plane keeps the host resize and gives the same edges as before."""
    from mindtheedge_b200.edge import Canny, canny_from_depth, edge_from_depth
    from oracle.canny import quantise_depth
    r = np.random.default_rng(4)
    with tempfile.TemporaryDirectory() as tmp:
        for k, (hw, dsize) in enumerate([((96, 320), (640, 192)), ((61, 97), (200, 130)), ((200, 300), (77, 51))]):
            d = r.uniform(3, 80, hw).astype(np.float32)
            d[r.random(hw) < 0.05] = -1
            for dt in (np.float32, np.float64):
                path = os.path.join(tmp, f"d{k}.npy")
                np.save(path, d.astype(dt))
                got = edge_from_depth(path, dsize, None, thresh_1=20, thresh_2=40, is_write_edge=False)
                host = cv2.resize(d.astype(dt), dsize, interpolation=cv2.INTER_LINEAR)
                ref = canny_from_depth(torch.from_numpy(host).cuda(), [(20, 40)])[0].cpu().numpy()
                assert got.shape == (dsize[1], dsize[0]) and np.array_equal(got, ref), (k, dt)
                assert np.array_equal(Canny(quantise_depth(host, 0.0, 80.0), 20, 40), ref)


def _half_res(depths):
    """Host downsampling of the bench set to half resolution, before any timing or comparison."""
    return np.stack([cv2.resize(d, (d.shape[1] // 2, d.shape[0] // 2), interpolation=cv2.INTER_LINEAR)
                     for d in depths])


@pytest.fixture(scope="module")
def kitti():
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import bench
    depths, gts = bench.kitti_like_set(12, 7000)
    return _half_res(depths), gts, bench.KITTI_CROP


@pytest.mark.parametrize("per_image", [False, True])
def test_sweep_counts_half_resolution(kitti, per_image):
    """sweep_counts on half-resolution depth (device resize) equals sweep_counts on cv2.resize'd depth: 12 Canny
    settings, KITTI crop."""
    from mindtheedge_b200.eval_depth_edges import sweep_counts
    half, gts, crop = kitti
    H, W = gts.shape[1:]
    host = np.stack([cv2.resize(d, (W, H), interpolation=cv2.INTER_LINEAR) for d in half])
    rng = list(range(20, 241, 20))
    g = torch.from_numpy(gts).cuda()
    got = sweep_counts(torch.from_numpy(half).cuda(), g, rng, crop, 0.0, 80.0, per_image=per_image)
    ref = sweep_counts(torch.from_numpy(host).cuda(), g, rng, crop, 0.0, 80.0, per_image=per_image)
    assert torch.equal(got, ref)
    assert got.shape == ((len(half), 12, 4) if per_image else (12, 4))
    assert int(ref[..., 3].sum()) > 0


def _mixed_predictions(half, gts):
    """Mixed resolutions and dtypes: half-size float32 (device), full-size float32 (no resize), 3/4-size float32
    (device, another source shape), half-size float64 (host cv2.resize), a one-row float32 plane (host)."""
    H, W = gts.shape[1:]
    preds = []
    for i, d in enumerate(half):
        kind = i % 5
        if kind == 0:
            preds.append(d)
        elif kind == 1:
            preds.append(cv2.resize(d, (W, H), interpolation=cv2.INTER_LINEAR))
        elif kind == 2:
            preds.append(cv2.resize(d, (W * 3 // 4, H * 3 // 4), interpolation=cv2.INTER_LINEAR))
        elif kind == 3:
            preds.append(d.astype(np.float64))
        else:
            preds.append(np.ascontiguousarray(d[d.shape[0] // 2:d.shape[0] // 2 + 1]))
    return preds


@pytest.mark.parametrize("per_image", [False, True])
@pytest.mark.parametrize("branch", ["crop", "mask"])
def test_pr_evaluation_arrays_mixed_resolution(kitti, per_image, branch):
    """pr_evaluation_arrays from mixed-resolution predictions equals the same call on host-resized arrays, with the
    list crop and with a mask image, per_image on and off."""
    from mindtheedge_b200.eval_depth_edges import pr_evaluation_arrays
    half, gts, crop = kitti
    H, W = gts.shape[1:]
    preds = _mixed_predictions(half, gts)
    host = [p if p.shape == (H, W) else cv2.resize(p, (W, H), interpolation=cv2.INTER_LINEAR) for p in preds]
    gts255 = [g * 255 for g in gts]
    kw = dict(per_image=per_image, batch=4)
    if branch == "mask":
        m = np.zeros((H, W))
        m[100:300, 50:1100] = 1.0
        m[300:360, 50:1100] = 0.5
        kw["mask"] = m
    else:
        kw["gt_crop"] = crop
    got = pr_evaluation_arrays(preds, gts255, **kw)
    ref = pr_evaluation_arrays(host, gts255, **kw)
    assert got[0] == ref[0] and got[1] == ref[1]
    assert torch.equal(got[2], ref[2])
    if per_image:
        assert torch.equal(got[3], ref[3]) and np.array_equal(got[4], ref[4])
