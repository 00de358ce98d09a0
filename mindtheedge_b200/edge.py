"""Depth -> edge extraction: drop-in for the reference ``edge.py`` /
``packnet_sfm/utils/edge.py``.

* ``edge_from_depth``  same signature and return value as ``edge.py:73-93``
  (file path in, ``np.uint8[H,W]`` in {0,255} out, optional image write);
  ``edge_from_depth_cfg`` is the cfg-taking twin of ``utils/edge.py:64-89``.
* ``Canny``            ``cv2.Canny(u8, t1, t2)`` replacement for the bare calls in
  ``models/model_wrapper.py:399-401``.
* ``chamfer_distance`` / ``compute_edge_metrics``  the in-training "light" edge metric of
  ``utils/edge.py:20-62`` and ``models/model_wrapper.py:376-442`` (3 Canny settings, chamfer
  precision / recall / F1) without the host round trip and the scipy EDT.
* ``canny_from_depth`` the tensor-level op the evaluation pipeline uses: a batch
  of depth planes and T threshold pairs in, either the T edge planes or the
  single "birth level" plane out (no host round trip).

* ``resize_linear``    ``cv2.resize(depth, (W, H), interpolation=cv2.INTER_LINEAR)`` of ``edge.py:76-78`` on the
  device, bit-exact for float32 planes of at least 2 x 2 (``mte_resize_linear``).

All arithmetic after the file read runs in libmte.so (``mte_resize_linear``, ``mte_canny_from_depth``); there is no
CPU fallback.  File decode stays on the host (IO).  The optional resize to the GT size is per-pixel arithmetic and
runs on the device for float32 planes of at least 2 x 2; for the inputs whose ``cv2.resize`` arithmetic is not pinned
(float64, one-row or one-column planes, DESIGN.md section 2) it stays ``cv2.resize`` on the host, so that no result
differs from the reference.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib, runtime

__all__ = ["canny_from_depth", "resize_linear", "resize_supported", "edge_from_depth", "edge_from_depth_cfg", "Canny", "read_depth_file",
           "chamfer_counts", "chamfer_distance", "compute_edge_metrics"]

_DT = {torch.float32: _lib.MTE_F32, torch.float64: _lib.MTE_F64, torch.uint8: _lib.MTE_U8}


def _canny_from_depth_cuda(depth, lows, highs, min_depth, max_depth, want_edges, want_levels):
    """CUDA implementation of ``mte::canny_from_depth``: depth [N,H,W] -> (edges [T,N,H,W] or empty, levels [N,H,W]
    or empty), both uint8."""
    with runtime.on_device(depth) as dev:
        d = depth.contiguous()
        N, H, W = d.shape
        T = len(lows)
        lo = (C.c_int32 * T)(*[int(v) for v in lows])
        hi = (C.c_int32 * T)(*[int(v) for v in highs])
        edges = torch.empty((T, N, H, W) if want_edges else (0,), dtype=torch.uint8, device=dev)
        levels = torch.empty((N, H, W) if want_levels else (0,), dtype=torch.uint8, device=dev)
        ws = runtime.workspace(dev, _lib.lib.mte_canny_workspace_bytes(N, H, W, T))
        runtime.call("mte_canny_from_depth", dev, d.data_ptr(), _DT[d.dtype], N, H, W, float(min_depth),
                     float(max_depth), lo, hi, T, edges.data_ptr() if want_edges else None,
                     levels.data_ptr() if want_levels else None, ws.data_ptr(), ws.numel(),
                     runtime.current_stream_ptr(dev))
    return edges, levels


runtime.define_op("canny_from_depth(Tensor depth, int[] lows, int[] highs, float min_depth, float max_depth, "
                  "bool want_edges, bool want_levels) -> (Tensor, Tensor)", _canny_from_depth_cuda)


def canny_from_depth(depth: torch.Tensor, pairs: Sequence[Tuple[int, int]], min_depth: float = 0.0,
                     max_depth: float = 80.0, *, want_edges: bool = True, want_levels: bool = False):
    """depth: CUDA tensor [N,H,W] (or [H,W]) of float32/float64 metres, or uint8
    (already quantised).  pairs: (low, high) per Canny setting.

    Returns ``edges`` uint8 [T,N,H,W] in {0,255} and/or ``levels`` uint8 [N,H,W]
    (index of the first pair at which the pixel is an edge, 255 = never; needs
    nested pairs, strictest first).  Runs as the torch custom op ``mte::canny_from_depth``."""
    runtime.require_cuda(depth, "depth")
    if depth.dtype not in _DT:
        raise _lib.MteError(f"unsupported depth dtype {depth.dtype}")
    squeeze = depth.dim() == 2
    d = depth.unsqueeze(0) if squeeze else depth
    if d.dim() != 3:
        raise _lib.MteError("depth must be [N,H,W] or [H,W]")
    lows = [int(np.floor(p[0])) for p in pairs]
    highs = [int(np.floor(p[1])) for p in pairs]
    edges, levels = torch.ops.mte.canny_from_depth(d, lows, highs, float(min_depth), float(max_depth),
                                                   bool(want_edges), bool(want_levels))
    edges = edges if want_edges else None
    levels = levels if want_levels else None
    if squeeze:
        edges = None if edges is None else edges[:, 0]
        levels = None if levels is None else levels[0]
    if want_edges and want_levels:
        return edges, levels
    return edges if want_edges else levels


def _resize_linear_cuda(src, H, W):
    """CUDA implementation of ``mte::resize_linear``: src [N,h,w] -> [N,H,W] of the same dtype."""
    with runtime.on_device(src) as dev:
        s = src.contiguous()
        N, h, w = s.shape
        out = torch.empty((N, H, W), dtype=s.dtype, device=dev)
        runtime.call("mte_resize_linear", dev, s.data_ptr(), _DT.get(s.dtype, -1), N, h, w, out.data_ptr(), H, W,
                     runtime.current_stream_ptr(dev))
    return out


runtime.define_op("resize_linear(Tensor src, int H, int W) -> Tensor", _resize_linear_cuda)


def resize_supported(dtype, shape) -> bool:
    """Whether ``resize_linear`` takes a plane of this dtype (NumPy or torch) and [h,w] (or [N,h,w]) shape: float32
    with h, w >= 2, the inputs on which the kernel is pinned bit for bit against ``cv2.resize``."""
    f32 = dtype == torch.float32 if isinstance(dtype, torch.dtype) else np.dtype(dtype) == np.float32
    return f32 and len(shape) in (2, 3) and min(shape[-2:]) >= 2


def resize_linear(src: torch.Tensor, size) -> torch.Tensor:
    """``cv2.resize(src, (W, H), interpolation=cv2.INTER_LINEAR)`` on the device, bit for bit.

    src   CUDA float32 [N,h,w] or [h,w], h and w >= 2 (other inputs raise ``MteError``: see ``resize_supported``).
    size  (H, W) -- rows first, unlike cv2's dsize.
    ->    float32 [N,H,W] or [H,W] on src's device.  Torch custom op ``mte::resize_linear``."""
    runtime.require_cuda(src, "src")
    if src.dim() not in (2, 3):
        raise _lib.MteError("src must be [N,h,w] or [h,w]")
    if not resize_supported(src.dtype, tuple(src.shape)):
        raise _lib.MteError(f"resize_linear takes float32 planes of at least 2 x 2, got {src.dtype} "
                            f"{tuple(src.shape)}")
    H, W = (int(v) for v in size)
    squeeze = src.dim() == 2
    out = torch.ops.mte.resize_linear(src.unsqueeze(0) if squeeze else src, H, W)
    return out[0] if squeeze else out


def read_depth_file(file: str) -> np.ndarray:
    """edge.py:95-116 (``.npy`` as stored; ``.png`` as raw integer values with 0 -> -1)."""
    ext = file.split(".")[-1]
    if ext == "npy":
        return np.load(file)
    if ext == "png":
        from PIL import Image
        im = Image.open(file)
        if im.mode == "RGBA":
            im = im.convert("RGB")
        png = np.array(im, dtype=int)
        depth = png.astype(np.float64)
        depth[png == 0] = -1.0
        return depth
    raise ValueError(f"unsupported depth file {file!r}")


def _edges_of_array(depth_im: np.ndarray, new_shape, min_depth, max_depth, thresh_1, thresh_2) -> np.ndarray:
    on_device = new_shape is not None and resize_supported(depth_im.dtype, depth_im.shape) and depth_im.ndim == 2
    if new_shape is not None and not on_device:
        import cv2
        depth_im = cv2.resize(depth_im, new_shape, interpolation=cv2.INTER_LINEAR)
    if depth_im.dtype not in (np.float32, np.float64):
        depth_im = depth_im.astype(np.float64)
    d = torch.from_numpy(np.ascontiguousarray(depth_im)).cuda(non_blocking=True)
    if on_device:   # new_shape is cv2's dsize, (width, height)
        d = resize_linear(d, (int(new_shape[1]), int(new_shape[0])))
    e = canny_from_depth(d, [(thresh_1, thresh_2)], min_depth, max_depth)
    return e[0].cpu().numpy()


def edge_from_depth(depth_gt, new_shape, name_edge_im, min_depth=0.0, max_depth=80.0, thresh_1=20, thresh_2=40,
                    is_write_edge=True):
    """Drop-in for ``edge.edge_from_depth`` (edge.py:73-93)."""
    depth_im = read_depth_file(depth_gt.split("\n")[0])
    edge_im = _edges_of_array(depth_im, new_shape, min_depth, max_depth, thresh_1, thresh_2)
    if is_write_edge:
        import cv2
        cv2.imwrite(name_edge_im, edge_im)
    return edge_im


def edge_from_depth_cfg(depth_gt, new_shape, name_edge_im, cfg, thresh_1=20, thresh_2=40, is_write_edge=True):
    """Drop-in for ``packnet_sfm.utils.edge.edge_from_depth`` (utils/edge.py:64-89)."""
    return edge_from_depth(depth_gt, new_shape, name_edge_im, cfg.analysis.min_depth, cfg.analysis.max_depth,
                           thresh_1, thresh_2, is_write_edge)


def Canny(image: np.ndarray, threshold1, threshold2) -> np.ndarray:
    """``cv2.Canny(image_u8, t1, t2)`` (aperture 3, L2gradient=False) on the GPU."""
    img = np.ascontiguousarray(image)
    if img.dtype != np.uint8 or img.ndim != 2:
        raise _lib.MteError("Canny expects a 2-D uint8 image")
    d = torch.from_numpy(img).cuda(non_blocking=True)
    return canny_from_depth(d, [(threshold1, threshold2)])[0].cpu().numpy()


# ---------------------------------------------------------------------------
# in-training "light" edge metric
# ---------------------------------------------------------------------------
def _chamfer_counts_cuda(pred, gt, thresh, want_map):
    with runtime.on_device(pred, gt) as dev:
        pred, gt = pred.contiguous(), gt.contiguous()
        N, H, W = pred.shape
        out = torch.empty((N, 4), dtype=torch.float64, device=dev)
        cond = torch.empty((N, H, W) if want_map else (0,), dtype=torch.int8, device=dev)
        ws = runtime.workspace(dev, _lib.lib.mte_chamfer_workspace_bytes(N, H, W))
        runtime.call("mte_chamfer_counts", dev, pred.data_ptr(), gt.data_ptr(), N, H, W, float(thresh),
                     out.data_ptr(), cond.data_ptr() if want_map else None, ws.data_ptr(), ws.numel(),
                     runtime.current_stream_ptr(dev))
    return out, cond


runtime.define_op("chamfer_counts(Tensor pred, Tensor gt, float thresh, bool want_map) -> (Tensor, Tensor)",
                  _chamfer_counts_cuda)


def chamfer_counts(pred: torch.Tensor, gt: torch.Tensor, edge_to_edge_thresh: float = 5, want_map: bool = False):
    """pred, gt: CUDA uint8 [N,H,W] edge maps (set = value/255 > 0.5).
    -> float64 [N,4] on the device: sum of the exact Euclidean distances from every pred pixel to the nearest
    gt pixel, number of pred pixels, number of pred pixels closer than the threshold, 0; and, with ``want_map``,
    the int8 [N,H,W] map (-1 not a pred pixel, 1 close, 0 not).  Torch custom op ``mte::chamfer_counts``."""
    runtime.require_cuda(pred, "pred")
    runtime.require_cuda(gt, "gt")
    if pred.dtype != torch.uint8 or gt.dtype != torch.uint8 or pred.shape != gt.shape or pred.dim() != 3:
        raise _lib.MteError("chamfer_counts expects two uint8 [N,H,W] maps of the same shape")
    out, cond = torch.ops.mte.chamfer_counts(pred, gt, float(edge_to_edge_thresh), bool(want_map))
    return (out, cond) if want_map else out


def chamfer_distance(im_pred, im_gt, mask=None, edge_to_edge_thresh=5):
    """Drop-in for ``packnet_sfm.utils.edge.chamfer_distance`` (utils/edge.py:20-62) for 2-D maps:
    -> (c_dist, percentage, edges_cond_reshaped).  ``mask`` must be None: the reference's mask branch only
    broadcasts for 3-channel images (utils/edge.py:27-28) and no call site passes one."""
    if mask is not None:
        raise NotImplementedError("chamfer_distance: the mask branch of the reference is 3-channel only and unused")
    p = np.ascontiguousarray(im_pred)
    g = np.ascontiguousarray(im_gt)
    if p.ndim != 2 or p.shape != g.shape:
        raise _lib.MteError("chamfer_distance expects two 2-D maps of the same shape")
    # value / 255 > 0.5 for any numeric dtype -> the u8 convention of the kernel
    pb = torch.from_numpy(((p / 255) > 0.5).astype(np.uint8) * 255).cuda()
    gb = torch.from_numpy(((g / 255) > 0.5).astype(np.uint8) * 255).cuda()
    out, cond = chamfer_counts(pb[None], gb[None], edge_to_edge_thresh, want_map=True)
    s, n, k, _ = out[0].cpu().numpy()
    with np.errstate(invalid="ignore", divide="ignore"):
        c_dist = np.float64(s) / np.float64(n)
        percentage = np.float64(k) / np.float64(n)
    return c_dist, percentage, cond[0].cpu().numpy().astype(np.float64)


def compute_edge_metrics(depth: torch.Tensor, edge: torch.Tensor, gt_crop=None, edge_model: bool = False):
    """Device version of ``ModelWrapper.compute_edge_metrics`` (models/model_wrapper.py:376-442).

    depth  CUDA [H,W] (or [1,1,H,W]): predicted DEPTH at the GT size (``inv2depth`` + resize already applied),
           or, with ``edge_model``, the predicted edge probability map (thresholds 0.5 / 0.75 / 0.9).
    edge   CUDA [H,W] GT edge map in [0,1] (the reference multiplies by 255 and binarises at 0.5, here in the
           map's own floating dtype, as NumPy would; other dtypes in float32).
    ->     the 9 numbers the reference appends: for each of the three settings, chamfer precision
           (pred px within < 5 px of a GT px), recall (the converse) and their harmonic mean."""
    d = depth.reshape(depth.shape[-2], depth.shape[-1])
    g = edge.reshape(edge.shape[-2], edge.shape[-1])
    runtime.require_cuda(d, "depth")
    runtime.require_cuda(g, "edge")
    if edge_model:
        preds = torch.stack([(d > t).to(torch.uint8) * 255 for t in (0.5, 0.75, 0.9)])
    else:
        d = d.float()
        # depth * (255 / max) -> uint8 (model_wrapper.py:396-397), then the three Canny settings of :399-401 in one
        # nested sweep (strictest first)
        mx = float(d.max().item())
        lv = canny_from_depth(d, [(30, 60), (20, 40), (10, 20)], float("-inf"), mx, want_edges=False,
                              want_levels=True)
        preds = torch.stack([(lv <= t).to(torch.uint8) * 255 for t in (2, 1, 0)])
    g = g if g.is_floating_point() else g.float()
    gt = ((g * 255) / 255 > 0.5).to(torch.uint8) * 255
    if gt_crop is not None and len(gt_crop) > 0:
        c = gt_crop
        gt = gt[c[2]:c[3], c[0]:c[1]]
        preds = preds[:, c[2]:c[3], c[0]:c[1]]
    gts = gt[None].expand_as(preds).contiguous()
    preds = preds.contiguous()
    a = chamfer_counts(preds, gts).cpu().numpy()   # pred -> gt
    b = chamfer_counts(gts, preds).cpu().numpy()   # gt -> pred
    out = []
    with np.errstate(invalid="ignore", divide="ignore"):
        for i in range(3):
            p1 = np.float64(a[i, 2]) / np.float64(a[i, 1])
            p2 = np.float64(b[i, 2]) / np.float64(b[i, 1])
            out += [p1, p2, 2 * ((p1 * p2) / (p1 + p2))]
    return out
