"""Depth-edge precision/recall evaluation: drop-in for the reference
``eval_depth_edges.py``.

Function names, arguments and return values follow the reference
(``evaluate_boundaries`` :67, ``evaluate_boundaries_bin`` :18,
``compute_rec_prec_f1`` :147, ``pr_evaluation`` :232,
``mean_recall_at_precision_range`` :365).  The per-pixel work -- Canny
extraction for every threshold, binarise + crop, the bipartite matcher and the
four counts -- runs in libmte.so on the GPU; the final P/R/AUC arithmetic on
``[T]`` vectors stays in NumPy, exactly as in the reference (SURVEY.md a16).

Differences from the reference wiring, none of which changes a count:
* predicted edge maps are never written to disk; the reference round-trips them
  through a lossy JPEG and re-thresholds at 0.5 (edge.py:90-91,
  eval_depth_edges.py:191-194), which flips no pixel of a {0,255} map;
* the 12 Canny settings share one NMS pass and one hysteresis pass (a single
  "birth level" plane), and all (image, threshold) matchings run concurrently
  instead of in a 4-process pool (:262, :296);
* with ``torch.distributed`` initialised, images are sharded over ranks and the
  ``int64[T,4]`` counts are summed with ONE all-reduce (mirrors the Python
  ``sum`` at :298-301).
"""
from __future__ import annotations

import ctypes as C
import os
from collections import namedtuple
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import _lib, runtime
from .edge import canny_from_depth, read_depth_file, resize_linear, resize_supported

__all__ = [
    "EvalResult", "_pred_eval", "pr_counts", "correspond_pixels_batch", "evaluate_boundaries", "evaluate_boundaries_bin",
    "compute_rec_prec_f1", "pr_evaluation", "pr_evaluation_arrays", "mean_recall_at_precision_range",
    "shard_indices", "all_reduce_counts", "sweep_counts", "evaluate_boundaries_batch",
]

_DT = {torch.float32: _lib.MTE_F32, torch.float64: _lib.MTE_F64, torch.uint8: _lib.MTE_U8}


# ---------------------------------------------------------------------------
# tensor-level ops
# ---------------------------------------------------------------------------
def _pr_counts_cuda(pred, gt, thresholds, n_levels, max_dist, crop, apply_thinning=False, per_image=False):
    """CUDA implementation of ``mte::pr_counts`` -> int64 [T,4] (count_r, sum_r, count_p, sum_p), or with
    ``per_image`` int64 [N,T,4]."""
    with runtime.on_device(pred, gt) as dev:
        pred, gt = pred.contiguous(), gt.contiguous()
        N, H, W = pred.shape
        if pred.dtype == torch.uint8:
            T, thr = int(n_levels), None
        else:
            t = np.ascontiguousarray(np.asarray(thresholds, dtype=np.float64))
            T = int(t.shape[0])
            thr = t.ctypes.data_as(C.POINTER(C.c_double))
        out = torch.zeros((N, T, 4) if per_image else (T, 4), dtype=torch.int64, device=dev)
        cr = None if len(crop) == 0 else (C.c_int32 * 4)(*[int(v) for v in crop])
        query = _lib.lib.mte_pr_thin_workspace_bytes if apply_thinning else _lib.lib.mte_pr_workspace_bytes
        ws = runtime.workspace(dev, query(N, H, W, T, float(max_dist)))
        runtime.call("mte_pr_counts_per_image" if per_image else "mte_pr_counts", dev, pred.data_ptr(),
                     _DT[pred.dtype], gt.data_ptr(), N, H, W, cr, thr, T, float(max_dist), int(bool(apply_thinning)),
                     out.data_ptr(), ws.data_ptr(), ws.numel(), runtime.current_stream_ptr(dev))
    return out


def _correspond_pixels_cuda(a, b, max_dist, want_maps):
    with runtime.on_device(a, b) as dev:
        a, b = a.contiguous(), b.contiguous()
        Pn, h, w = a.shape
        ma = torch.empty(a.shape if want_maps else (0,), dtype=torch.uint8, device=dev)
        mb = torch.empty(b.shape if want_maps else (0,), dtype=torch.uint8, device=dev)
        cnt = torch.empty(Pn, dtype=torch.int64, device=dev)
        ws = runtime.workspace(dev, _lib.lib.mte_match_workspace_bytes(Pn, h, w, float(max_dist)))
        runtime.call("mte_correspond_pixels", dev, a.data_ptr(), b.data_ptr(), Pn, h, w, float(max_dist),
                     ma.data_ptr() if want_maps else None, mb.data_ptr() if want_maps else None, cnt.data_ptr(),
                     ws.data_ptr(), ws.numel(), runtime.current_stream_ptr(dev))
    return ma, mb, cnt


runtime.define_op("pr_counts(Tensor pred, Tensor gt, float[] thresholds, int n_levels, float max_dist, int[] crop, "
                  "bool apply_thinning=False, bool per_image=False) -> Tensor", _pr_counts_cuda)
runtime.define_op("correspond_pixels(Tensor a, Tensor b, float max_dist, bool want_maps) -> (Tensor, Tensor, Tensor)",
                  _correspond_pixels_cuda)


def pr_counts(pred: torch.Tensor, gt: torch.Tensor, thresholds=None, *, n_levels: Optional[int] = None,
              max_dist: float = 0.0075, crop: Optional[Sequence[int]] = None,
              out: Optional[torch.Tensor] = None, apply_thinning: bool = False, per_image: bool = False) -> torch.Tensor:
    """Counts for a batch of images, one GT map each (torch custom op ``mte::pr_counts``).

    pred  [N,H,W] CUDA: float32/float64 strength map (``pred >= thresholds[t]``) or uint8 level
          plane from ``canny_from_depth(..., want_levels=True)`` (edge at t iff level <= t; give
          ``n_levels``).
    gt    [N,H,W] uint8, non-zero = boundary.
    crop  ``[x0, x1, y0, y1]`` as the reference's ``gt_crop`` (python slices ``[y0:y1, x0:x1]``).
    apply_thinning  thin every binarised window before matching (``evaluate_boundaries``' default): the crop is
          applied first, so thinning zero-pads at the crop border; ``sum_p`` counts the thinned pixels.  Thresholds
          may then come in any order and repeat.
    per_image  return the counts of every image instead of their sum: int64 [N,T,4], row (i, t) for image i and
          threshold t, from the same single launch chain; summed over i it equals the default result.
    ->    int64 [T,4] on the device, columns count_r, sum_r, count_p, sum_p, summed over the
          batch (``per_image``: [N,T,4]) and ACCUMULATED into ``out`` when given."""
    runtime.require_cuda(pred, "pred")
    runtime.require_cuda(gt, "gt")
    if pred.dim() == 2:
        pred, gt = pred.unsqueeze(0), gt.unsqueeze(0)
    if pred.dtype not in _DT:
        raise _lib.MteError(f"unsupported pred dtype {pred.dtype}")
    if gt.dtype != torch.uint8:
        gt = (gt != 0).to(torch.uint8)
    if gt.shape != pred.shape:
        raise _lib.MteError("pred and gt must have the same [N,H,W] shape")
    if pred.dtype == torch.uint8:
        if n_levels is None:
            raise _lib.MteError("n_levels is required with a uint8 level plane")
        thr = []
    else:
        thr = [float(v) for v in np.asarray(thresholds, dtype=np.float64)]
    c = torch.ops.mte.pr_counts(pred, gt, thr, int(n_levels or 0), float(max_dist),
                                [] if crop is None else [int(v) for v in crop], bool(apply_thinning),
                                bool(per_image))
    if out is None:
        return c
    out += c
    return out


def correspond_pixels_batch(a: torch.Tensor, b: torch.Tensor, max_dist: float = 0.0075, want_maps: bool = True):
    """Maximum matching between boundary maps a[k], b[k] ([P,h,w] uint8 CUDA; torch custom op
    ``mte::correspond_pixels``).  -> (match_a, match_b, count int64[P])."""
    runtime.require_cuda(a, "a")
    runtime.require_cuda(b, "b")
    ma, mb, cnt = torch.ops.mte.correspond_pixels(a, b, float(max_dist), bool(want_maps))
    return (ma, mb, cnt) if want_maps else (None, None, cnt)


# ---------------------------------------------------------------------------
# NumPy-level mirrors of the reference functions
# ---------------------------------------------------------------------------
def _threshold_grid(thresholds):
    if isinstance(thresholds, int):
        return np.linspace(1.0 / (thresholds + 1), 1.0 - 1.0 / (thresholds + 1), thresholds)
    if isinstance(thresholds, np.ndarray):
        if thresholds.ndim != 1:
            raise ValueError("thresholds array should have 1 dimension, not {}".format(thresholds.ndim))
        return thresholds
    raise ValueError("thresholds should be an int or a NumPy array, not a {}".format(type(thresholds)))


def evaluate_boundaries(predicted_boundaries, gt_boundaries, thresholds=99, max_dist=0.0075,
                        apply_thinning=True, progress=None):
    """eval_depth_edges.py:67-145 -> (count_r, sum_r, count_p, sum_p, thresholds)."""
    thresholds = _threshold_grid(thresholds)
    T = thresholds.shape[0]
    pred = np.ascontiguousarray(predicted_boundaries)
    if pred.dtype not in (np.float32, np.float64):
        pred = pred.astype(np.float64)
    count_r = np.zeros(T)
    sum_r = np.zeros(T)
    count_p = np.zeros(T)
    sum_p = np.zeros(T)
    d_pred = torch.from_numpy(pred).cuda()
    if len(gt_boundaries) == 1 and (not apply_thinning or T <= _lib.MTE_MAX_THRESHOLDS):
        g_np = np.asarray(gt_boundaries[0])
        gt = torch.from_numpy(np.ascontiguousarray(g_np != 0).astype(np.uint8)).cuda()
        c = pr_counts(d_pred[None], gt[None], thresholds, max_dist=max_dist,
                      apply_thinning=bool(apply_thinning)).cpu().numpy()
        # the matcher sees "non-zero = boundary", but sum_r is gt.sum() (eval_depth_edges.py:138): for maps that are
        # not 0/1 (255-valued, soft, or multiplied by a fractional mask image) the two differ
        sum_r[:] = float(g_np.sum())
        return (c[:, 0].astype(np.float64), sum_r, c[:, 2].astype(np.float64), c[:, 3].astype(np.float64), thresholds)
    # general path (several GT maps, or more thresholds than one thinned sweep takes): binarise per threshold, thin,
    # match against every GT
    from .bsds import thin as _thin
    thr_dev = torch.from_numpy(np.asarray(thresholds, dtype=np.float64)).cuda()
    bins = (d_pred.double()[None] >= thr_dev[:, None, None]).to(torch.uint8)  # [T,h,w]
    if apply_thinning:
        bins = _thin.binary_thin_batch(bins)
    sum_p[:] = bins.flatten(1).sum(1).cpu().numpy()
    acc = torch.zeros_like(bins)
    for g in gt_boundaries:
        g_np = np.asarray(g)
        gt = torch.from_numpy(np.ascontiguousarray(g_np != 0).astype(np.uint8)).cuda()
        ma, mb, _ = correspond_pixels_batch(bins, gt[None].expand_as(bins).contiguous(), max_dist)
        acc |= ma
        sum_r += float(g_np.sum())
        count_r += mb.flatten(1).sum(1).cpu().numpy()
    count_p[:] = acc.flatten(1).sum(1).cpu().numpy()
    return count_r, sum_r, count_p, sum_p, thresholds


def evaluate_boundaries_bin(predicted_boundaries_bin, gt_boundaries, max_dist=0.0075, apply_thinning=True):
    """eval_depth_edges.py:18-65 -> (count_r, sum_r, count_p, sum_p)."""
    b = (np.asarray(predicted_boundaries_bin) != 0).astype(np.float64)
    c_r, s_r, c_p, s_p, _ = evaluate_boundaries(b, gt_boundaries, thresholds=np.array([0.5]), max_dist=max_dist,
                                                apply_thinning=apply_thinning)
    return c_r[0], s_r[0], c_p[0], s_p[0]


def evaluate_boundaries_batch(preds, gts, thresholds=99, max_dist=0.0075, apply_thinning=True):
    """``evaluate_boundaries`` for a list of 2-D predicted maps with one GT map each ->
    ``[evaluate_boundaries(p, [g], thresholds, max_dist, apply_thinning) for p, g in zip(preds, gts)]``, element for
    element.  Maps of one shape and dtype go to the device in one ``pr_counts(..., per_image=True)`` call; the cases
    the single-GT device path does not take (thinning with more than ``MTE_MAX_THRESHOLDS`` thresholds) run image by
    image."""
    thr = _threshold_grid(thresholds)
    T = thr.shape[0]
    if apply_thinning and T > _lib.MTE_MAX_THRESHOLDS:
        return [evaluate_boundaries(p, [g], thresholds, max_dist, apply_thinning) for p, g in zip(preds, gts)]
    maps = []
    for p in preds:
        p = np.ascontiguousarray(p)
        maps.append(p if p.dtype in (np.float32, np.float64) else p.astype(np.float64))
    groups = {}
    for i, p in enumerate(maps):
        groups.setdefault((p.shape, p.dtype), []).append(i)
    out = [None] * len(maps)
    for idx in groups.values():
        d_pred = torch.from_numpy(np.stack([maps[i] for i in idx])).cuda()
        g_np = [np.asarray(gts[i]) for i in idx]
        gt = torch.from_numpy(np.stack([(g != 0).astype(np.uint8) for g in g_np])).cuda()
        c = pr_counts(d_pred, gt, thr, max_dist=max_dist, apply_thinning=bool(apply_thinning),
                      per_image=True).cpu().numpy()
        for k, i in enumerate(idx):
            # sum_r is gt.sum() as in evaluate_boundaries (non-binary GT maps included)
            out[i] = (c[k, :, 0].astype(np.float64), np.full(T, float(g_np[k].sum())), c[k, :, 2].astype(np.float64),
                      c[k, :, 3].astype(np.float64), thr)
    return out


def compute_rec_prec_f1(count_r, sum_r, count_p, sum_p):
    """eval_depth_edges.py:147-161."""
    rec = count_r / (sum_r + (sum_r == 0))
    prec = count_p / (sum_p + (sum_p == 0))
    f1_denom = (prec + rec + ((prec + rec) == 0))
    f1 = 2.0 * prec * rec / f1_denom
    return rec, prec, f1


def mean_recall_at_precision_range(arr, small_lim=0.0, large_lim=1.0):
    """eval_depth_edges.py:365-375."""
    interp_x = np.array(range(int(small_lim * 100), int(large_lim * 100))) / 100
    interp_y = np.interp(interp_x, arr[:, 0], arr[:, 1])
    interp_y[interp_y < 0] = 0
    interp_y[interp_y > 1] = 1
    return np.mean(interp_y)


EvalResult = namedtuple('EvalResult', ['count_r_overall', 'sum_r_overall',
                                       'count_p_overall', 'sum_p_overall',
                                       'count_r_best', 'sum_r_best',
                                       'count_p_best', 'sum_p_best',
                                       'used_thresholds', 'recall', 'precision'])


def _crop_or_mask(crop):
    """``_pred_eval``'s ``crop`` argument (eval_depth_edges.py:182-189): the ``str()`` of a ``[x0,x1,y0,y1]`` list (or
    ``[]``), or the path of a mask IMAGE whose channel 0 / 255 multiplies both maps.  -> (crop list or None, mask)"""
    import ast
    import cv2
    if isinstance(crop, str):
        path = crop.split("\n")[0]
        if os.path.exists(path):
            return None, cv2.imread(path)[:, :, 0] / 255
        crop = ast.literal_eval(crop)
    return list(crop), None


def _pred_eval(pred_path, gt_path, crop):
    """Drop-in for eval_depth_edges.py:179-230: one predicted edge image against one GT edge image, binarised at
    0.5, cropped (or multiplied by a mask image), ``evaluate_boundaries(thresholds=1, apply_thinning=False,
    max_dist=0.002)`` -> ``EvalResult``."""
    import cv2
    crop, mask = _crop_or_mask(crop)

    def load(path):
        im = cv2.imread(path.split("\n")[0])[:, :, 0] / 255
        im[im > 0.5] = 1.0
        im[im < 0.5] = 0.0
        if mask is not None:
            return im * mask
        if len(crop) > 0:
            return im[crop[2]:crop[3], crop[0]:crop[1]]
        return im

    pred, gt_b = load(pred_path), load(gt_path)
    return _eval_result(*evaluate_boundaries(pred, [gt_b], thresholds=1, apply_thinning=False, max_dist=0.002))


def _eval_result(count_r, sum_r, count_p, sum_p, used_thresholds):
    """eval_depth_edges.py:212-230: the ``EvalResult`` of ``_pred_eval`` from its [T] count vectors."""
    rec, prec, f1 = compute_rec_prec_f1(count_r, sum_r, count_p, sum_p)
    best_ndx = np.argmax(f1)
    return EvalResult(count_r, sum_r, count_p, sum_p, count_r[best_ndx], sum_r[best_ndx], count_p[best_ndx],
                      sum_p[best_ndx], used_thresholds, rec, prec)


def _dist_info():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def shard_indices(n_items: int, rank: Optional[int] = None, world: Optional[int] = None) -> List[int]:
    """Image i of the evaluation goes to rank i mod R (SURVEY.md 8e)."""
    if rank is None or world is None:
        rank, world = _dist_info()
    return list(range(rank, n_items, world))


def all_reduce_counts(counts: torch.Tensor) -> torch.Tensor:
    """The ONE collective of the evaluation: integer sum of the int64[T,4] counts over ranks
    (the distributed form of the Python ``sum`` at eval_depth_edges.py:298-301).  Exact, so the
    result does not depend on the number of ranks."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(counts, op=dist.ReduceOp.SUM)
    return counts


_REORDER = {}


def _reorder_index(inv, device):
    """Cached device index that maps the strictest-first sweep order back to the caller's threshold order (a fresh
    pageable host -> device copy per call would synchronise the stream every evaluation)."""
    key = (inv, str(device))
    idx = _REORDER.get(key)
    if idx is None:
        idx = torch.tensor(inv, dtype=torch.long, device=device)
        _REORDER[key] = idx
    return idx


_SIDE_STREAMS: dict = {}


def _side_streams(device, n):
    key = (torch.device(device).index, n)
    if key not in _SIDE_STREAMS:
        _SIDE_STREAMS[key] = [torch.cuda.Stream(device) for _ in range(n)]
    return _SIDE_STREAMS[key]


def _sweep_chunk(depth, gt, pairs, gt_crop, min_depth, max_depth, max_dist, per_image=False):
    levels = canny_from_depth(depth, pairs, min_depth, max_depth, want_edges=False, want_levels=True)
    return pr_counts(levels, gt, n_levels=len(pairs), max_dist=max_dist, crop=gt_crop, per_image=per_image)


def sweep_counts(depth: torch.Tensor, gt: torch.Tensor, edge_thresh_range, gt_crop, min_depth, max_depth,
                 max_dist=0.002, out=None, pipeline_chunks: Optional[int] = None,
                 per_image: bool = False) -> torch.Tensor:
    """Device part of ``pr_evaluation`` for a batch: depth [N,h,w], gt [N,H,W] uint8 -> int64[len(range),4].
    Depth at another size than the GT is resized to it on the device first (``resize_linear``, bit-exact
    ``cv2.resize`` INTER_LINEAR as edge.py:76-78; float32 of at least 2 x 2 only, anything else raises).
    Thresholds are swept strictest first internally (the level plane needs nested pairs) and returned in the
    caller's order.  ``per_image`` returns the counts of every image,
    int64[N,len(range),4] (``_pred_eval``'s counts of image i at every setting in row i), from the same launches.

    ``pipeline_chunks`` > 1 cuts the batch into chunks on side streams (a chunk's NMS + hysteresis next to another
    chunk's matcher; counts are integer sums, the result does not depend on the chunking).  Measured on the bench set:
    no gain (1.686 / 1.684 / 1.690 / 1.671 ms for 1-4 chunks) -- the step is the chain NMS -> hysteresis -> matcher of
    its SLOWEST image, which no reordering of other images shortens -- so the default is one chunk."""
    if depth.shape[-2:] != gt.shape[-2:]:   # edge.py:76-78: the prediction is resized to the GT size first
        depth = resize_linear(depth, tuple(gt.shape[-2:]))
    order = np.argsort(-np.asarray(edge_thresh_range), kind="stable")
    pairs = [(int(edge_thresh_range[i] / 2), int(edge_thresh_range[i])) for i in order]
    N = depth.shape[0] if depth.dim() == 3 else 1
    chunks = pipeline_chunks if pipeline_chunks is not None else 1
    if chunks <= 1 or depth.dim() != 3:
        c = _sweep_chunk(depth, gt, pairs, gt_crop, min_depth, max_depth, max_dist, per_image)
    else:
        main = torch.cuda.current_stream(depth.device)
        bounds = [round(k * N / chunks) for k in range(chunks + 1)]
        parts = []
        for k, st in enumerate(_side_streams(depth.device, chunks)):
            st.wait_stream(main)
            with torch.cuda.stream(st):
                parts.append(_sweep_chunk(depth[bounds[k]:bounds[k + 1]], gt[bounds[k]:bounds[k + 1]], pairs, gt_crop,
                                          min_depth, max_depth, max_dist, per_image))
        for p, st in zip(parts, _side_streams(depth.device, chunks)):
            main.wait_stream(st)
            p.record_stream(main)
        if per_image:   # every chunk's rows at its images' offsets
            c = torch.cat(parts)
        else:
            c = parts[0]
            for p in parts[1:]:
                c = c + p
    idx = _reorder_index(tuple(int(v) for v in np.argsort(order)), c.device)
    c = c[:, idx] if per_image else c[idx]
    if out is not None:
        out += c
        return out
    return c


def _device_resizable(d: np.ndarray, H: int, W: int) -> bool:
    """A prediction that ``resize_linear`` brings to the GT size [H,W] on the device (float32 planes of at least
    2 x 2); every other plane of another size keeps the host ``cv2.resize``."""
    return d.ndim == 2 and d.shape != (H, W) and resize_supported(d.dtype, d.shape)


def _depth_planes(depths, chunk, H, W, dev):
    """depths[i] for i in chunk at the GT size [H,W], as one device tensor [len(chunk),H,W]: float32 when every plane
    is float32, float64 otherwise (the quantisation runs in the plane's own float type, edge.py:85-87).  Planes that
    ``_device_resizable`` takes are uploaded at their own size and resized on the device, one ``resize_linear`` per
    source shape; the others are resized with ``cv2.resize`` on the host (edge.py:76-78) as before."""
    import cv2
    host, on_dev = {}, {}
    for j, i in enumerate(chunk):
        d = np.asarray(depths[i])
        if _device_resizable(d, H, W):
            on_dev.setdefault(d.shape, []).append(j)
            continue
        if d.shape != (H, W):
            d = cv2.resize(d, (W, H), interpolation=cv2.INTER_LINEAR)
        host[j] = d if d.dtype == np.float32 else d.astype(np.float64)
    if not on_dev:
        return torch.from_numpy(np.stack([host[j] for j in range(len(chunk))])).to(dev, non_blocking=True)
    dtype = torch.float32 if all(d.dtype == np.float32 for d in host.values()) else torch.float64
    out = torch.empty((len(chunk), H, W), dtype=dtype, device=dev)
    if host:
        js = sorted(host)
        out[js] = torch.from_numpy(np.stack([host[j] for j in js])).to(dev, non_blocking=True).to(dtype)
    for js in on_dev.values():
        src = torch.from_numpy(np.stack([np.asarray(depths[chunk[j]]) for j in js])).to(dev, non_blocking=True)
        r = resize_linear(src, (H, W))
        if len(js) == len(chunk):
            return r if dtype == torch.float32 else r.to(dtype)
        out[js] = r.to(dtype)
    return out


def pr_evaluation_arrays(depths: Sequence[np.ndarray], gts: Sequence[np.ndarray], edge_thresh_range=None,
                         gt_crop=(44, 1197, 153, 371), min_depth=0.0, max_depth=80.0, batch: int = 32,
                         mask: Optional[np.ndarray] = None, per_image: bool = False):
    """Array-level ``pr_evaluation``: predicted depth maps (any size; resized to the GT size with cv2.INTER_LINEAR
    as edge.py:76-78 does -- on the device, bit-exact, for float32 maps of at least 2 x 2, with ``cv2.resize`` on the
    host for the others) and GT edge images (uint8, >127 = edge).
    Images are sharded over ``torch.distributed`` ranks when initialised.  ``mask`` is the mask-image branch of
    ``_pred_eval`` (eval_depth_edges.py:182-186, 198-200, 209-210): a float plane in [0,1] that multiplies both maps
    instead of the crop.
    -> (precision_vec, recall_vec, counts int64[T,4]; with a mask the sum_r column is returned separately as float64,
    see ``_masked_evaluation``).
    ``per_image`` appends the counts of every image, in list order: (..., rows int64[N,T,4], sum_r float64[N]).
    ``sum_r[i]`` is image i's ``sum_r`` as ``_pred_eval`` computes it: the GT pixels in the crop (``rows[i, :, 1]``),
    with a mask the fractional ``(gt * mask).sum()``.  Under ``torch.distributed`` every rank fills its own rows of
    zero arrays and ONE integer all-reduce sums them (exact: the result does not depend on the number of ranks);
    ``counts`` is then the sum of the rows."""
    if edge_thresh_range is None:
        edge_thresh_range = list(range(20, 241, 20))
    if mask is not None:
        return _masked_evaluation(depths, gts, edge_thresh_range, np.asarray(mask), min_depth, max_depth, batch,
                                  per_image)
    rank, world = _dist_info()
    dev = torch.device("cuda", torch.cuda.current_device())
    counts = torch.zeros((len(edge_thresh_range), 4), dtype=torch.int64, device=dev)
    rows = torch.zeros((len(depths), len(edge_thresh_range), 4), dtype=torch.int64, device=dev) if per_image else None
    mine = shard_indices(len(depths), rank, world)
    # group by GT shape, source shape (of the planes resized on the device) and depth dtype so every launch is a
    # dense batch; the quantisation runs in the array's own float type (edge.py:85-87), so float32 and float64 maps
    # must not be mixed
    by_shape = {}
    for i in mine:
        d = np.asarray(depths[i])
        dt = np.float32 if d.dtype == np.float32 else np.float64
        H, W = gts[i].shape[:2]
        src = d.shape if _device_resizable(d, H, W) else None
        by_shape.setdefault(((H, W), src, dt), []).append(i)
    for ((H, W), _src, dtype), idx in by_shape.items():
        for s in range(0, len(idx), batch):
            chunk = idx[s:s + batch]
            d_dev = _depth_planes(depths, chunk, H, W, dev)
            # _pred_eval: value/255 > 0.5 -> edge (eval_depth_edges.py:202-205)
            g_dev = torch.from_numpy(np.stack([(np.asarray(gts[i]) > 127).astype(np.uint8) for i in chunk])).to(
                dev, non_blocking=True)
            if per_image:
                rows[torch.tensor(chunk, device=dev)] = sweep_counts(d_dev, g_dev, edge_thresh_range, gt_crop,
                                                                     min_depth, max_depth, per_image=True)
            else:
                sweep_counts(d_dev, g_dev, edge_thresh_range, gt_crop, min_depth, max_depth, out=counts)
    if per_image:
        all_reduce_counts(rows)
        counts = rows.sum(0)
    else:
        all_reduce_counts(counts)
    c = counts.cpu().numpy().astype(np.float64)
    rec, prec, _ = compute_rec_prec_f1(c[:, 0], c[:, 1], c[:, 2], c[:, 3])
    if per_image:
        sum_r = rows[:, 0, 1].cpu().numpy().astype(np.float64)
        return [float(p) for p in prec], [float(r) for r in rec], counts, rows, sum_r
    return [float(p) for p in prec], [float(r) for r in rec], counts


def _masked_evaluation(depths, gts, edge_thresh_range, mask, min_depth, max_depth, batch, per_image=False):
    """``pr_evaluation`` with a mask image instead of a crop.  Per image and Canny setting the reference evaluates
    ``pred * mask`` (binarised again at ``>= 0.5`` by ``thresholds=1``) against ``gt * mask`` (boundary where non-zero)
    on the FULL plane, so: predicted pixel kept iff ``mask >= 0.5``, GT pixel kept iff ``mask != 0``, the matching
    radius is that of the uncropped plane, and ``sum_r`` is the fractional ``(gt * mask).sum()`` (float64, summed per
    image, then over images in list order -- eval_depth_edges.py:138, 299).  ``per_image`` as in
    ``pr_evaluation_arrays``, ``sum_r[i]`` being image i's ``(gt * mask).sum()``."""
    rank, world = _dist_info()
    dev = torch.device("cuda", torch.cuda.current_device())
    T = len(edge_thresh_range)
    counts = torch.zeros((T, 4), dtype=torch.int64, device=dev)
    keep_p = torch.from_numpy(np.ascontiguousarray(mask >= 0.5)).to(dev)
    keep_g = torch.from_numpy(np.ascontiguousarray(mask != 0)).to(dev)
    order = np.argsort(-np.asarray(edge_thresh_range), kind="stable")
    pairs = [(int(edge_thresh_range[i] / 2), int(edge_thresh_range[i])) for i in order]
    mine = shard_indices(len(depths), rank, world)
    sum_r = 0.0
    rows = torch.zeros((len(depths), T, 4), dtype=torch.int64, device=dev) if per_image else None
    sum_r_img = torch.zeros(len(depths), dtype=torch.float64, device=dev) if per_image else None
    H, W = mask.shape
    for s0 in range(0, len(mine), batch):
        chunk = mine[s0:s0 + batch]
        d_dev = _depth_planes(depths, chunk, H, W, dev)
        gb = [(np.asarray(gts[i]) > 127) for i in chunk]
        for i, g in zip(chunk, gb):
            s_i = (g.astype(np.float64) * mask).sum()
            sum_r = sum_r + s_i
            if per_image:
                sum_r_img[i] = s_i
        g_dev = torch.from_numpy(np.stack(gb)).to(dev)
        levels = canny_from_depth(d_dev, pairs, min_depth, max_depth, want_edges=False, want_levels=True)
        levels = torch.where(keep_p[None], levels, torch.full_like(levels, 255))
        c = pr_counts(levels, (g_dev & keep_g[None]).to(torch.uint8), n_levels=T, max_dist=0.002, crop=None,
                      per_image=per_image)
        idx = _reorder_index(tuple(int(v) for v in np.argsort(order)), c.device)
        if per_image:
            rows[torch.tensor(chunk, device=dev)] = c[:, idx]
        else:
            counts += c[idx]
    if per_image:
        all_reduce_counts(rows)
        counts = rows.sum(0)
        all_reduce_counts(sum_r_img)   # one writer per entry, all others add 0.0: exact
    else:
        all_reduce_counts(counts)
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([sum_r], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        sum_r = float(t.item())
    c = counts.cpu().numpy().astype(np.float64)
    rec, prec, _ = compute_rec_prec_f1(c[:, 0], np.full(T, sum_r), c[:, 2], c[:, 3])
    if per_image:
        return [float(p) for p in prec], [float(r) for r in rec], counts, rows, sum_r_img.cpu().numpy()
    return [float(p) for p in prec], [float(r) for r in rec], counts


def pr_evaluation(edge_list, pred_list, edge_thresh_range=None, gt_crop=[44, 1197, 153, 371], min_depth=0.0,
                  max_depth=80.0, save_folder="temp_output", num_workers=4, per_image=False):
    """Drop-in for eval_depth_edges.py:232-348 -> (precision_vec, recall_vec).
    ``save_folder`` and ``num_workers`` are accepted for signature compatibility; nothing is
    written to disk and no process pool is forked.
    ``per_image=True`` -> (precision_vec, recall_vec, results): ``results[i][k]`` is the ``EvalResult`` that
    ``_pred_eval`` gives for image i at Canny setting k (eval_depth_edges.py:296, before the sum at :298-301), from
    the same batched device calls."""
    import cv2
    depth_pred_list, edge_gt_list = list(pred_list), list(edge_list)
    if len(edge_gt_list) > len(depth_pred_list):  # multiscale GT list: keep the first entry of each group (:255-258)
        ratio = len(edge_gt_list) / len(depth_pred_list)
        edge_gt_list = edge_gt_list[0:len(edge_gt_list):int(ratio)]
    gts = [cv2.imread(p.split("\n")[0])[:, :, 0] for p in edge_gt_list]
    depths = [read_depth_file(p.split("\n")[0]) for p in depth_pred_list]
    # gt_crop is handed to _pred_eval as str(gt_crop) (:291-294): a path to an existing mask image selects the
    # mask branch
    crop, mask = _crop_or_mask(gt_crop if isinstance(gt_crop, str) else list(gt_crop))
    if not per_image:
        prec, rec, _ = pr_evaluation_arrays(depths, gts, edge_thresh_range, crop, min_depth, max_depth, mask=mask)
        return prec, rec
    prec, rec, _, rows, sum_r = pr_evaluation_arrays(depths, gts, edge_thresh_range, crop, min_depth, max_depth,
                                                     mask=mask, per_image=True)
    rows = rows.cpu().numpy().astype(np.float64)
    # _pred_eval evaluates one binarised edge image (thresholds=1): [1]-vectors, used threshold 0.5
    results = [[_eval_result(r[0:1], np.array([s]), r[2:3], r[3:4], _threshold_grid(1)) for r in img_rows]
               for img_rows, s in zip(rows, sum_r)]
    return prec, rec, results
