"""Oracle for the in-training "light" edge metric (TEST INFRASTRUCTURE).

Restates ``chamfer_distance`` of packnet_code/packnet_sfm/utils/edge.py:20-62
(2-D inputs, no mask): Euclidean distance transform of the non-GT pixels, mean
distance at predicted pixels and the share of predicted pixels closer than
``edge_to_edge_thresh`` to a GT pixel.
"""
from __future__ import annotations

import numpy as np
from scipy import ndimage


def chamfer_distance(im_pred, im_gt, edge_to_edge_thresh=5):
    gt = (np.asarray(im_gt) / 255) > 0.5
    pred = (np.asarray(im_pred) / 255) > 0.5
    dist = ndimage.distance_transform_edt(~gt)
    n_pred = pred.sum()
    with np.errstate(invalid="ignore", divide="ignore"):
        c_dist = float((dist * pred).sum() / n_pred)
        close = int((dist[pred] < edge_to_edge_thresh).sum())
        percentage = float(close / n_pred)
    return c_dist, percentage, close, int(n_pred)


def compute_edge_metrics(depth, gt_edge01, gt_crop=None, edge_model=False):
    """Restates ModelWrapper.compute_edge_metrics (packnet_code/packnet_sfm/models/model_wrapper.py:376-442) for
    a depth-predicting model: depth [H,W] float32 already at the GT size, gt_edge01 [H,W] in [0,1].

    edge_model: depth is the predicted edge probability map, binarised as ``depth > t`` for t = 0.5, 0.75, 0.9 in
    its own dtype.  This branch follows the documented rule only; unlike the depth branch it is not pinned to a
    golden of the reference."""
    gt_edge = np.asarray(gt_edge01) * 255
    depth = np.asarray(depth)
    if edge_model:
        ims = [(depth > t).astype(np.uint8) * 255 for t in (0.5, 0.75, 0.9)]
    else:
        import cv2
        vis = (depth * (255.0 / np.max(depth))).astype(np.uint8)
        ims = [cv2.Canny(vis, 10, 20), cv2.Canny(vis, 20, 40), cv2.Canny(vis, 30, 60)]
    if gt_crop is not None and len(gt_crop) > 0:
        c = gt_crop
        gt_edge = gt_edge[c[2]:c[3], c[0]:c[1]]
        ims = [im[c[2]:c[3], c[0]:c[1]] for im in ims]
    out = []
    with np.errstate(invalid="ignore", divide="ignore"):
        for im in ims:
            _, p1, _, _ = chamfer_distance(im, gt_edge)
            _, p2, _, _ = chamfer_distance(gt_edge, im)
            out += [p1, p2, 2 * ((p1 * p2) / (p1 + p2))]
    return out
