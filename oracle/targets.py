"""Oracle for the on-device target preparation (TEST INFRASTRUCTURE).

Restates, in NumPy, the dataloader steps of the reference that ``mindtheedge_b200.targets`` replaces:
``resize_depth_preserve`` (packnet_code/packnet_sfm/datasets/augmentations.py:58-100), the ``/255 if max > 1`` rule of
``resize_sample`` (:193-199), the normal decode of ``datasets/gta_dataset.py:413`` and the float32 cast of
``to_tensor_sample`` (:226-251)."""
from __future__ import annotations

import numpy as np


def resize_depth_preserve(depth, shape):
    """Every valid (> 0) source pixel is dropped onto (int(y * H/h), int(x * W/w)); when several land on the same
    output pixel the one that comes last in raster order stays (NumPy's repeated-index assignment)."""
    d = np.asarray(depth)
    if d.ndim > 2:          # [h,w,1] as the reference holds it; a 2-D map keeps its 1-pixel axes
        d = np.squeeze(d)
    h, w = d.shape
    ys, xs = np.nonzero(d > 0)  # raster order
    Y = (ys * (shape[0] / h)).astype(np.int32)
    X = (xs * (shape[1] / w)).astype(np.int32)
    keep = (Y < shape[0]) & (X < shape[1])
    out = np.zeros(shape)
    out[Y[keep], X[keep]] = d[ys[keep], xs[keep]]
    return out


def edge_target(edge_u8, shape):
    e = resize_depth_preserve(edge_u8, shape)
    if np.max(e) > 1:
        e = e / 255
    return e.astype(np.float32)


def decode_normals(normal_u8):
    return ((360. * (normal_u8 / 255.) - 180) * (np.pi / 180)).astype(np.float32)
