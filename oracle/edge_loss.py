"""Oracle for the training edge loss (TEST INFRASTRUCTURE, see oracle/__init__.py).

Restates ``packnet_code/packnet_sfm/losses/grad_loss.py``:

* directional 3x3 responses and the per-pixel pick by the quantised normal
  angle                                     -> grad_loss.py:20-31, 65-95
* resize, sigmoid(g - T), weight * loss     -> grad_loss.py:122-159
* class-balanced soft-label BCE + mask rule -> grad_loss.py:161-219

Two independent restatements are kept so they can check each other:

``edge_loss_torch``  fp32 torch-CPU ops + autograd (same op family and dtype as
                     the reference, so it is also the timed CPU baseline);
``edge_loss_np64``   fp64 NumPy with the analytic backward of SURVEY.md A.1.

Pinned against golden vectors produced by the reference ``GradLoss`` itself
(tests/golden/make_golden.py -> tests/golden/edge_loss_*.npz).
"""
from __future__ import annotations

import math

import numpy as np
import torch
import torch.nn.functional as F

# grad_loss.py:20-31 -- the four cross-correlation stencils, indexed v,h,lr,rl.
STENCILS = np.array(
    [
        [[-1, -2, -1], [0, 0, 0], [1, 2, 1]],      # v
        [[-1, 0, 1], [-2, 0, 2], [-1, 0, 1]],      # h
        [[-2, -1, 0], [-1, 0, 1], [0, 1, 2]],      # lr
        [[0, 1, 2], [-1, 0, 1], [-2, -1, 0]],      # rl
    ],
    dtype=np.float64,
)
DIR_V, DIR_H, DIR_LR, DIR_RL = 0, 1, 2, 3
EPS = 1e-3  # grad_loss.py:167,180


def direction_index(theta: np.ndarray) -> np.ndarray:
    """Quantise the normal angle to one of the four stencils.

    grad_loss.py:80-93.  The reference compares an fp32 tensor with Python
    floats, which torch rounds to fp32 first, so the band limits are the
    fp32-rounded k*pi/8.  Anything outside the three bands (incl. NaN) keeps the
    horizontal response.
    """
    t = np.asarray(theta, dtype=np.float32)
    b = [np.float32(k * np.pi / 8) for k in range(9)]
    d = np.full(t.shape, DIR_H, dtype=np.int8)
    band_v = ((t >= -b[5]) & (t < -b[3])) | ((t >= b[3]) & (t < b[5]))
    band_rl = ((t >= -b[7]) & (t < -b[5])) | ((t >= b[1]) & (t < b[3]))
    band_lr = ((t >= -b[3]) & (t < -b[1])) | ((t >= b[5]) & (t < b[7]))
    d[band_v] = DIR_V
    d[band_rl] = DIR_RL
    d[band_lr] = DIR_LR
    return d


def _stencil_bank(dtype=torch.float32, device="cpu") -> torch.Tensor:
    return torch.tensor(STENCILS, dtype=dtype, device=device).unsqueeze(1)  # [4,1,3,3]


def direction_index_torch(theta: torch.Tensor) -> torch.Tensor:
    """Same quantisation as ``direction_index`` with torch ops on theta's device."""
    t = theta.float()
    b = [float(np.float32(k * np.pi / 8)) for k in range(9)]
    d = torch.full_like(t, DIR_H, dtype=torch.long)
    band_v = ((t >= -b[5]) & (t < -b[3])) | ((t >= b[3]) & (t < b[5]))
    band_rl = ((t >= -b[7]) & (t < -b[5])) | ((t >= b[1]) & (t < b[3]))
    band_lr = ((t >= -b[3]) & (t < -b[1])) | ((t >= b[5]) & (t < b[7]))
    d[band_v] = DIR_V
    d[band_rl] = DIR_RL
    d[band_lr] = DIR_LR
    return d


def attention_loss2(output, target, mask=None, is_spatially_adaptive=False):
    """losses/attention_loss.py:21-49."""
    eps = 1e-14
    if not is_spatially_adaptive:
        num_pos = torch.sum(target == 1).float()
        num_neg = torch.sum(target == 0).float()
        alpha = num_neg / (num_pos + num_neg)
    else:
        box = torch.ones(1, 1, 15, 15, dtype=target.dtype, device=target.device)
        pos = F.conv2d(target, box, padding=7) / 225
        alpha = 1 - pos
        alpha = torch.where(alpha >= (1.0 - eps), torch.full_like(alpha, 0.5), alpha)
    p_clip = torch.clamp(output, min=eps, max=1.0 - eps)
    w = target * alpha * (4 ** ((1.0 - p_clip) ** 0.5)) + (1.0 - target) * (1.0 - alpha) * (4 ** (p_clip ** 0.5))
    w = w.detach()
    if mask is not None:
        w = w * mask
    return torch.mean(F.binary_cross_entropy(output, target, w, reduction="none"))


def edge_loss_torch(
    output: torch.Tensor,
    gt_edge: torch.Tensor,
    gt_mask: torch.Tensor | None = None,
    is_grad: bool = True,
    is_sigmoid: bool = True,
    sigmoid_thresh: float = 4,
    gt_normals: torch.Tensor | None = None,
    *,
    weight: float = 1.0,
    pos_to_neg: float = 1.0,
    edge_loss_type: str = "cross_entropy",
):
    """``GradLoss(edge_loss_type).forward`` on CPU (or any device) tensors -> (loss, grad_map).

    ``output`` may require grad; ``loss.backward()`` then gives the reference
    gradient through plain autograd.  Besides ``cross_entropy`` the type string may
    name ``attention_loss`` / ``spatially_adaptive`` (losses/attention_loss.py:21-49)
    and ``dice`` (grad_loss.py:150-156), combined as the reference's chain of ``if``s does.
    """
    H, W = gt_edge.shape[-2:]
    x = F.interpolate(output, size=(H, W), mode="bilinear")  # grad_loss.py:127
    if is_grad:
        resp = F.conv2d(x, _stencil_bank(x.dtype, x.device), padding=1)  # [B,4,H,W]
        if gt_normals is None:
            g = torch.sqrt(resp[:, 0:1] ** 2 + resp[:, 1:2] ** 2 + 1e-6)  # :73
        else:
            d = direction_index_torch(gt_normals.detach())
            g = torch.gather(resp, 1, d).abs()
    else:
        g = x
    p = torch.sigmoid(g - sigmoid_thresh) if is_sigmoid else g

    e = gt_edge
    if edge_loss_type != "cross_entropy":
        base = None
        if "cross_entropy" in edge_loss_type:
            base = edge_loss_torch(output, gt_edge, gt_mask, is_grad, is_sigmoid, sigmoid_thresh, gt_normals,
                                   weight=1.0, pos_to_neg=pos_to_neg)[0]
        if "attention_loss" in edge_loss_type:
            base = attention_loss2(p, e, gt_mask, False)
        if "spatially_adaptive" in edge_loss_type:
            base = attention_loss2(p, e, gt_mask, True)
        if "dice" in edge_loss_type:  # grad_loss.py:150-156
            base = base + 1000 * ((torch.sum(p ** 2) + torch.sum(e ** 2) + 0.0001) /
                                  (2 * torch.sum(p * e) + 0.0001)) / e.numel()
        return weight * base.mean(), g.detach()
    m = torch.ones_like(e) if gt_mask is None else gt_mask
    pos = -e * torch.log(p + EPS)
    neg = -(1 - e) * torch.log(1 - p + EPS)
    w_pos = (e * m).sum(dim=(1, 2, 3))
    w_neg = ((1 - e) * m).sum(dim=(1, 2, 3))
    if w_neg.sum() == 0:
        alpha = torch.ones_like(w_neg)
    else:
        alpha = w_neg / (w_pos + w_neg)
    vals = set(torch.unique(m).tolist())
    if vals == {0.0, 1.0}:  # grad_loss.py:183-187
        keep = (m != 0).to(e.dtype)
        pos = torch.where(m == 0, torch.zeros_like(pos), pos)
        neg = torch.where(m == 0, torch.zeros_like(neg), neg)
        valid = keep.sum()
    else:
        valid = float(e.numel())
    per_image = pos_to_neg * alpha * pos.sum(dim=(1, 2, 3)) + (1 - alpha) * neg.sum(dim=(1, 2, 3))
    loss = weight * (per_image.sum() / valid)
    return loss, g.detach()


# ---------------------------------------------------------------------------
# fp64 NumPy restatement with the analytic backward (SURVEY.md A.1)
# ---------------------------------------------------------------------------

def _pad1(x):
    return np.pad(x, ((0, 0), (1, 1), (1, 1)))


def responses_np(x: np.ndarray) -> np.ndarray:
    """All four zero-padded cross-correlations.  x: [B,H,W] -> [4,B,H,W]."""
    xp = _pad1(x.astype(np.float64))
    B, H, W = x.shape
    out = np.zeros((4, B, H, W))
    for d in range(4):
        for a in range(3):
            for b in range(3):
                k = STENCILS[d, a, b]
                if k:
                    out[d] += k * xp[:, a:a + H, b:b + W]
    return out


def bilinear_matrix(n_in: int, n_out: int) -> np.ndarray:
    """1-D weights of F.interpolate(mode='bilinear', align_corners=False).

    The reference computes the source coordinate in fp32 (area_pixel_compute_scale / _source_index with the float
    opmath type): scale = float(n_in) / float(n_out), src = scale * (o + 0.5) - 0.5 rounded once
    (torch's CPU kernel agrees with that to 1e-7 where two roundings are 1e-5 off).  For a
    scale that is not dyadic (1242 -> 1280) that coordinate is off the exact one by up to ~1e-4 px, which moves the
    interpolated value by up to 7e-5 of the depth range, so the weights are built from the same fp32 coordinate (the
    interpolation itself stays fp64).  For dyadic scales the coordinate is exact either way."""
    M = np.zeros((n_out, n_in))
    scale = np.float32(n_in) / np.float32(n_out)
    for o in range(n_out):
        src = float(np.float32(float(scale) * (o + 0.5) - 0.5))   # fp64 product + sum is exact: one fp32 rounding
        src = max(src, 0.0)
        i0 = min(int(math.floor(src)), n_in - 1)
        i1 = min(i0 + 1, n_in - 1)
        f = src - i0
        M[o, i0] += 1 - f
        M[o, i1] += f
    return M


def edge_loss_np64(
    output, gt_edge, gt_mask=None, is_grad=True, is_sigmoid=True, sigmoid_thresh=4.0,
    gt_normals=None, *, weight=1.0, pos_to_neg=1.0, upstream=1.0,
):
    """fp64 loss, grad map and d loss / d output.  Arrays are [B,1,h,w]."""
    out = np.asarray(output, dtype=np.float64)[:, 0]
    e = np.asarray(gt_edge, dtype=np.float64)[:, 0]
    B, H, W = e.shape
    h, w = out.shape[1:]
    same = (h, w) == (H, W)
    if same:
        x = out
    else:
        Mr, Mc = bilinear_matrix(h, H), bilinear_matrix(w, W)
        x = Mr @ out @ Mc.T          # matmul: a plain 3-operand einsum contracts in one O(h*w*H*W) loop
    m = np.ones_like(e) if gt_mask is None else np.asarray(gt_mask, dtype=np.float64)[:, 0]

    if is_grad:
        r = responses_np(x)
        if gt_normals is None:
            g = np.sqrt(r[0] ** 2 + r[1] ** 2 + 1e-6)
            d = None
        else:
            d = direction_index(np.asarray(gt_normals)[:, 0])
            c = np.take_along_axis(r, d[None].astype(np.int64), axis=0)[0]
            g = np.abs(c)
    else:
        g = x
    p = 1.0 / (1.0 + np.exp(sigmoid_thresh - g)) if is_sigmoid else g

    w_pos = (e * m).sum(axis=(1, 2))
    w_neg = ((1 - e) * m).sum(axis=(1, 2))
    with np.errstate(invalid="ignore", divide="ignore"):
        alpha = np.ones_like(w_neg) if w_neg.sum() == 0 else w_neg / (w_pos + w_neg)
    vals = set(np.unique(m).tolist())
    if vals == {0.0, 1.0}:
        Mk = (m != 0).astype(np.float64)
        valid = Mk.sum()
    else:
        Mk = np.ones_like(m)
        valid = float(e.size)
    sp = (Mk * e * np.log(p + EPS)).sum(axis=(1, 2))
    sn = (Mk * (1 - e) * np.log(1 - p + EPS)).sum(axis=(1, 2))
    loss = weight / valid * np.sum(-pos_to_neg * alpha * sp - (1 - alpha) * sn)

    a = alpha[:, None, None]
    dl_dp = upstream * weight / valid * Mk * (
        -pos_to_neg * a * e / (p + EPS) + (1 - a) * (1 - e) / (1 - p + EPS))
    dl_dg = dl_dp * p * (1 - p) if is_sigmoid else dl_dp
    if is_grad:
        if d is None:
            coeff = [dl_dg * r[0] / g, dl_dg * r[1] / g, 0 * g, 0 * g]
        else:
            s = dl_dg * np.sign(c)
            coeff = [np.where(d == k, s, 0.0) for k in range(4)]
        dx = np.zeros_like(x)
        for k in range(4):
            sp_ = _pad1(coeff[k])
            for a_ in range(3):
                for b_ in range(3):
                    kv = STENCILS[k, a_, b_]
                    if kv:
                        # x[i+a-1, j+b-1] feeds c[i,j]  =>  dx[m] += K[a,b]*s[m-(a-1,b-1)]
                        dx += kv * sp_[:, 2 - a_:2 - a_ + H, 2 - b_:2 - b_ + W]
    else:
        dx = dl_dg
    if not same:
        dx = Mr.T @ dx @ Mc
    return loss, g[:, None], dx[:, None]
