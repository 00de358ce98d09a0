"""Every two-kernel edge-loss path against the oracle, at shapes that cross strip seams and row blocks.

The shipped configuration (directional normals, sigmoid, no mask, prediction at target size) runs the one-pass
kernel and is covered by test_edge_loss_gpu.py.  This file reaches, through shapes, alignment and arguments only,
what the planner (make_plan / mte_edge_loss_bwd in csrc/edge_loss.cu) selects for everything else:

  forward   edge_loss_fwd_kernel<VEC, NONE|MAG|DIR, MASK, INV, SIG>
  backward  pointwise (is_grad=0), edge_loss_bwd_kernel<VEC, MAG|DIR, ...> (non-stash: magnitude mode, or any scale
            resized), edge_loss_bwd_stash_kernel<1, ...> and edge_loss_bwd_ring_kernel<...> (directional, same size)
  resize    resize_fwd_kernel / resize_bwd_kernel (prediction size != target size)
  alt       mte_edge_loss_alt_* (attention / spatially adaptive / dice)

Reference and tolerance (BASELINE.json north star, RTOL = 1e-5): the loss within 1e-5 relative of the fp64 oracle
(edge_loss_np64), the grad map within 1e-5 of its max, d loss / d pred within 1e-5 of its max of the fp32 torch
oracle (autograd).  The inputs keep both fp32 implementations on the same bits, so no pixel needs an exemption:
  * depths are powers of two (plus a flat block per image): every 3x3 response is exact in fp32 whatever the summation order,
    so sign(c) never depends on it, and 1/(1/d) == d exactly for the fused inv2depth;
  * power-of-two resize ratios have dyadic bilinear weights (multiples of 1/8 for x4), so the resized depth stays exact too
    (non-integer ratios run the magnitude and map modes, which have no sign);
  * the depth range is tied to sigmoid_thresh so that p = sigmoid(g - T) stays below ~0.995: where the sigmoid
    saturates, one ulp of p moves (1-p)/(1-p+eps) by more than 1e-5 of the gradient's max (the fp32 artefact
    test_edge_loss_gpu._check_gradient has to classify); and without the sigmoid |c| < 1, as the reference's
    log(1 - p + eps) requires (one case checks the NaN it returns otherwise).

test_coverage_manifest (CPU only) restates the planner for every case below and checks that each reachable kernel
instantiation runs at least once with two or more strips, two or more row blocks and a partial last strip.
"""
import math
import zlib

import numpy as np
import pytest
import torch

RTOL = 1e-5

DIR, MAG, NONE = "dir", "mag", "none"

# ---- the planner, restated (csrc/edge_loss.cu make_plan, csrc/edge_loss_kernels.cuh) -------------------------------
# K_FWD_RH: row height of the forward's shape-spread criterion (the forward itself plans strip rows, not row blocks);
# K_BWD_RH: kBwdRH, the row height of a work item of the non-ring backward kernels
K_FWD_RH, K_BWD_RH = 6, 8
K_HALO_LANES = 30                       # writing lanes of an overlapped forward / stash strip


def _bwd_lanes(vec):                    # bwd_lanes(): the non-stash backward needs two halo lanes per side at VEC=1
    return 32 - 2 * (2 if vec == 1 else 1)


def plan(case):
    """What make_plan / mte_edge_loss_bwd / the Python layer choose for a case: VEC, forward mode, backward family and
    per scale (resized, strips, row blocks, partial last strip) of the forward and of the backward."""
    mode, masked, inv, sig = case["mode"], case["mask"] != "none", case["inv"], case["sig"]
    scales = case["scales"]
    resized = [(h, w) != (H, W) for (_B, h, w, H, W) in scales]
    # VEC=4 needs W % 4 == 0 and 16-byte aligned planes; a misaligned (offset) view sends the call to VEC=1
    vec = 1 if case["offset"] or any(W % 4 for (*_, W) in scales) else 4
    fused = mode == DIR and not masked and not any(resized) and vec == 4 and all(W >= 4 for (*_, W) in scales)
    if mode == NONE:
        bwd = "pointwise"
    elif fused:
        bwd = "fused"
    elif mode == DIR and not any(resized):
        bwd = "ring_v4" if vec == 4 else "stash_v1"
    else:
        bwd = "nonstash"
    fwd_lanes = 32 if mode == NONE else K_HALO_LANES
    bwd_lanes = {"nonstash": _bwd_lanes(vec), "stash_v1": K_HALO_LANES, "ring_v4": K_HALO_LANES}.get(bwd)
    out = dict(vec=vec, mode=mode, mask=masked, inv=inv, sig=sig, bwd=bwd, resized=any(resized), scales=[])
    for (_B, _h, _w, H, W) in scales:
        s = dict(fwd_strips=math.ceil(W / (fwd_lanes * vec)), fwd_partial=W % (fwd_lanes * vec) != 0,
                 fwd_row_blocks=math.ceil(H / K_FWD_RH))
        if bwd_lanes:
            s.update(bwd_strips=math.ceil(W / (bwd_lanes * vec)), bwd_partial=W % (bwd_lanes * vec) != 0,
                     bwd_row_blocks=math.ceil(H / K_BWD_RH))
        out["scales"].append(s)
    return out


def _instantiations(p):
    """Kernel template instantiations a planned case launches (mask kind kept: binary / soft are runtime branches of
    the same instantiation that both need to be reached)."""
    if p["bwd"] == "fused":
        return []       # the one-pass kernel (edge_loss_fused.cu) replaces both
    return [("fwd", p["vec"], p["mode"], p["mask_kind"], p["inv"], p["sig"]),
            ("bwd", p["bwd"], p["vec"] if p["bwd"] != "pointwise" else None, p["mode"], p["mask_kind"], p["inv"],
             p["sig"])]


# ---- the configuration matrix -------------------------------------------------------------------------------------
PARAMS = [  # (sigmoid_thresh, weight, pos_to_neg), rotated through the matrix
    (4.0, 1.0, 1.0), (2.5, 10.0, 1.0), (6.0, 1.0, 0.35), (4.0, 3.0, 2.0)]


def _matrix():
    cases = []
    k = 0
    for mode in (DIR, MAG, NONE):
        for mask in ("none", "binary", "soft"):
            for inv in (False, True):
                for sig in (True, False):
                    for vec in (4, 1):
                        for route in ("same", "resize"):
                            if route == "resize" and (mode != DIR or inv):
                                continue   # inv2depth with a resize is refused (MTE_ERR_ARG); see test_inverse_...
                            if route == "same" and mode == DIR and mask == "none" and vec == 4:
                                continue   # the one-pass kernel (test_edge_loss_gpu.py)
                            # VEC=1 through a ragged width (sigmoid cases) or, at W % 4 == 0, through a view whose
                            # storage offset is not 16-byte aligned (the others)
                            offset = vec == 1 and not sig
                            W = 121 if (vec == 1 and not offset) else 244
                            if route == "resize":
                                H, W = 38, (122 if W == 121 else W)
                                scales = [(2, H // 2, W // 2, H, W)]      # x2 upsample: exact bilinear weights
                            else:
                                scales = [(2, 37, W, 37, W)]
                            T, weight, p2n = PARAMS[k % len(PARAMS)]
                            k += 1
                            cases.append(dict(mode=mode, mask=mask, inv=inv, sig=sig, offset=offset, scales=scales,
                                              T=T, weight=weight, p2n=p2n))
    return cases


def _cid(c):
    (B, h, w, H, W), = c["scales"][:1]
    size = f"{B}x{h}x{w}" + (f"-{H}x{W}" if (h, w) != (H, W) else "")
    return (f"{c['mode']}-{c['mask']}-{'inv' if c['inv'] else 'depth'}-{'sig' if c['sig'] else 'nosig'}-"
            f"{'off' if c['offset'] else 'al'}-{size}" + (f"-x{len(c['scales'])}" if len(c["scales"]) > 1 else ""))


MATRIX = _matrix()

# ---- shapes around the structural limits, per kernel family -------------------------------------------------------
SHAPES = [
    (1, 1, 121), (2, 5, 29), (3, 19, 58), (1, 13, 63), (2, 8, 31), (1, 1, 1), (1, 2, 5), (4, 3, 2),  # VEC=1
    (2, 3, 132), (1, 1, 244), (3, 17, 124), (2, 9, 8), (1, 6, 4), (5, 23, 368),                    # VEC=4
]
FAMILIES = [  # (mode, mask, inv, sig, T, weight, p2n): one per backward family and forward mode
    (NONE, "soft", False, True, 2.5, 1.0, 1.0),
    (MAG, "binary", False, True, 4.0, 10.0, 0.5),
    (MAG, "none", True, False, 4.0, 1.0, 1.0),
    (DIR, "binary", True, True, 4.0, 10.0, 1.0),       # stash_v1 / ring_v4
    (DIR, "none", False, False, 4.0, 1.0, 1.0),        # stash_v1 at VEC=1, one-pass kernel at VEC=4 (not asserted)
]


def _shape_cases():
    cases = []
    for fam in FAMILIES:
        mode, mask, inv, sig, T, weight, p2n = fam
        for (B, H, W) in SHAPES:
            cases.append(dict(mode=mode, mask=mask, inv=inv, sig=sig, offset=False, scales=[(B, H, W, H, W)], T=T,
                              weight=weight, p2n=p2n))
        if not inv and mode != NONE:   # the non-stash backward at the same shapes (predictions downsampled by 2)
            for (B, H, W) in SHAPES:
                cases.append(dict(mode=mode, mask=mask, inv=inv, sig=sig, offset=False,
                                  scales=[(B, 2 * H, 2 * W, H, W)], T=T, weight=weight, p2n=p2n))
    # one KITTI-size case per mode (4 x 384 x 1280: many CTAs per image, the grid caps in make_plan)
    cases.append(dict(mode=DIR, mask="binary", inv=False, sig=True, offset=False, scales=[(4, 384, 1280, 384, 1280)],
                      T=4.0, weight=10.0, p2n=1.0))
    cases.append(dict(mode=MAG, mask="none", inv=False, sig=True, offset=False, scales=[(4, 384, 1280, 384, 1280)],
                      T=4.0, weight=10.0, p2n=1.0))
    cases.append(dict(mode=NONE, mask="soft", inv=True, sig=True, offset=False, scales=[(4, 384, 1280, 384, 1280)],
                      T=4.0, weight=1.0, p2n=1.0))
    # one 4-scale pyramid per mode; the directional one has scale 2 resized, which sends every scale to the non-stash
    # backward
    pyr = [(2, 96 >> s, 320 >> s, 96 >> s, 320 >> s) for s in range(4)]
    pyr_rs = list(pyr)
    pyr_rs[2] = (2, 12, 40, 24, 80)
    cases.append(dict(mode=DIR, mask="none", inv=False, sig=True, offset=False, scales=pyr_rs, T=4.0, weight=10.0,
                      p2n=1.0))
    cases.append(dict(mode=DIR, mask="soft", inv=True, sig=True, offset=False, scales=pyr, T=4.0, weight=10.0,
                      p2n=1.0))
    cases.append(dict(mode=MAG, mask="binary", inv=True, sig=False, offset=False, scales=pyr, T=4.0, weight=1.0,
                      p2n=1.0))
    cases.append(dict(mode=NONE, mask="binary", inv=False, sig=False, offset=True, scales=pyr, T=4.0, weight=1.0,
                      p2n=1.0))
    # all-zero / all-one masks: value set {0} or {1} is not binary, so the mask only enters alpha (all alpha = 1 when
    # it is all zero: no negatives anywhere)
    for mode in (MAG, NONE):
        for mk in ("zeros", "ones"):
            cases.append(dict(mode=mode, mask=mk, inv=False, sig=True, offset=False, scales=[(2, 37, 244, 37, 244)],
                              T=4.0, weight=2.0, p2n=0.7))
    return cases


SHAPE_CASES = _shape_cases()


# ---- inputs ---------------------------------------------------------------------------------------------------------
def _depth_exponents(mode, sig, T):
    """Range of the power-of-two depths: keeps p = sigmoid(g - T) out of saturation (g - T <= ~5), or |c| < 1 / the
    map in (0, 1) without the sigmoid.  A 3x3 response is at most 4 * max depth (6 * for the magnitude)."""
    if mode == NONE:
        return (-2, 2) if sig else (-8, -1)
    if not sig:
        return (-10, -3)                   # |c| <= 4 * 2^-3 * sqrt(2) < 0.71
    return (-6, int(math.floor(math.log2((T + 5) / 6))))


def _plane_inputs(c, B, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    lo, hi = _depth_exponents(c["mode"], c["sig"], c["T"])
    e = torch.randint(lo, hi + 1, (B, 1, H, W), generator=g)
    depth = torch.pow(2.0, e.double()).float()
    if H >= 4 and W >= 4:   # a flat block: responses exactly 0 (sign 0 passes no gradient)
        depth[:, :, H // 4:H // 2 + 1, W // 4:W // 2 + 1] = depth[:, :, H // 4:H // 4 + 1, W // 4:W // 4 + 1]
    u = torch.rand(B, 1, H, W, generator=g)
    edge = torch.where(u < 0.03, torch.ones_like(u),
                       (u < 0.15).float() * torch.rand(B, 1, H, W, generator=g).clamp(min=0.3))
    k = torch.randint(0, 256, (B, 1, H, W), generator=g).float()
    normal = ((360 * k / 255 - 180) * np.pi / 180).float()
    kind = c["mask"]
    mask = None
    if kind == "binary":
        mask = (torch.rand(B, 1, H, W, generator=g) < 0.7).float()
        mask.view(B, -1)[:, 0] = 1.0            # every image keeps pixels, and the value set is exactly {0, 1}
        mask.view(-1)[-1] = 0.0 if mask.numel() > 1 else 1.0
    elif kind == "soft":
        mask = torch.randint(0, 5, (B, 1, H, W), generator=g).float() / 4
        mask.view(B, -1)[:, 0] = 0.5             # some value outside {0, 1}
    elif kind == "zeros":
        mask = torch.zeros(B, 1, H, W)
    elif kind == "ones":
        mask = torch.ones(B, 1, H, W)
    return depth, edge, normal, mask


def _scale_inputs(c, seed):
    """Per scale: (prediction as given to the library [inverse depth with inv], depth at prediction size, edge, normal,
    mask) on the CPU."""
    out = []
    for i, (B, h, w, H, W) in enumerate(c["scales"]):
        depth, edge, normal, mask = _plane_inputs(c, B, H, W, seed + 17 * i)
        if (h, w) != (H, W):
            depth = _plane_inputs(c, B, h, w, seed + 17 * i + 5)[0]
        pred = 1.0 / depth if c["inv"] else depth
        out.append((pred, depth, edge, normal, mask))
    return out


def _cuda(t, offset):
    """To the device; with offset, as a contiguous view one float past a 16-byte boundary."""
    if t is None:
        return None
    if not offset:
        return t.cuda()
    buf = torch.empty(t.numel() + 1, device="cuda")
    v = buf[1:].view(t.shape)
    v.copy_(t)
    assert v.is_contiguous() and v.data_ptr() % 16 != 0
    return v


def _plane_close(got, ref, what, rtol=RTOL):
    scale = max(float(np.abs(ref).max()), 1e-30)
    err = float(np.abs(got.astype(np.float64) - ref).max())
    assert err <= rtol * scale, f"{what}: max abs err {err:.3e} vs scale {scale:.3e} ({err / scale:.2e} rel)"


def _references(c, inputs, upstream=None):
    """fp64 loss and grad maps (edge_loss_np64), fp32 autograd d objective / d pred (edge_loss_torch).  upstream:
    (a, [b_s]) for the objective a * total + sum_s b_s * per[s]; default total."""
    from oracle.edge_loss import edge_loss_np64, edge_loss_torch
    n = len(inputs)
    weights = c.get("scale_weights") or [1.0 / n] * n
    a, b = upstream or (1.0, [0.0] * n)
    common = dict(is_grad=c["mode"] != NONE, is_sigmoid=c["sig"], sigmoid_thresh=c["T"])
    loss64, maps64, per64, dx64 = 0.0, [], [], []
    obj, xs = 0.0, []
    for s, (pred, depth, edge, normal, mask) in enumerate(inputs):
        nrm = normal if c["mode"] == DIR else None
        l64, g64, d64 = edge_loss_np64(depth.numpy(), edge.numpy(), None if mask is None else mask.numpy(),
                                       common["is_grad"], c["sig"], c["T"], None if nrm is None else nrm.numpy(),
                                       weight=c["weight"], pos_to_neg=c["p2n"], upstream=a * weights[s] + b[s])
        loss64 += weights[s] * l64
        per64.append(l64)
        maps64.append(g64)
        dx64.append(None if c["inv"] else d64)      # d / d depth; with inv2depth the chain factor is not applied
        x = pred.clone().requires_grad_(True)
        d = 1.0 / x.clamp(min=1e-6) if c["inv"] else x
        l, _ = edge_loss_torch(d, edge, mask, common["is_grad"], c["sig"], c["T"], nrm, weight=c["weight"],
                               pos_to_neg=c["p2n"])
        obj = obj + (a * weights[s] + b[s]) * l
        xs.append(x)
    obj.backward()
    return loss64, per64, maps64, [x.grad.numpy() for x in xs], dx64


def _run(c, inputs, upstream=None):
    from mindtheedge_b200.losses import multiscale_edge_loss
    n = len(inputs)
    off = c["offset"]
    xs = [_cuda(p, off).requires_grad_(True) for (p, *_r) in inputs]
    edges = [_cuda(e, off) for (_p, _d, e, _n, _m) in inputs]
    normals = [_cuda(nm, off) for (*_r, nm, _m) in inputs] if c["mode"] == DIR else None
    masks = [_cuda(m, off) for (*_r, m) in inputs] if c["mask"] != "none" else None
    total, per, maps = multiscale_edge_loss(xs, edges, masks, normals, scale_weights=c.get("scale_weights"),
                                            is_grad=c["mode"] != NONE, is_sigmoid=c["sig"], sigmoid_thresh=c["T"],
                                            weight=c["weight"], pos_to_neg=c["p2n"], pred_is_inverse=c["inv"])
    a, b = upstream or (1.0, [0.0] * n)
    obj = a * total
    for s in range(n):
        if b[s]:
            obj = obj + b[s] * per[s]
    obj.backward()
    return (total.item(), [v.item() for v in per], [m.cpu().numpy() for m in maps],
            [x.grad.cpu().numpy() for x in xs])


def _check(c, seed, upstream=None):
    inputs = _scale_inputs(c, seed)
    loss64, per64, maps64, grads_ref, dx64 = _references(c, inputs, upstream)
    total, per, maps, grads = _run(c, inputs, upstream)
    label = _cid(c)
    assert np.isfinite(loss64), label
    assert abs(total - loss64) <= RTOL * abs(loss64), (label, total, loss64)
    for s, (_B, h, w, H, W) in enumerate(c["scales"]):
        assert abs(per[s] - per64[s]) <= RTOL * abs(per64[s]), (label, s, per[s], per64[s])
        _plane_close(maps[s], maps64[s], f"{label} grad map {s}")
        if (h, w) == (H, W):
            _plane_close(grads[s], grads_ref[s], f"{label} d/dpred {s}")
        else:
            _check_resized_gradient(grads[s], grads_ref[s], dx64[s], f"{label} d/dpred {s}")


def _check_resized_gradient(got, ref, exact, label):
    """d loss / d pred through the resize adjoint: within 1e-5 of max of the fp64 oracle everywhere, and of the fp32
    torch oracle everywhere except where the torch oracle itself is off the fp64 adjoint by more than that -- its fp32
    scatter-add of a large upsampling (thousands of terms of both signs per source pixel) drifts there."""
    tol = RTOL * max(float(np.abs(ref).max()), 1e-30)
    got = got.astype(np.float64)
    err_exact = np.abs(got - exact)
    assert float(err_exact.max()) <= tol, f"{label}: vs fp64 adjoint {float(err_exact.max()) / tol:.2f} x tol"
    drift = np.abs(ref - exact) > tol
    unexplained = (np.abs(got - ref) > tol) & ~drift
    assert not unexplained.any(), f"{label}: {int(unexplained.sum())} pixels off the torch oracle, which is exact there"
    if drift.any():
        print(f"{label}: {int(drift.sum())} pixels where the torch oracle's fp32 scatter-add drifts "
              f"{float(np.abs(ref - exact).max()) / tol:.1f} x tol from the fp64 adjoint")


@pytest.mark.gpu
@pytest.mark.parametrize("case", MATRIX, ids=_cid)
def test_configuration_matrix(case):
    _check(case, seed=zlib.crc32(_cid(case).encode()) % 10007)


@pytest.mark.gpu
@pytest.mark.parametrize("case", SHAPE_CASES, ids=lambda c: _cid(c) + (f"-{c['mask']}" if c["mask"] in ("zeros", "ones") else ""))
def test_shapes(case):
    _check(case, seed=sum(x for s in case["scales"] for x in s))


# ---- resize ratios ------------------------------------------------------------------------------------------------
RESIZE = [  # (B, h, w, H, W, mode): power-of-two ratios run the directional mode (exact), the others magnitude / map
    (2, 24, 32, 48, 64, DIR), (1, 12, 30, 48, 120, DIR), (2, 96, 128, 48, 64, DIR), (1, 192, 244, 48, 61, DIR),
    (1, 375, 1242, 384, 1280, MAG), (1, 375, 1242, 384, 1280, NONE), (2, 60, 100, 48, 64, MAG),
    (2, 60, 100, 48, 64, NONE), (1, 1, 50, 96, 100, MAG), (1, 2, 3, 96, 120, MAG), (2, 48, 1, 96, 128, NONE),
    (1, 2, 2, 128, 64, DIR), (1, 1, 1, 96, 97, NONE),
]


def _pow2_ratio(a, b):
    """a -> b by a power-of-two factor: the bilinear weights are dyadic and the resized depth exact in fp32."""
    lo, hi = min(a, b), max(a, b)
    return hi % lo == 0 and (hi // lo) & (hi // lo - 1) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("r", RESIZE, ids=lambda r: f"{r[5]}-{r[0]}x{r[1]}x{r[2]}-{r[3]}x{r[4]}")
def test_resize(r):
    """resize_fwd_kernel and its gather adjoint resize_bwd_kernel (with its +-1 window slack) at up- and down-sampling
    ratios x2, x4, 1/2, 1/4, non-integer, and 1- or 2-pixel sources upsampled to >= 96: forward values, grad map and
    d loss / d pred after the adjoint."""
    B, h, w, H, W, mode = r
    assert mode != DIR or (_pow2_ratio(h, H) and _pow2_ratio(w, W))
    for mask in ("none", "binary"):
        c = dict(mode=mode, mask=mask, inv=False, sig=True, offset=False, scales=[(B, h, w, H, W)], T=4.0,
                 weight=10.0, p2n=1.0)
        _check(c, seed=h * w + H)


@pytest.mark.gpu
def test_inverse_with_resize_is_refused():
    """inv2depth fused after a resize would differ from the reference (it precedes the head), so the library refuses
    pred_is_inverse with any resized scale instead of computing something else."""
    from mindtheedge_b200 import _lib
    from mindtheedge_b200.losses import multiscale_edge_loss
    c = dict(mode=MAG, mask="none", inv=True, sig=True, offset=False, scales=[(1, 16, 32, 16, 32), (1, 8, 8, 16, 16)],
             T=4.0, weight=1.0, p2n=1.0)
    inputs = _scale_inputs(c, 3)
    xs = [p.cuda().requires_grad_(True) for (p, *_r) in inputs]
    with pytest.raises(_lib.MteError, match="code"):
        multiscale_edge_loss(xs, [e.cuda() for (_p, _d, e, _n, _m) in inputs], None, None, pred_is_inverse=True)


@pytest.mark.gpu
def test_nan_parity_without_sigmoid():
    """is_grad with is_sigmoid=0 takes |c| as a probability: where |c| > 1 the reference's log(1 - p + eps) is NaN, and
    so must the loss be."""
    from mindtheedge_b200.losses import edge_loss
    from oracle.edge_loss import edge_loss_np64, edge_loss_torch
    for mode in (DIR, MAG):
        c = dict(mode=mode, mask="none", inv=False, sig=True, offset=False, scales=[(2, 37, 121, 37, 121)], T=4.0,
                 weight=1.0, p2n=1.0)
        (pred, depth, edge, normal, _m), = _scale_inputs(c, 11)
        nrm = normal if mode == DIR else None
        with np.errstate(invalid="ignore"):
            l64 = edge_loss_np64(depth.numpy(), edge.numpy(), None, True, False, 4.0,
                                 None if nrm is None else nrm.numpy())[0]
        lt, _ = edge_loss_torch(depth, edge, None, True, False, 4.0, nrm)
        lg, _ = edge_loss(pred.cuda(), edge.cuda(), None, True, False, 4.0, None if nrm is None else nrm.cuda())
        assert np.isnan(l64) and torch.isnan(lt) and torch.isnan(lg), (mode, l64, lt.item(), lg.item())


# ---- upstream gradients on the two-kernel path ----------------------------------------------------------------------
UPSTREAM = [
    dict(mode=MAG, mask="soft", inv=False, sig=True, offset=False,
         scales=[(2, 96 >> s, 320 >> s, 96 >> s, 320 >> s) for s in range(4)], T=4.0, weight=10.0, p2n=1.0,
         scale_weights=[0.4, 0.3, 0.2, 0.1]),
    dict(mode=DIR, mask="binary", inv=True, sig=True, offset=False,
         scales=[(2, 96 >> s, 324 >> s, 96 >> s, 324 >> s) for s in range(4)], T=4.0, weight=10.0, p2n=1.0,
         scale_weights=[0.25, 0.25, 0.25, 0.25]),
    dict(mode=DIR, mask="none", inv=False, sig=True, offset=False,
         scales=[(2, 48, 160, 96, 320), (2, 48, 160, 48, 160), (2, 24, 80, 24, 80), (2, 12, 40, 12, 40)], T=4.0,
         weight=10.0, p2n=1.0, scale_weights=[0.5, 0.2, 0.2, 0.1]),
    dict(mode=NONE, mask="binary", inv=True, sig=False, offset=False,
         scales=[(2, 96 >> s, 320 >> s, 96 >> s, 320 >> s) for s in range(4)], T=4.0, weight=1.0, p2n=1.0,
         scale_weights=[0.4, 0.3, 0.2, 0.1]),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", UPSTREAM, ids=_cid)
def test_per_scale_upstream(case):
    """Backward of a * total + sum_s b_s * per[s] (a not in {0, 1}, some b_s negative, some zero): the two-kernel
    backward reads grad_loss[0] * scale_weight + grad_loss[1 + s] per scale."""
    _check(case, seed=91, upstream=(0.7, [1.5, 0.0, -0.8, 0.0]))


# ---- alternative loss types -----------------------------------------------------------------------------------------
ALT_TYPES = ["attention_loss", "spatially_adaptive", "spatially_adaptive_dice", "cross_entropy_dice"]
ALT = [  # (B, h, w, H, W, normals, mask, is_grad)
    (2, 37, 121, 37, 121, True, False, True),        # VEC=1 stash (ragged)
    (2, 96, 320, 96, 320, True, False, True),
    (1, 384, 1280, 384, 1280, True, False, True),
    (2, 33, 98, 33, 98, True, True, True),           # mask
    (2, 37, 121, 37, 121, False, False, True),       # magnitude mode
    (2, 37, 121, 37, 121, False, True, False),       # is_grad = 0 (the map is the probability)
    (2, 24, 60, 48, 120, True, False, True),         # prediction size != target size (x2)
]


@pytest.mark.gpu
@pytest.mark.parametrize("a", ALT, ids=lambda a: f"{a[0]}x{a[1]}x{a[2]}-{a[3]}x{a[4]}-{'n' if a[5] else 'mag'}"
                         f"{'-mask' if a[6] else ''}{'' if a[7] else '-map'}")
@pytest.mark.parametrize("ltype", ALT_TYPES)
def test_alt_loss_types(ltype, a):
    """GradLoss('attention_loss' / 'spatially_adaptive' / +dice / 'cross_entropy_dice') against edge_loss_torch: loss
    within 1e-5 relative, grad map and d loss / d pred within 1e-5 of their max."""
    from mindtheedge_b200.losses import GradLoss
    from oracle.edge_loss import edge_loss_torch
    B, h, w, H, W, with_normals, masked, is_grad = a
    c = dict(mode=(DIR if with_normals else MAG) if is_grad else NONE, mask="binary" if masked else "none", inv=False,
             sig=True, offset=False, scales=[(B, h, w, H, W)], T=4.0, weight=3.0, p2n=1.0)
    (pred, depth, edge, normal, mask), = _scale_inputs(c, B * H + W)
    nrm = normal if with_normals else None
    xr = depth.clone().requires_grad_(True)
    lr, gr = edge_loss_torch(xr, edge, mask, is_grad, True, 4.0, nrm, weight=3.0, edge_loss_type=ltype)
    lr.backward()
    xg = depth.cuda().requires_grad_(True)
    head = GradLoss(ltype, True, [], 3.0, 1.0)
    lg, gg = head(xg, edge.cuda(), None if mask is None else mask.cuda(), is_grad, True, 4.0,
                  None if nrm is None else nrm.cuda())
    lg.backward()
    assert abs(lg.item() - lr.item()) <= RTOL * abs(lr.item()), (lg.item(), lr.item())
    _plane_close(gg.cpu().numpy(), gr.numpy(), f"{ltype} grad map")
    _plane_close(xg.grad.cpu().numpy(), xr.grad.numpy(), f"{ltype} d/dpred")


# ---- coverage manifest (CPU) --------------------------------------------------------------------------------------
def _required():
    """Every instantiation the two-kernel path can reach: forward <VEC, mode, mask kind, INV, SIG> and its backward
    family, except the directional ones the one-pass kernel takes (no mask, VEC=4, same size), and the non-stash
    directional backward with INV (it needs a resized scale, and inv2depth with a resize is refused)."""
    req = set()
    for mode in (DIR, MAG, NONE):
        for mk in ("none", "binary", "soft"):
            for inv in (False, True):
                for sig in (True, False):
                    for vec in (4, 1):
                        routes = [False, True] if mode == DIR and not inv else [False]
                        for rs in routes:
                            W = 244 if vec == 4 else 121
                            scales = [(1, 8, W // 2, 16, W)] if rs else [(1, 16, W, 16, W)]
                            p = plan(dict(mode=mode, mask=mk, inv=inv, sig=sig, offset=False, scales=scales))
                            p["mask_kind"] = mk
                            for k in _instantiations(p):
                                req.add(k)
    return req


def test_coverage_manifest():
    """Each reachable kernel instantiation of the two-kernel path (and each mask kind of it) is run by at least one
    case above on a scale with >= 2 strips, >= 2 row blocks and a partial last strip, in the forward and in the
    backward.  The planner is restated in plan(); if make_plan changes, this is the test that names the cases to
    update."""
    cases = MATRIX + SHAPE_CASES + UPSTREAM
    covered = {}
    for c in cases:
        p = plan(c)
        p["mask_kind"] = c["mask"] if c["mask"] in ("none", "binary", "soft") else "soft"
        good = any(s["fwd_strips"] >= 2 and s["fwd_row_blocks"] >= 2 and s["fwd_partial"] and
                   ("bwd_strips" not in s or (s["bwd_strips"] >= 2 and s["bwd_row_blocks"] >= 2 and s["bwd_partial"]))
                   for s in p["scales"])
        for k in _instantiations(p):
            covered[k] = covered.get(k, False) or good
    req = _required()
    # forward: 2 VEC x 3 modes x 3 mask kinds x INV x SIG, less the two directional INV ones only the one-pass kernel
    # runs; backward: pointwise 12, non-stash magnitude 24 and directional 12 (no INV), stash_v1 12, ring_v4 8
    assert len(req) == 70 + 12 + 24 + 12 + 12 + 8, len(req)
    missing = sorted(str(k) for k in req if not covered.get(k))
    assert not missing, "instantiations without a multi-strip, multi-row-block, partial-strip case:\n" + "\n".join(missing)
    # VEC=1 is reached both through a ragged width and through a misaligned view at W % 4 == 0, for every mode
    for mode in (DIR, MAG, NONE):
        for how in ("ragged", "offset"):
            assert any(plan(c)["vec"] == 1 and c["mode"] == mode and
                       (c["offset"] if how == "offset" else any(s[-1] % 4 for s in c["scales"])) for c in MATRIX), \
                (mode, how)
    # non-default sigmoid_thresh, pos_to_neg and weight occur
    assert any(c["T"] != 4 for c in MATRIX) and any(c["p2n"] != 1 for c in MATRIX) and any(c["weight"] != 1 for c in MATRIX)
    # the shape families: H = 1, H below a row block, H not a multiple of either row height, W % 4 in {1, 2, 3},
    # widths just above one strip, B > 1 with several backward CTAs per image
    Ws = {s[-1] for c in SHAPE_CASES for s in c["scales"]}
    Hs = {s[-2] for c in SHAPE_CASES for s in c["scales"]}
    assert {W % 4 for W in Ws} >= {1, 2, 3} and 1 in Hs and any(h < K_FWD_RH for h in Hs)
    assert any(h % K_FWD_RH and h % K_BWD_RH for h in Hs)
    assert {121, 29, 132, 31} <= Ws
    several = [c for c in SHAPE_CASES + MATRIX for s, ps in zip(c["scales"], plan(c)["scales"])
               if s[0] > 1 and ps.get("bwd_strips", 0) * ps.get("bwd_row_blocks", 0) > 8]
    assert several
