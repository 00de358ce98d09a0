"""Every kernel path of the DEE post-process (``tools.dee_postprocess``) and of the level hysteresis it shares with the
Canny sweep, against the oracle, bit-exact.

``test_dee_gpu.py`` checks the default configuration (fp64 output, all three stages).  Here each path is reached only
through shapes, dtypes, alignment, flags and values, on the release library:

* front: ``dee_front_tma_kernel<NRM, NMS, HYST>`` (fp32, W % 4 == 0, H, W >= 4, 16-byte aligned base) and
  ``dee_front_kernel<float / double>`` (everything else; an fp32 plane at a TMA-eligible shape gets there through a
  view that starts one element into its buffer);
* hysteresis (``canny::run_level_hysteresis``, one pair for DEE): the shared-memory union-find with its bitmaps in
  shared memory, the same kernel with the bitmaps in global scratch ("BIG", planes too large for the opt-in shared
  memory), and the L2 kernel (W % 16 != 0, or more reachable candidates than the shared-memory kernel holds);
  the flood's changed-word worklist and its full-sweep mode once more than ``WORK_CAP`` words change;
* finish: ``dee_finish_kernel``'s float4 path (fp32 in and out, W % 4 == 0) and its scalar path, and the slicing of
  batches beyond 65,535 images.

The expected edges are the oracle's result in the dtype the reference computes in (float64 after the NMS, the input
dtype for the hysteresis of a raw map), cast once to ``out_dtype``; the u8 normals equal ``normals_u8``.
``test_path_manifest`` restates the host's planning rules and checks that every path above is taken by some case, with
each case clear of the size boundaries; it needs no GPU.
"""
import itertools

import numpy as np
import pytest
import torch

from synth import prob_map

# ---- the host's planning rules (dee.cu: run / make_plane_map / dee_finish_kernel; canny.cu: run_level_hysteresis) ----
OPTIN = 232448        # cudaDevAttrMaxSharedMemoryPerBlockOptin of a B200 (227 KB)
HYST_STATIC = 7456    # static shared memory of canny_uf_hyst_smem_kernel<false / true> (cuobjdump -res-usage, sm_100a)
WORK_CAP = 4096       # canny.cu kWorkCap: flood worklist entries before the full sweep
GRID_Y = 65535        # dee.cu: images per dee_finish_kernel launch (one per blockIdx.y)


def _a16(n):
    return (n + 15) // 16 * 16


def front_path(dtype, H, W, aligned=True):
    return "tma" if dtype == np.float32 and W % 4 == 0 and H >= 4 and W >= 4 and aligned else "generic"


def hyst_plan(H, W):
    """(kernel, candidate cap) of run_level_hysteresis: 'smem', 'big' or 'l2'."""
    budget = OPTIN - HYST_STATIC - 1024
    WPR = (W + 31) // 32
    nW = H * WPR
    if W % 16 or budget <= 0 or nW * 32 >= 1 << 31:
        return "l2", 0
    bitmapB, rankB = _a16(nW * 4), _a16((nW + 1) // 2 * 2)
    regionX = budget - (bitmapB + rankB + 2 * WORK_CAP * 2 + 64)
    cap = int(regionX * 8 / 41) - 64
    kernel = "smem"
    if not (regionX >= bitmapB and cap >= 8192 and nW < 65536):
        kernel = "big"
        regionX = budget - (2 * WORK_CAP * 4 + 64)
        cap = int(regionX * 8 / 41) - 64
    cap = min(cap, 65535) & ~31
    if kernel == "big":  # the parked neighbour ids must also fit behind the global bitmaps
        nid_off = (2 * nW * 4 + (nW + 1) // 2 * 2 + 15) & ~15
        cap = min(cap, (H * W * 4 - nid_off) // 16)
    return kernel, cap


def big_boundary(W):
    """Smallest H at which a plane of width W leaves shared memory (None: never / L2)."""
    if W % 16:
        return None
    H = 1
    while hyst_plan(H, W)[0] == "smem":
        H += 1
    return H


def finish_path(in_dtype, out_dtype, N, H, W):
    vec = in_dtype == np.float32 and out_dtype == np.float32 and (H * W) % 4 == 0 and W % 4 == 0
    return ("vector" if vec else "scalar"), -(-N // GRID_Y)


def seeded_words(strong):
    """Bitmap words (rows padded to whole 32-bit words) holding a strong pixel: the flood's first worklist."""
    H, W = strong.shape
    WPR = (W + 31) // 32
    pad = np.zeros((H, WPR * 32), bool)
    pad[:, :W] = strong
    return int(pad.reshape(H, WPR, 32).any(axis=2).sum())


def dee_strong(p, t_high):
    """The oracle's strong mask (oracle.dee.hysteresis): interior pixels above t_high, in the array's own dtype."""
    s = np.zeros(p.shape, bool)
    if p.shape[0] > 2 and p.shape[1] > 2:
        s[1:-1, 1:-1] = p[1:-1, 1:-1] > t_high
    return s


# ---- the reference rule, literally (tools.py:49-92) --------------------------------------------------------------
def hysteresis_loop(img, t_low=0.3, t_high=0.7):
    img = np.asarray(img)
    H, W = img.shape
    temp = np.copy(img)
    if H > 2 and W > 2:
        lab = {}
        for y in range(1, H - 1):
            for x in range(1, W - 1):
                v = img[y, x]
                lab[y, x] = 2 if v > t_high else (0 if v < t_low else 1)
        stack = [k for k, v in lab.items() if v == 2]
        while stack:
            y, x = stack.pop()
            for dy in (-1, 0, 1):
                for dx in (-1, 0, 1):
                    k = (y + dy, x + dx)
                    if lab.get(k) == 1:
                        lab[k] = 2
                        stack.append(k)
        for (y, x), v in lab.items():
            temp[y, x] = 2 if v == 2 else 0
    with np.errstate(invalid="ignore", divide="ignore"):
        temp = temp / np.max(temp)
        return img * temp


def _eq(a, b):
    return a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a, b, equal_nan=True)


def _pin_planes():
    r = np.random.default_rng(17)
    f32 = lambda t: float(np.float32(t))
    up = lambda t: float(np.nextafter(np.float32(t), np.float32(np.inf)))
    dn = lambda t: float(np.nextafter(np.float32(t), np.float32(-np.inf)))
    specials = [np.nan, np.inf, -np.inf, -0.0, 0.0, 0.3, 0.7, f32(0.3), f32(0.7), up(0.3), dn(0.3), up(0.7), dn(0.7),
                0.5, 0.1, 0.9]
    planes = []
    for k in range(10):
        H, W = int(r.integers(3, 9)), int(r.integers(3, 9))
        p = r.choice(specials + list(r.uniform(0, 1, 8)), size=(H, W))
        planes.append(p)
    p = r.uniform(0, 1, (6, 7)); p[0, 3] = np.nan; planes.append(p)                       # NaN border
    p = r.uniform(0, 1, (6, 7)); p[5, 0] = np.inf; planes.append(p)                       # +Inf border
    p = r.uniform(0, 1, (6, 7)); p[2, 6] = -np.inf; p[1:-1, 1:-1] *= 0.5; planes.append(p)  # no strong, -Inf border
    planes.append(np.zeros((5, 5)))
    p = np.full((6, 6), 0.5); p[2, 2] = np.nan; p[3, 4] = 0.9; p[:, 0] = -2.0; planes.append(p)  # NaN bridge
    for shape in [(1, 1), (1, 5), (5, 1), (2, 2), (2, 6), (6, 2)]:
        p = r.uniform(-1, 1, shape); p.flat[0] = -3.0; planes.append(p)
    planes.append(-r.uniform(0.1, 1, (2, 4)))
    return planes


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_oracle_hysteresis_matches_reference_rule(dtype):
    """CPU: oracle.dee.hysteresis (ndimage.label) against the reference rule written as a loop, on planes carrying
    NaN, +-Inf, -0.0, values at and next to both thresholds, NaN / Inf borders, an all-zero plane, H or W <= 2 and
    t_low > t_high; against the unmodified tools.py too when the reference is staged."""
    from oracle import dee as odee
    from oracle import ref_loader
    ref = ref_loader.load_tools() if ref_loader.available() else None
    pairs = [(0.3, 0.7), (0.7, 0.3), (0.5, 0.5), (0.1, 0.3)]
    for k, p in enumerate(_pin_planes()):
        p = p.astype(dtype)
        for tl, th in pairs:
            exp = hysteresis_loop(p, tl, th)
            with np.errstate(all="ignore"):
                got = odee.hysteresis(p, tl, th)
                assert _eq(got, exp), (k, tl, th, p, got, exp)
                if ref is not None:
                    assert _eq(ref.hysteresis(np.copy(p), tl, th), exp), (k, tl, th)


# ---- running the library ------------------------------------------------------------------------------------------
FLAGS = [f for f in itertools.product((True, False), repeat=3) if any(f)]   # (normals, nms, hysteresis): 7


def _flag_id(f):
    return "-".join(n for n, on in zip(("nrm", "nms", "hyst"), f) if on)


def _to_device(probs, aligned):
    t = torch.from_numpy(np.ascontiguousarray(probs))
    if aligned:
        return t.cuda()
    buf = torch.zeros(probs.size + 1, dtype=t.dtype, device="cuda")
    buf[1:].copy_(t.reshape(-1))
    return buf[1:1 + probs.size].view(probs.shape)


def run_dee(probs, flags=(True, True, True), out=np.float32, aligned=True, tl=0.3, th=0.7):
    from mindtheedge_b200.tools import dee_postprocess
    x = _to_device(probs, aligned)
    if aligned:
        assert x.data_ptr() % 16 == 0
    else:
        assert x.data_ptr() % 16 != 0
    nrm, e = dee_postprocess(x, normals=flags[0], nms=flags[1], hysteresis=flags[2], t_low=tl, t_high=th,
                             out_dtype=torch.float32 if out == np.float32 else torch.float64)
    return (None if nrm is None else nrm.cpu().numpy()), (None if e is None else e.cpu().numpy())


def expected_edges(p, nms, hyst, tl=0.3, th=0.7):
    from oracle import dee as odee
    with np.errstate(all="ignore"):
        if nms:
            e = odee.non_max_suppression(p)
            return odee.hysteresis(e, tl, th) if hyst else e
        return odee.hysteresis(p, tl, th)


def check(probs, flags=(True, True, True), out=np.float32, tl=0.3, th=0.7, fronts=None, tag=""):
    """Run every front the shape allows (or the given ones), compare each with the oracle and with each other."""
    from oracle import dee as odee
    N, H, W = probs.shape
    if fronts is None:
        fronts = [True, False] if front_path(probs.dtype, H, W) == "tma" else [True]
    res = [run_dee(probs, flags, out, a, tl, th) for a in fronts]
    for k in range(N):
        if flags[0]:
            with np.errstate(all="ignore"):
                ref_n = odee.normals_u8(probs[k])
            for (nrm, _), a in zip(res, fronts):
                assert nrm.dtype == np.uint8 and np.array_equal(nrm[k], ref_n), (tag, "normals", k, a)
        if flags[1] or flags[2]:
            ref = expected_edges(probs[k], flags[1], flags[2], tl, th)
            with np.errstate(all="ignore"):
                ref = ref.astype(out)
            for (_, e), a in zip(res, fronts):
                assert _eq(e[k], ref), (tag, "edges", k, a, int((~((e[k] == ref) | (np.isnan(e[k]) & np.isnan(ref)))).sum()))
    for (n1, e1), (n2, e2) in zip(res, res[1:]):   # the TMA and generic fronts agree bit for bit, output for output
        assert (n1 is None) == (n2 is None) and (n1 is None or np.array_equal(n1, n2)), tag
        assert (e1 is None) == (e2 is None) and (e1 is None or np.array_equal(e1.view(np.uint8), e2.view(np.uint8))), tag
    return res[0]


def _matrix_planes(dtype):
    H, W = 70, 260   # 3 x 3 TMA tiles (128 x 31) and 5 x 5 generic tiles (64 x 16), partial last ones
    a = prob_map(H, W, 5)
    b = prob_map(H, W, 6)
    r = np.random.default_rng(7)
    idx = r.integers(2, H - 2, 12), r.integers(2, W - 2, 12)
    b[idx[0][:4], idx[1][:4]] = np.nan
    b[idx[0][4:8], idx[1][4:8]] = np.inf
    b[idx[0][8:], idx[1][8:]] = [0.3, 0.7, np.float32(0.3), -0.0]
    b[0, :] = r.uniform(-0.5, 3.0, W)   # raw border values that decide the max in the raw-map hysteresis
    c = prob_map(H, W, 8) * 0.5         # no strong pixel: a 0 / 0 NaN plane after the NMS
    return np.stack([a, b, c]).astype(dtype)


MATRIX = [(f, i, o) for f in FLAGS for i in (np.float32, np.float64) for o in (np.float32, np.float64)
          if f[1] or f[2] or o == np.float32]


@pytest.mark.gpu
@pytest.mark.parametrize("flags,in_dt,out_dt", MATRIX,
                         ids=[f"{_flag_id(f)}-in{np.dtype(i).itemsize * 8}-out{np.dtype(o).itemsize * 8}" for f, i, o in MATRIX])
def test_configuration_matrix(flags, in_dt, out_dt):
    """Each flag combination x input dtype x output dtype, fp32 planes through both front kernels (aligned: TMA;
    one element into the buffer: generic), at a shape with several tiles of each front and partial last tiles."""
    check(_matrix_planes(in_dt), flags, out_dt, tag=(flags, in_dt, out_dt))


@pytest.mark.gpu
def test_bench_configuration():
    """bench.py's dee workload: fp32 in, fp32 out, normals + NMS + hysteresis, 8 x 384 x 1280."""
    probs = np.stack([prob_map(384, 1280, 300 + k) for k in range(8)])
    probs[5] *= 0.5
    nrm, e = check(probs, fronts=[True], tag="bench")
    assert e.dtype == np.float32 and (e[0] > 0).any()


SHAPES = [(1, 1), (1, 9), (9, 1), (2, 2), (2, 9), (9, 2), (3, 3),
          (4, 4), (4, 5), (5, 4), (6, 9), (6, 10), (6, 11)] + \
         [(h, w) for h in (30, 31, 32, 62, 63) for w in (128, 132, 260)] + \
         [(375, 1242), (384, 1280), (480, 1280), (640, 1280), (1216, 1936)]


def _shape_planes(H, W, dtype):
    r = np.random.default_rng(H * 7919 + W)
    a = prob_map(H, W, H + W)
    b = np.where(r.random((H, W)) < 0.35, r.uniform(0.3, 1.0, (H, W)), r.uniform(-0.2, 0.3, (H, W)))
    return np.stack([a, b.astype(np.float32)]).astype(dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES, ids=[f"{h}x{w}" for h, w in SHAPES])
def test_shapes(shape):
    """Tiny planes (no interior: NMS output zero, hysteresis img * img / max), the TMA limits, the tile sizes, KITTI
    raw frames (generic front, L2 hysteresis), both sides of the shared-memory / BIG boundary and DDAD size (BIG with
    one pair): all three stages in fp32 and fp64, and the hysteresis of the raw map."""
    H, W = shape
    for dt in (np.float32, np.float64):
        probs = _shape_planes(H, W, dt)
        check(probs, (True, True, True), dt, tag=(shape, dt))
        check(probs, (False, False, True), dt, tag=(shape, dt, "raw"))


# ---- values that decide labels -------------------------------------------------------------------------------------
THRESHOLDS = [(0.3, 0.7), (0.2, 0.5), (0.1, 0.3), (0.7, 0.9), (0.25, 0.5), (0.5, 0.5), (0.6, 0.4)]


def _threshold_values(t, dtype):
    """float32(t), both fp32 neighbours of it, and for fp64 planes t itself and both fp64 neighbours."""
    f = np.float32(t)
    vals = {float(f), float(np.nextafter(f, np.float32(np.inf))), float(np.nextafter(f, np.float32(-np.inf)))}
    if dtype == np.float64:
        vals |= {t, float(np.nextafter(t, np.inf)), float(np.nextafter(t, -np.inf))}
    return sorted(vals)


def _raw_threshold_plane(vals, dtype, S=1.0):
    """One row per value: the value alone (an edge iff strong) and the value next to a strong pixel (an edge iff a
    candidate)."""
    H, W = 3 * len(vals) + 4, 16
    p = np.zeros((H, W), dtype)
    for i, v in enumerate(vals):
        y = 2 + 3 * i
        p[y, 2] = v
        p[y, 6], p[y, 7] = S, v
    return p


def _ridge_threshold_plane(vals, dtype, S=1.0):
    """Rows constant along x (no x gradient), so the NMS keeps the value of each ridge row unchanged: per value a row
    between two strong rows (an edge iff a candidate, compared in fp64) and a lone row (an edge iff strong)."""
    rows = []
    for v in vals:
        rows += [0, 0, S, v, S, 0, 0, 0, 0, v, 0, 0]
    rows = [0] + rows + [0]
    return np.repeat(np.array(rows, dtype)[:, None], 20, axis=1)


@pytest.mark.gpu
@pytest.mark.parametrize("tl,th", THRESHOLDS)
def test_pixels_on_thresholds(tl, th):
    """Pixels at float32(t), its fp32 neighbours and (fp64 planes) t and its fp64 neighbours, for both thresholds:
    raw hysteresis compares in the input dtype with the thresholds rounded to it; after the NMS the comparison is in
    fp64 (the TMA front uses the fp32 thresholds rounded down / up, which must decide the same)."""
    for dt in (np.float32, np.float64):
        vals = sorted(set(_threshold_values(tl, dt) + _threshold_values(th, dt)))
        for out in (np.float32, np.float64):
            check(_raw_threshold_plane(vals, dt)[None], (False, False, True), out, tl, th, tag=("raw", dt, out))
            check(_ridge_threshold_plane(vals, dt)[None], (True, True, True), out, tl, th, tag=("nms", dt, out))


def _value_planes():
    """Same-shape planes for one batch, so that a wrong per-image statistic shows."""
    H, W = 20, 36
    r = np.random.default_rng(23)
    base = lambda: r.uniform(0.0, 0.25, (H, W))   # below every t_low used with these planes but one
    planes = []
    p = base(); p[5, 3:9] = 0.5; p[5, 2] = 0.9; p[5, 9] = np.nan; p[5, 10:20] = 0.5; planes.append(p)  # NaN bridge
    p = base(); p[8, 8] = np.inf; p[9, 9:14] = 0.5; p[12, 20] = np.inf; planes.append(p)                # +Inf interior
    p = base(); p[4, 4] = 0.95; p[0, 7] = np.nan; planes.append(p)                                      # NaN border
    p = base(); p[4, 4] = 0.95; p[H - 1, 30] = np.inf; planes.append(p)                                 # +Inf border
    p = base(); p[4, 4] = 0.95; p[:, 0] = -5.0; p[:, W - 1] = 3.0; planes.append(p)                    # border max 3
    p = base(); p[0, :] = -1.0; p[:, 0] = -2.0; p[H - 1, :] = -0.5; p[:, W - 1] = -0.25; planes.append(p)  # no strong
    p = base(); p[1:-1, 1:-1] = r.uniform(0.75, 1.0, (H - 2, W - 2)); planes.append(p)                  # all strong
    p = base(); p[3, 3] = -np.inf; p[10, 10] = 0.9; p[10, 11] = -np.inf; p[10, 12] = 0.5; planes.append(p)
    planes.append(prob_map(H, W, 77).astype(np.float64))
    planes.append(np.zeros((H, W)))
    return np.stack(planes)


@pytest.mark.gpu
def test_values_that_decide_labels():
    """NaN bridging a strong pixel to a weak run (NaN is a candidate), +Inf interior pixels, a NaN / +Inf / negative
    border (np.max over the raw border: NaN plane, 2 / inf, or a border maximum), no strong pixel (0 / 0), an all-strong
    interior, -Inf next to a strong pixel: mixed in one batch, raw and after the NMS, every dtype and front."""
    probs = _value_planes()
    for dt in (np.float32, np.float64):
        p = probs.astype(dt)
        for out in (np.float32, np.float64):
            e = check(p, (False, False, True), out, tag=("raw", dt, out))[1]
            check(p, (True, True, True), out, tag=("nms", dt, out))
            if out == np.float32:
                assert np.isnan(e[2]).all() and (e[0][5, 10:20] > 0).all() and np.isinf(e[1][8, 8])
                assert (e[3][1:-1, 1:-1][~np.isnan(e[3][1:-1, 1:-1])] == 0).all()
    for tl, th in [(0.5, 0.5), (0.6, 0.4), (0.1, 0.3)]:
        check(probs.astype(np.float32), (False, False, True), np.float32, tl, th, tag=("raw", tl, th))


# ---- hysteresis structures (raw mode: the label plane is whatever the input says) -----------------------------------
STRUCT_SHAPES = [(480, 1280), (1216, 1936), (375, 1242)]


def serpentine(H, W, weak=0.5, strong=0.9):
    """A one-pixel weak path filling the plane, strong only at its start: it crosses every tile, one flood round or
    more per row."""
    p = np.zeros((H, W), np.float32)
    rows = list(range(1, H - 1, 2))
    for k, y in enumerate(rows):
        p[y, 1:W - 1] = weak
        if k + 1 < len(rows):
            p[y + 1, W - 2 if k % 2 == 0 else 1] = weak
    p[1, 1] = strong
    return p


def lattice(H, W, seed=31):
    """Weak clusters below the percolation density, and a strong pixel in every bitmap word of every other row: the
    flood's first worklist overflows (full-sweep mode), and a dropped seed leaves its cluster dark."""
    r = np.random.default_rng(seed)
    p = np.where(r.random((H, W)) < 0.3, r.uniform(0.3, 0.7, (H, W)), r.uniform(0.0, 0.3, (H, W))).astype(np.float32)
    p[1:H - 1:2, 5:W - 1:32] = 0.95
    return p


@pytest.mark.gpu
@pytest.mark.parametrize("shape", STRUCT_SHAPES, ids=[f"{h}x{w}" for h, w in STRUCT_SHAPES])
def test_hysteresis_structures(shape):
    H, W = shape
    probs = np.stack([serpentine(H, W), lattice(H, W)])
    _, e = check(probs, (False, False, True), np.float32, tag=shape)
    assert (e[0][probs[0] > 0] > 0).all()


# ---- Canny (u8 images through canny_from_depth) ---------------------------------------------------------------------
NESTED = [(int(t / 2), int(t)) for t in range(240, 19, -20)]
HANDOFF_PAIRS = [(80, 160), (40, 80), (10, 20)]
CANNY_SHAPES = [(640, 1280), (1216, 1936)]


def u8_scene(H, W, seed):
    import cv2
    r = np.random.default_rng(seed)
    d = np.full((H, W), 100.0)
    for _ in range(24):
        y0, x0 = r.integers(0, H), r.integers(0, W)
        h, w = r.integers(1, max(2, H // 3)), r.integers(1, max(2, W // 3))
        d[y0:y0 + h, x0:x0 + w] = r.uniform(0, 255)
    d = cv2.GaussianBlur(d, (5, 5), 1.5) + r.normal(0, 1.0, (H, W))
    return np.clip(d, 0, 255).astype(np.uint8)


def u8_noise(H, W, seed=5):
    return np.random.default_rng(seed).integers(0, 256, (H, W)).astype(np.uint8)


def canny_cases():
    """(name, images, pairs) of test_canny_paths."""
    cases = []
    for H, W in CANNY_SHAPES:
        imgs = np.stack([u8_scene(H, W, 1), u8_scene(H, W, 2)])
        cases += [(f"{H}x{W}-one", imgs, [(20, 40)]), (f"{H}x{W}-nested", imgs, NESTED)]
    cases.append(("640x1280-handoff", np.stack([u8_scene(640, 1280, 3), u8_noise(640, 1280)]), HANDOFF_PAIRS))
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("k", range(5), ids=["640x1280-one", "640x1280-nested", "1216x1936-one", "1216x1936-nested",
                                              "640x1280-handoff"])
def test_canny_paths(k):
    """BIG hysteresis with one pair and with the 12 nested pairs, and an image whose reachable set is beyond the BIG
    kernel's candidate capacity, handed to the L2 kernel next to one that stays: edges and levels against cv2.Canny."""
    import cv2
    from mindtheedge_b200.edge import canny_from_depth
    name, imgs, pairs = canny_cases()[k]
    edges, levels = canny_from_depth(torch.from_numpy(imgs).cuda(), pairs, want_edges=True, want_levels=True)
    edges, levels = edges.cpu().numpy(), levels.cpu().numpy()
    for n in range(len(imgs)):
        for t, (lo, hi) in enumerate(pairs):
            ref = cv2.Canny(imgs[n], lo, hi)
            assert np.array_equal(edges[t, n], ref), (name, n, t, int((edges[t, n] != ref).sum()))
            assert np.array_equal((levels[n] <= t) * 255, ref), (name, n, t)


# ---- a batch beyond one finish launch -----------------------------------------------------------------------------
N_LARGE, N_PATTERNS = 65543, 19   # 19 does not divide 65,535 = 3 * 5 * 17 * 257: image 65,535 + k differs from image k


def small_patterns():
    r = np.random.default_rng(41)
    pats = []
    for k in range(N_PATTERNS):
        p = r.uniform(0.0, 1.0, (8, 8))
        kind = k % 4
        if kind == 1:
            p[0 if k % 2 else 7, r.integers(0, 8)] = np.nan       # NaN border: a NaN plane
        elif kind == 2:
            p *= 0.65                                             # no strong pixel
        elif kind == 3:
            p[1:-1, 1:-1] = r.uniform(0.75, 1.0, (6, 6))          # all strong
        if k % 3 == 0:
            p[:, 0] = -r.uniform(0.0, 2.0, 8)
        if k % 5 == 0:
            p[:, 7] = r.uniform(1.0, 4.0, 8)                      # the border decides the max
        if k == 6:
            p[3, 0] = np.inf
        pats.append(p.astype(np.float32))
    return np.stack(pats)


@pytest.mark.gpu
def test_batch_beyond_one_finish_launch():
    """65,543 planes of 8 x 8, fp32 in and out (float4 finish, two launches of 65,535 and 8 images), 19 patterns in a
    cycle: every image against its pattern's oracle result, raw hysteresis and all three stages."""
    from oracle import dee as odee
    pats = small_patterns()
    idx = np.arange(N_LARGE) % N_PATTERNS
    probs = pats[idx]
    for flags in [(False, False, True), (True, True, True)]:
        nrm, e = run_dee(probs, flags, np.float32, True)
        for k in range(N_PATTERNS):
            sel = idx == k
            ref = expected_edges(pats[k], flags[1], flags[2])
            with np.errstate(all="ignore"):
                ref = ref.astype(np.float32)
            got = e[sel]
            assert _eq(got, np.broadcast_to(ref, got.shape).copy()), (flags, k, np.nonzero(~np.all(
                (got == ref) | (np.isnan(got) & np.isnan(ref)), axis=(1, 2)))[0][:8])
            if flags[0]:
                assert np.array_equal(nrm[sel], np.broadcast_to(odee.normals_u8(pats[k]), got.shape)), k
        del nrm, e


# ---- coverage manifest (no GPU work) ------------------------------------------------------------------------------
def _margin_ok(value, boundary):
    return value <= 0.9 * boundary or value >= 1.1 * boundary


def test_path_manifest():
    """Restates which front, hysteresis kernel, flood mode and finish path every case above selects; each path must be
    taken by at least one case, and each case must lie at least 10 % away from the shared-memory / BIG boundary, the
    flood worklist capacity and the candidate capacity (so that a shift of the opt-in shared memory or of the kernel's
    static shared memory cannot move a case across silently).  The batch-slice boundary (65,535 images) is exact and
    is straddled on purpose."""
    seen = set()
    problems = []

    def dee_case(tag, dtype, out, N, H, W, aligned=True, hyst=True, strong=None):
        seen.add(("front", front_path(dtype, H, W, aligned)))
        if not hyst:
            return
        kernel, _ = hyst_plan(H, W)
        seen.add(("hyst", kernel, "T=1"))
        fin, slices = finish_path(dtype, out, N, H, W)
        seen.add(("finish", fin))
        seen.add(("slices", slices))
        hb = big_boundary(W)
        if hb is not None and not _margin_ok(H, hb):
            problems.append((tag, "BIG boundary", H, hb))
        if strong is not None and kernel != "l2":
            words = max(seeded_words(s) for s in strong)
            seen.add(("flood", "full" if words > WORK_CAP else "worklist"))
            if not _margin_ok(words, WORK_CAP):
                problems.append((tag, "worklist", words))

    for flags, i, o in MATRIX:
        planes = _matrix_planes(i)
        for aligned in ((True, False) if i == np.float32 else (True,)):
            dee_case(("matrix", flags), i, o, *planes.shape, aligned, flags[2])
    for H, W in SHAPES:
        for dt in (np.float32, np.float64):
            dee_case(("shape", H, W), dt, dt, 2, H, W, True)
            if front_path(dt, H, W) == "tma":
                dee_case(("shape", H, W), dt, dt, 2, H, W, False)
    for H, W in STRUCT_SHAPES:
        s = [dee_strong(serpentine(H, W), 0.7), dee_strong(lattice(H, W), 0.7)]
        dee_case(("struct", H, W), np.float32, np.float32, 2, H, W, True, True, s[1:])
        dee_case(("struct", H, W), np.float32, np.float32, 2, H, W, True, True, s[:1])
    dee_case("batch", np.float32, np.float32, N_LARGE, 8, 8)
    for name, imgs, pairs in canny_cases():
        import cv2
        N, H, W = imgs.shape
        kernel, cap = hyst_plan(H, W)
        seen.add(("hyst", kernel, "T=1" if len(pairs) == 1 else "T>1"))
        hb = big_boundary(W)
        if hb is not None and not _margin_ok(H, hb):
            problems.append((name, "BIG boundary", H, hb))
        if len(pairs) > 1 and kernel != "l2":
            lo, hi = pairs[-1]   # the reachable set of nested pairs is the loosest pair's edge set
            for n in range(N):
                reach = int((cv2.Canny(imgs[n], lo, hi) > 0).sum())
                seen.add(("handoff", reach > cap))
                if not _margin_ok(reach, cap):
                    problems.append((name, n, "candidate cap", reach, cap))
    assert not problems, problems
    want = {("front", "tma"), ("front", "generic"),
            ("hyst", "smem", "T=1"), ("hyst", "big", "T=1"), ("hyst", "l2", "T=1"),
            ("hyst", "big", "T>1"),
            ("finish", "vector"), ("finish", "scalar"), ("slices", 1), ("slices", 2),
            ("flood", "full"), ("flood", "worklist"), ("handoff", True), ("handoff", False)}
    assert want <= seen, sorted(want - seen, key=str)
    # the numbers the boundary is derived from: 576 rows stay in shared memory at W = 1280, 577 do not
    assert big_boundary(1280) == 577 and hyst_plan(1216, 1936)[0] == "big" and hyst_plan(1216, 1936)[1] == 37216


@pytest.mark.gpu
def test_manifest_constants_match_device():
    assert torch.cuda.get_device_properties(0).shared_memory_per_block_optin == OPTIN
