"""The one-pass loss kernel's cross-CTA synchronisation over many launches.

edge_loss_fused_kernel meets all its CTAs once at a grid barrier and elects the last CTA by a ticket; the rescale
kernel behind it elects its last CTA by a counter of its own.  All three counters reset themselves, so the workspace
header is zero again after every launch.  Here about 100 fused + rescale steps run back to back inside ONE CUDA graph
on a single workspace, with rotating input sets and upstream gradients that alternate between the expected one (the
rescale kernel exits at once) and another one (it rescales d loss / d pred): every step must be bit-equal to the same
step run eagerly on a fresh workspace, and the header must be all zero afterwards.  Shapes whose grid is smaller than
the SM count (one CTA) and the benchmark's pyramid.
"""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

STEPS = 100
UPSTREAMS = (1.0, 0.3)   # 1 is what the fused kernel produces for (no expectation given): the rescale kernel exits


def _inputs(B, H, W, n, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    out = []
    for s in range(n):
        h, w = H >> s, W >> s
        inv = 1.0 / (torch.rand(B, 1, h, w, generator=g) * 79 + 1)
        u = torch.rand(B, 1, h, w, generator=g)
        edge = (u < 0.015).float() * torch.rand(B, 1, h, w, generator=g).clamp(min=0.3)
        k = torch.randint(0, 256, (B, 1, h, w), generator=g).float()
        normal = ((360 * k / 255 - 180) * np.pi / 180).float()
        out.append(tuple(t.cuda() for t in (inv, edge, normal)))
    return out


class _Step:
    """Output buffers and the C-ABI arguments of one fused + rescale step."""

    def __init__(self, scales, weights, upstream):
        from mindtheedge_b200.losses import _scales_struct
        n = len(scales)
        self.gmap = [torch.empty_like(e) for _, e, _ in scales]
        self.gpred = [torch.empty_like(p) for p, _, _ in scales]
        self.sc = _scales_struct([t[0] for t in scales], [t[1] for t in scales], [t[2] for t in scales], None,
                                 self.gmap, self.gpred, weights)
        self.loss = torch.zeros(1 + n, device="cuda")
        self.gl = torch.zeros(1 + n, device="cuda")
        self.gl[0] = upstream
        self.n = n

    def launch(self, at, ctx, ws, stream):
        from mindtheedge_b200 import _lib
        _lib.check(_lib.lib.mte_edge_loss_fwd_grad(self.sc, self.n, C.byref(at), None, self.loss.data_ptr(),
                                                   ctx.data_ptr(), ws.data_ptr(), ws.numel(), stream))
        _lib.check(_lib.lib.mte_edge_loss_grad_rescale(self.sc, self.n, self.gl.data_ptr(), ctx.data_ptr(), None,
                                                       stream))


def _buffers(sc, n):
    from mindtheedge_b200 import _lib
    ctx = torch.zeros(_lib.lib.mte_edge_loss_ctx_bytes(sc, n) // 4, device="cuda")
    ws = torch.zeros(_lib.lib.mte_edge_loss_workspace_bytes(sc, n), dtype=torch.uint8, device="cuda")
    return ctx, ws


@pytest.mark.parametrize("shape,n,sets", [((1, 2, 4), 1, 4), ((2, 1, 32), 1, 4), ((8, 384, 1280), 4, 3)],
                         ids=["1x2x4", "2x1x32", "bench_8x384x1280"])
def test_graph_of_steps_matches_eager_and_leaves_header_zero(shape, n, sets):
    from mindtheedge_b200 import _lib
    from mindtheedge_b200.losses import _attrs
    B, H, W = shape
    at = _attrs(True, True, True, 4.0, 10.0, 1.0)
    weights = [1.0 / n] * n
    inputs = [_inputs(B, H, W, n, seed=100 * sum(shape) + i) for i in range(sets)]
    # step k: input set k % sets, upstream gradient UPSTREAMS[(k // sets) % 2] -- every (set, upstream) pair recurs
    combo = [(k % sets, (k // sets) % 2) for k in range(STEPS)]
    steps = [_Step(inputs[s], weights, UPSTREAMS[u]) for s, u in combo]
    ctx, ws = _buffers(steps[0].sc, n)

    # eager reference: each (set, upstream) pair once, on a fresh workspace
    ref = {}
    stream = torch.cuda.current_stream().cuda_stream
    for s in range(sets):
        for u in range(len(UPSTREAMS)):
            st = _Step(inputs[s], weights, UPSTREAMS[u])
            c1, w1 = _buffers(st.sc, n)
            st.launch(at, c1, w1, stream)
            torch.cuda.synchronize()
            assert not w1[:_lib.MTE_WS_HEADER_BYTES].any()
            ref[(s, u)] = st
    for s in range(sets):   # the second upstream gradient really took the rescaling path: grad_pred * (0.3 w / w)
        for i in range(n):
            w32 = np.float32(weights[i])
            f = float(np.float32(np.float32(UPSTREAMS[1]) * w32) / w32)
            assert torch.equal(ref[(s, 1)].gpred[i], ref[(s, 0)].gpred[i] * f), (s, i)
            assert torch.equal(ref[(s, 1)].gmap[i], ref[(s, 0)].gmap[i])

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        for st in steps:
            st.launch(at, ctx, ws, side.cuda_stream)
    for st in steps:   # the capture ran nothing: clear the outputs so every checked value comes from the replay
        st.loss.zero_()
        for t in st.gmap + st.gpred:
            t.fill_(float("nan"))
    torch.cuda.synchronize()
    g.replay()
    torch.cuda.synchronize()
    assert not ws[:_lib.MTE_WS_HEADER_BYTES].any(), "workspace header not reset"
    for k, (st, key) in enumerate(zip(steps, combo)):
        r = ref[key]
        assert torch.equal(st.loss, r.loss), (k, st.loss, r.loss)
        for s in range(n):
            assert torch.equal(st.gmap[s], r.gmap[s]), (k, s)
            assert torch.equal(st.gpred[s], r.gpred[s]), (k, s)
