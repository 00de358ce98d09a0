#!/usr/bin/env python
"""Benchmark of the MindTheEdge depth-edge hot path on B200 (the driver's contract).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl mte|reference]
                    [--workload loss|auc|dee|ddad|train] [--dump-outputs DIR]

One JSON line on stdout (rank 0).  K is the number of timed steps of the workload's headline number.  With
--dump-outputs, rank 0 writes what the timed path computed in its last timed step as DIR/<name>.npy (see
dump_outputs); the inputs are seeded, so two builds run with the same arguments can be compared output for output.
The library must have been built before (__graft_entry__.build()): the bench compiles nothing.
Workloads = BASELINE.json configs:

loss   (headline; configs 1/3 loss shape) per GPU a batch of 8 images x the 4-scale pyramid (384x1280 ... 48x160,
       fp32, DEE normals, no mask, inv2depth fused) -> 5.22 Mpixel per step; a step is one forward + one backward
       of the edge loss.  The same line carries the KITTI-DE AUC evaluation under "auc_eval".
auc    (config 2) the 102 bundled KITTI-DE GT maps vs synthetic predicted depth, 12 Canny settings, exact matcher.
dee    (config 4) DEE annotation post-process (Sobel5 normals + NMS + hysteresis) over KITTI-size frames,
       frame-sharded, no collective.
ddad   (config 5) DDAD-size (1216x1936) AUC evaluation, image-sharded, one int64 all-reduce.
train  (config 3) a stock-PyTorch conv trunk emitting 4 inverse-depth scales under DistributedDataParallel + this
       loss + one SGD step; the same step with the eager-PyTorch port of the loss is timed beside it.

value      device-timed (CUDA events on the launching stream, max over ranks), inputs resident in HBM, steps rotate
           over input sets larger than L2 (or the inputs exceed L2 by themselves);
e2e        the same metric through the public torch API with HOST buffers: pinned H2D of every step's inputs
           (double-buffered on a copy stream) and D2H of the result inside the timed region;
roofline   algorithmic bytes (SURVEY.md 8d) / measured time vs MEASURED_PEAKS.json;
cpu_baseline  the reference's own CPU code (oracle/_ref, staged by oracle/make_ref.py: kind "reference") or, when it
           is not staged, the oracle port (kind "port") on a bounded sample, run in a subprocess of this bench;
`--impl reference` times that CPU arm alone (rank 0 only) on the same workload configuration.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

H0, W0, SCALES, B_PER_GPU = 384, 1280, 4, 8
LOSS_BYTES_PER_PX = 32.0   # fwd 16 (depth+edge+normal in, grad map out) + bwd 16 (recompute in, grad out)
AUC_BYTES_PER_PX = 7.0     # per (image, threshold): extraction 5 + counts 2 (SURVEY.md 8d)
DEE_BYTES_PER_PX = 9.0     # prob fp32 in, normal u8 + edge fp32 out
KITTI_N, KITTI_T = 102, 12
KITTI_CROP = [44, 1197, 153, 371]
DDAD_H, DDAD_W, DDAD_N = 1216, 1936, 8
DEE_FRAMES = 148   # one frame per SM for the one-CTA-per-frame hysteresis
DUMP_BYTES = 60 * 10**6   # --dump-outputs budget: stays under 64 MB with the .npy headers


def dump_outputs(out_dir, arrays):
    """Write every array as <out_dir>/<name>.npy: float64 for float64 data and integers wider than 16 bits, float32
    (exact) otherwise.  When the set exceeds DUMP_BYTES, every array keeps the same share of its elements at flat
    positions drawn by np.random.default_rng(0) (sorted), so that arrays of one size are sampled at the same positions
    in every run."""
    conv = {}
    for name, a in arrays.items():
        a = np.asarray(a)
        wide = a.dtype == np.float64 or (np.issubdtype(a.dtype, np.integer) and a.dtype.itemsize > 2)
        conv[name] = a.astype(np.float64 if wide else np.float32)
    total = sum(a.nbytes for a in conv.values())
    share = min(1.0, DUMP_BYTES / total) if total else 1.0
    picks = {}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in conv.items():
        if share < 1.0:
            if a.size not in picks:
                picks[a.size] = np.sort(np.random.default_rng(0).choice(a.size, int(a.size * share), replace=False))
            a = a.reshape(-1)[picks[a.size]]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def recorded_traffic(kind):
    """Per-step DRAM bytes of the dominant kernels from the committed ncu capture, if any."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(p)).get(kind)
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True).start()
        except Exception:
            self.proc = None

    def settle(self, step, seconds=0.25):
        """nvidia-smi needs ~0.1-0.2 s before its first sample: keep the GPU under the same load (untimed steps)
        until then, so that short timed regions are sampled under load as well."""
        t0 = time.perf_counter()
        while self.proc is not None and time.perf_counter() - t0 < seconds:
            step()
            torch.cuda.synchronize()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------
# plumbing
# ---------------------------------------------------------------------------
def dist_setup(n_gpus):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, local


def bind_to_gpu_cores(local, world):
    """Pin this rank to its own slice of the cores nvidia-smi reports for the GPU (all GPUs of these boxes report the
    same affinity mask, so the slice keeps the ranks' staging threads off each other's cores).  Pinned host buffers
    are allocated AFTER this, so first-touch places them next to those cores."""
    try:
        cores = sorted(os.sched_getaffinity(0))
        if world > 1 and len(cores) >= world:
            per = len(cores) // world
            os.sched_setaffinity(0, set(cores[local * per:(local + 1) * per]))
        return len(os.sched_getaffinity(0))
    except Exception:
        return None


def barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(ms, world, device):
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([ms], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    return ms


def h2d_probe(world, device, mb=256, reps=4):
    """Pinned host -> device copy bandwidth of this rank while ALL ranks copy at once (GB/s, min over ranks): names
    the limiter of the e2e numbers (PCIe per GPU at N=1, the shared host memory / root complex at N=8)."""
    h = torch.empty(mb << 20, dtype=torch.uint8).pin_memory()
    d = torch.empty(mb << 20, dtype=torch.uint8, device=device)
    d.copy_(h, non_blocking=True)
    barrier(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        d.copy_(h, non_blocking=True)
    e1.record()
    barrier(world)
    ms = max_over_ranks(e0.elapsed_time(e1), world, device)
    return round(reps * (mb << 20) / (ms * 1e-3) / 1e9, 1)


class DoubleBuffer:
    """e2e input staging: per step ONE pinned host buffer -> ONE device buffer, copied on a side stream while the
    previous step computes (two slots).  Every step's copy is issued inside the timed region."""

    def __init__(self, host_bufs, device):
        self.h = host_bufs                                   # two pinned uint8/float tensors (same layout)
        self.d = [torch.empty_like(b, device=device) for b in host_bufs]
        self.copy_stream = torch.cuda.Stream(device)
        self.ready = [torch.cuda.Event(), torch.cuda.Event()]
        self.free = [torch.cuda.Event(), torch.cuda.Event()]
        self.issued = 0

    def issue(self, j):
        s = j % 2
        with torch.cuda.stream(self.copy_stream):
            if j >= 2:
                self.copy_stream.wait_event(self.free[s])
            self.d[s].copy_(self.h[s], non_blocking=True)
            self.ready[s].record(self.copy_stream)

    def run(self, n, compute):
        """compute(slot, device_buffer) runs on the current stream.  Copy j+1 overlaps compute j."""
        main = torch.cuda.current_stream()
        self.issue(0)
        for i in range(n):
            if i + 1 < n:
                self.issue(i + 1)
            main.wait_event(self.ready[i % 2])
            compute(i % 2, self.d[i % 2])
            self.free[i % 2].record(main)


def time_region(fn, world, device, stream=None):
    """CUDA-event time of fn() on the launching stream, barrier + synchronize on both sides, max over ranks (ms)."""
    barrier(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    out = fn()
    e1.record(stream)
    barrier(world)
    return max_over_ranks(e0.elapsed_time(e1), world, device), out


# ---------------------------------------------------------------------------
# synthetic inputs (SURVEY.md 8d)
# ---------------------------------------------------------------------------
def loss_inputs(B, seed, device, pinned=False):
    """inverse depth, soft edges, u8-decoded normals at the 4 pyramid sizes."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    out = []
    for s in range(SCALES):
        h, w = H0 >> s, W0 >> s
        depth = torch.rand(B, 1, h, w, generator=g) * 79 + 1
        inv = 1.0 / depth
        u = torch.rand(B, 1, h, w, generator=g)
        edge = (u < 0.015).float() * torch.rand(B, 1, h, w, generator=g).clamp(min=0.3)
        k = torch.randint(0, 256, (B, 1, h, w), generator=g).float()
        normal = ((360 * k / 255 - 180) * np.pi / 180).float()
        out.append((inv, edge, normal))
    if device is not None:
        return [tuple(t.to(device) for t in sc) for sc in out]
    if pinned:
        return [tuple(t.pin_memory() for t in sc) for sc in out]
    return out


def loss_inputs_u8(B, seed):
    """The same step in the encoding the reference's dataloader holds (datasets/gta_dataset.py:406-422): inverse depth
    fp32 (stands for the trunk output), edge and normal planes as the u8 PNG values of the annotation pass."""
    g = torch.Generator().manual_seed(seed)
    shapes = [(B, H0 >> s, W0 >> s) for s in range(SCALES)]
    n_px = sum(b * h * w for b, h, w in shapes)
    inv = 1.0 / (torch.rand(n_px, generator=g) * 79 + 1)
    e8 = ((torch.rand(n_px, generator=g) < 0.015) * torch.randint(77, 256, (n_px,), generator=g)).to(torch.uint8)
    n8 = torch.randint(0, 256, (n_px,), generator=g).to(torch.uint8)
    return shapes, n_px, inv, e8, n8


def kitti_like_set(n, seed0):
    """BASELINE.json config 2: the reference's bundled KITTI-DE GT edge maps (tests/golden/kitti_de_gt.npz, packed from
    data/kitti_de/gt by tests/golden/make_kitti_gt.py) against SYNTHETIC predicted depth built as SURVEY.md 8(d)
    prescribes: the connected components of the non-edge pixels filled with U(3, 80) m plus N(0, 0.3^2) noise, seeded
    per image.  The annotated contours are mostly open curves, so they are closed by one 3x3 dilation before the
    labelling (without it the recipe leaves ~17 regions and ~400 predicted edge pixels per crop against ~3200 GT
    pixels; with it ~96 regions and ~1900).  Without the fixture: synthetic scenes at the bundled set's mean edge
    density (1.45 %)."""
    fx = os.path.join(ROOT, "tests", "golden", "kitti_de_gt.npz")
    if not os.path.exists(fx):
        from synth import scene_with_gt
        gts, depths = zip(*[scene_with_gt(H0, W0, seed0 + i, n_rect=18) for i in range(n)])
        return np.stack(depths), np.stack([(g > 127).astype(np.uint8) for g in gts])
    from scipy import ndimage
    z = np.load(fx)
    shp = tuple(int(v) for v in z["shape"])
    gt_all = np.unpackbits(z["bits"])[: int(np.prod(shp))].reshape(shp).astype(bool)
    depths, gts = [], []
    for i in range(n):
        g = gt_all[i % shp[0]]
        lab, k = ndimage.label(~ndimage.binary_dilation(g, iterations=1))
        lab = np.where(lab == 0, ndimage.maximum_filter(lab, size=5), lab)  # a contour pixel takes a neighbouring region
        r = np.random.default_rng(seed0 + i)
        vals = r.uniform(3.0, 80.0, k + 1).astype(np.float32)
        d = vals[lab] + r.normal(0.0, 0.3, g.shape).astype(np.float32)
        depths.append(d.astype(np.float32))
        gts.append(g.astype(np.uint8))
    return np.stack(depths), np.stack(gts)


def ddad_like_set(n, seed0):
    """BASELINE.json config 5: synthetic 1216x1936 scenes (SURVEY.md 8d: the bundled DDAD GT is 384x640, so GT =
    region boundaries of a piecewise-constant scene at ~1.1 % density; predicted depth = the scene shifted + noise)."""
    from synth import scene_with_gt
    gts, depths = zip(*[scene_with_gt(DDAD_H, DDAD_W, seed0 + i, n_rect=60) for i in range(n)])
    return np.stack(depths), np.stack([(g > 127).astype(np.uint8) for g in gts])


def dee_frames(n, seed0):
    """BASELINE.json config 4: DEE-like probability maps (blurred sigmoid noise + ridges), 16 distinct, tiled to n."""
    from synth import prob_map
    base = np.stack([prob_map(H0, W0, seed0 + i) for i in range(min(n, 16))])
    reps = (n + base.shape[0] - 1) // base.shape[0]
    return np.tile(base, (reps, 1, 1))[:n].copy()


# ---------------------------------------------------------------------------
# edge loss (headline)
# ---------------------------------------------------------------------------
def bench_loss(args, rank, world, device, outputs=None):
    import ctypes as C
    from mindtheedge_b200 import _lib
    from mindtheedge_b200.losses import _attrs, _scales_struct, multiscale_edge_loss
    from mindtheedge_b200.targets import prepare_targets

    px_per_step = sum(B_PER_GPU * (H0 >> s) * (W0 >> s) for s in range(SCALES))
    set_bytes = px_per_step * 21  # 3 input planes + 2 output planes fp32 + the 1-byte stash
    n_sets = max(3, int(np.ceil(400e6 / set_bytes)))  # working set >= 400 MB > 126 MB of L2
    sets = [loss_inputs(B_PER_GPU, 1000 * rank + i, device) for i in range(n_sets)]
    weights = [1.0 / SCALES] * SCALES
    at = _attrs(True, True, True, 4.0, 10.0, 1.0)
    stream = torch.cuda.Stream(device)
    fused = hasattr(_lib.lib, "mte_edge_loss_fwd_grad") and not os.environ.get("MTE_BENCH_TWO_KERNEL")
    keep = []
    with torch.cuda.stream(stream):
        st = stream.cuda_stream
        for sc in sets:
            pred = [t[0] for t in sc]; edge = [t[1] for t in sc]; normal = [t[2] for t in sc]
            gmap = [torch.empty_like(e) for e in edge]
            gpred = [torch.empty_like(p) for p in pred]
            stash = [torch.empty(e.shape, dtype=torch.uint8, device=device) for e in edge]
            f = _scales_struct(pred, edge, normal, None, gmap, None, weights, stash)
            b = _scales_struct(pred, edge, normal, None, gmap, gpred, weights, stash)
            losses = torch.zeros(1 + SCALES, device=device)
            ctx = torch.zeros(_lib.lib.mte_edge_loss_ctx_bytes(f, SCALES) // 4, device=device)
            ws = torch.zeros(_lib.lib.mte_edge_loss_workspace_bytes(f, SCALES), dtype=torch.uint8, device=device)
            gl = torch.zeros(1 + SCALES, device=device); gl[0] = 1.0
            keep.append((f, b, gmap, gpred, losses, ctx, ws, gl, stash))

        def launch_fwd(k):
            f, b, _gm, _gp, losses, ctx, ws, gl, _st = k
            _lib.check(_lib.lib.mte_edge_loss_fwd(f, SCALES, C.byref(at), losses.data_ptr(), ctx.data_ptr(),
                                                  ws.data_ptr(), ws.numel(), st))

        def launch_bwd(k):
            f, b, _gm, _gp, losses, ctx, ws, gl, _st = k
            _lib.check(_lib.lib.mte_edge_loss_bwd(b, SCALES, C.byref(at), gl.data_ptr(), ctx.data_ptr(),
                                                  ws.data_ptr(), ws.numel(), st))

        def launch_fused(k):
            # one pass: loss + grad map + d loss / d pred for the expected upstream gradient, then the device-side
            # "rescale only if the actual upstream gradient differs" kernel -- what loss.backward() runs
            f, b, _gm, _gp, losses, ctx, ws, gl, _st = k
            _lib.check(_lib.lib.mte_edge_loss_fwd_grad(b, SCALES, C.byref(at), None, losses.data_ptr(), ctx.data_ptr(),
                                                       ws.data_ptr(), ws.numel(), st))
            _lib.check(_lib.lib.mte_edge_loss_grad_rescale(b, SCALES, gl.data_ptr(), ctx.data_ptr(), None, st))

        def step(k):
            if fused:
                launch_fused(k)
            else:
                launch_fwd(k); launch_bwd(k)

        graphs = []
        for k in keep:
            step(k)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=stream):
                step(k)
            graphs.append(g)
        # one more graph holding a whole round of n_sets consecutive steps: replaying it keeps the GPU fed across steps
        round_graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(round_graph, stream=stream):
            for k in keep:
                step(k)
        for i in range(args.warmup):
            graphs[i % n_sets].replay()
        round_graph.replay()
        sampler = ClockSampler(torch.cuda.current_device())
        if rank == 0:
            sampler.start()
            sampler.settle(round_graph.replay)

        def timed():
            rounds, rest = divmod(args.steps, n_sets)
            for _ in range(rounds):
                round_graph.replay()
            for i in range(rest):
                graphs[i].replay()
        ms, _ = time_region(timed, world, device, stream)
        clocks = sampler.stop() if rank == 0 else None
    if outputs is not None:   # the last timed step ran on set (steps - 1) % n_sets; the kernel split below rewrites it
        _f, _b, gmap, gpred, losses = keep[(args.steps - 1) % n_sets][:5]
        outputs["loss"] = losses.cpu().numpy()   # weighted total, then each scale's loss
        for s in range(SCALES):
            outputs[f"grad_map_s{s}"] = gmap[s].cpu().numpy()
            outputs[f"grad_pred_s{s}"] = gpred[s].cpu().numpy()
    ms_per_step = ms / args.steps
    value = world * px_per_step / (ms_per_step * 1e-3) / 1e6
    loss_value = float(keep[0][4][0].item())

    # per-kernel split: graphs of n_sets back-to-back launches of ONE kernel (rotating input sets)
    def time_kernel(fn):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=stream):
            for k in keep:
                fn(k)
        for _ in range(3):
            g.replay()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 50
        a0.record(stream)
        for _ in range(reps):
            g.replay()
        a1.record(stream)
        torch.cuda.synchronize()
        return a0.elapsed_time(a1) / (reps * n_sets)

    with torch.cuda.stream(stream):
        if fused:
            def only_fused(k):
                f, b, _gm, _gp, losses, ctx, ws, gl, _st = k
                _lib.check(_lib.lib.mte_edge_loss_fwd_grad(b, SCALES, C.byref(at), None, losses.data_ptr(),
                                                           ctx.data_ptr(), ws.data_ptr(), ws.numel(), st))
            split = {"fwd_grad_us": round(time_kernel(only_fused) * 1e3, 2)}
            for k in keep:   # the stash the two-kernel backward reads
                launch_fwd(k)
            split["two_kernel_fwd_us"] = round(time_kernel(launch_fwd) * 1e3, 2)
            split["two_kernel_bwd_us"] = round(time_kernel(launch_bwd) * 1e3, 2)
        else:
            tf, tb = time_kernel(launch_fwd), time_kernel(launch_bwd)
            split = {"fwd_us": round(tf * 1e3, 2), "bwd_us": round(tb * 1e3, 2)}

    # ---- end to end through the public API with HOST buffers in the reference dataloader's encoding: inverse depth
    # fp32 + u8 edge + u8 normal planes (6 B/px) in ONE pinned buffer per step, decoded on the device
    # (targets.prepare_targets), double-buffered against the previous step's compute; loss read back every step
    def staged_u8(seed):
        shapes, n_px, inv, e8, n8 = loss_inputs_u8(B_PER_GPU, seed)
        h = torch.empty(6 * n_px, dtype=torch.uint8).pin_memory()
        h[:4 * n_px].view(torch.float32).copy_(inv)
        h[4 * n_px:5 * n_px].copy_(e8)
        h[5 * n_px:].copy_(n8)
        return shapes, n_px, h

    shapes, n_px, h0 = staged_u8(77 + rank)
    _, _, h1 = staged_u8(177 + rank)
    db = DoubleBuffer([h0, h1], device)
    loss_host = torch.empty(1, dtype=torch.float32).pin_memory()

    def views(dbuf):
        inv_v, e_v, n_v, o = [], [], [], 0
        d_inv = dbuf[:4 * n_px].view(torch.float32)
        for b, h, w in shapes:
            inv_v.append(d_inv[o:o + b * h * w].view(b, 1, h, w))
            e_v.append(dbuf[4 * n_px + o:4 * n_px + o + b * h * w].view(b, h, w))
            n_v.append(dbuf[5 * n_px + o:5 * n_px + o + b * h * w].view(b, h, w))
            o += b * h * w
        return inv_v, e_v, n_v
    dviews = [views(d) for d in db.d]

    def compute_u8(slot, _dbuf):
        inv_v, e_v, n_v = dviews[slot]
        edges, normals = prepare_targets(e_v, n_v)
        inv = [t.requires_grad_(True) for t in inv_v]
        total, _, _ = multiscale_edge_loss(inv, edges, None, normals, weight=10.0, pred_is_inverse=True)
        total.backward()
        loss_host.copy_(total.detach().reshape(1), non_blocking=True)
        for t in inv:
            t.grad = None
            t.requires_grad_(False)

    n_e2e = max(5, min(args.steps, 30))
    db.run(3, compute_u8)
    ms_eager, _ = time_region(lambda: db.run(n_e2e, compute_u8), world, device)
    ms_eager /= n_e2e
    # The eager step above is bound by ~25 Python-level op calls (about 0.8 ms of host time, more than the 0.57 ms the
    # PCIe copy takes), so the headline e2e captures the SAME public-API calls once per staging slot in a CUDA graph
    # (what a training loop that captures its step does) and replays them: the copy then is the only limiter.
    e2e_graphs = []
    side = torch.cuda.Stream(device)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for slot in range(2):
            inv_v, e_v, n_v = dviews[slot]

            def captured(inv_v=inv_v, e_v=e_v, n_v=n_v):
                edges, normals = prepare_targets(e_v, n_v)
                inv = [t.detach().requires_grad_(True) for t in inv_v]
                total, _, _ = multiscale_edge_loss(inv, edges, None, normals, weight=10.0, pred_is_inverse=True)
                grads = torch.autograd.grad(total, inv)
                loss_host.copy_(total.detach().reshape(1), non_blocking=True)
                return grads
            for _ in range(2):
                captured()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                keep_grads = captured()
            e2e_graphs.append((g, keep_grads))
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()

    def compute_graph(slot, _dbuf):
        e2e_graphs[slot][0].replay()

    db.run(3, compute_graph)
    ms_e2e, _ = time_region(lambda: db.run(n_e2e, compute_graph), world, device)
    ms_e2e /= n_e2e
    e2e_value = world * px_per_step / (ms_e2e * 1e-3) / 1e6

    # the same with all three planes shipped as fp32 (12 B/px), the layout of the tensors the reference head receives
    planes = [loss_inputs(B_PER_GPU, 5000 + 1000 * rank + i, None) for i in range(2)]
    n32 = sum(t.numel() for sc in planes[0] for t in sc)
    hb = []
    for pl in planes:
        h = torch.empty(n32, dtype=torch.float32).pin_memory()
        o = 0
        for sc in pl:
            for t in sc:
                h[o:o + t.numel()].copy_(t.reshape(-1)); o += t.numel()
        hb.append(h)
    db32 = DoubleBuffer(hb, device)

    def views32(dbuf):
        out, o = [], 0
        for sc in planes[0]:
            vs = []
            for t in sc:
                vs.append(dbuf[o:o + t.numel()].view(t.shape)); o += t.numel()
            out.append(tuple(vs))
        return out
    dv32 = [views32(d) for d in db32.d]

    def compute_f32(slot, _dbuf):
        sc = dv32[slot]
        inv = [s[0].requires_grad_(True) for s in sc]
        total, _, _ = multiscale_edge_loss(inv, [s[1] for s in sc], None, [s[2] for s in sc], weight=10.0,
                                           pred_is_inverse=True)
        total.backward()
        loss_host.copy_(total.detach().reshape(1), non_blocking=True)
        for t in inv:
            t.grad = None
            t.requires_grad_(False)

    db32.run(3, compute_f32)
    ms_f32, _ = time_region(lambda: db32.run(n_e2e, compute_f32), world, device)
    ms_f32 /= n_e2e
    h2d_gbs = h2d_probe(world, device)

    peak, peak_src = measured_peak_gbs()
    achieved = LOSS_BYTES_PER_PX * px_per_step / (ms_per_step * 1e-3) / 1e9
    kernels = ("edge_loss_fused_kernel (loss + grad map + d loss/d pred in one pass) + edge_loss_rescale_kernel "
               "(exits at once when the upstream gradient is the expected one)") if fused else \
        "edge_loss_fwd_kernel + edge_loss_bwd_ring_kernel"
    out = {
        "metric": "edge_loss_fwd_bwd_throughput", "value": round(value, 1), "unit": "Mpixel/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_per_step, 5),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "edge loss fwd+bwd, batch 8/GPU x 4-scale pyramid 384x1280..48x160 fp32, DEE normals, "
                               "no mask, inv2depth fused (BASELINE.json config 3 loss shape)",
                   "pixels_per_step_per_gpu": px_per_step, "l2_policy": f"rotating {n_sets} input sets "
                   f"({n_sets * set_bytes / 1e6:.0f} MB > L2)",
                   "launch": f"CUDA graph replay, {n_sets} steps x 2 kernels per graph",
                   "parallelism": f"dp{world} (batch-sharded, no data-path collective in the loss)"},
        "e2e": {"value": round(e2e_value, 1), "unit": "Mpixel/s", "h2d_bytes_per_step": 6 * n_px,
                "d2h_bytes_per_step": 4, "ms_per_step": round(ms_e2e, 4),
                "api": "targets.prepare_targets (u8 edge / normal planes as the reference dataloader holds them, "
                       "gta_dataset.py:406-422, decoded on the device) + losses.multiscale_edge_loss + autograd.grad, "
                       "captured once per staging slot with torch.cuda.graph and replayed; H2D double-buffered on a "
                       "copy stream, loss copied back every step", "h2d_probe_gbs": h2d_gbs,
                "eager_ms_per_step": round(ms_eager, 4),
                "eager_value": round(world * px_per_step / (ms_eager * 1e-3) / 1e6, 1)},
        "e2e_f32_targets": {"value": round(world * px_per_step / (ms_f32 * 1e-3) / 1e6, 1), "unit": "Mpixel/s",
                            "h2d_bytes_per_step": n32 * 4, "d2h_bytes_per_step": 4, "ms_per_step": round(ms_f32, 4),
                            "api": "losses.multiscale_edge_loss + backward on fp32 host planes (12 B/px)"},
        "gpu_launches": 2 * args.steps,
        "roofline": {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                     "frac": round(achieved / peak, 4), "traffic": recorded_traffic("edge_loss_fwd_bwd"),
                     "kernel": kernels, **split,
                     "algorithmic_bytes_per_px": LOSS_BYTES_PER_PX, "peak_source": peak_src},
        "loss_value": loss_value,
        "clocks": clocks,
    }
    return out


# ---------------------------------------------------------------------------
# AUC evaluation (KITTI-DE wiring; DDAD-size variant)
# ---------------------------------------------------------------------------
def _auc_of(counts):
    from mindtheedge_b200.eval_depth_edges import compute_rec_prec_f1, mean_recall_at_precision_range
    cn = counts.cpu().numpy().astype(np.float64)
    rec, prec, _ = compute_rec_prec_f1(cn[:, 0], cn[:, 1], cn[:, 2], cn[:, 3])
    return float(mean_recall_at_precision_range(np.vstack((prec, rec)).transpose()))


def bench_auc(args, rank, world, device, steps=None, warmup=None, ddad=False):
    from mindtheedge_b200.eval_depth_edges import sweep_counts
    import torch.distributed as dist
    steps = steps or args.steps
    warmup = warmup if warmup is not None else args.warmup
    rng = list(range(20, 241, 20))
    seed = int(os.environ.get("MTE_BENCH_SEED", "7000"))
    if ddad:
        n_img, H, W = DDAD_N, DDAD_H, DDAD_W
        crop = KITTI_CROP   # the reference applies its default crop to every dataset (SURVEY.md Appendix B #10)
        depths, gts = ddad_like_set(n_img, 300 + 1000 * rank)
    else:
        n_img, H, W, crop = KITTI_N, H0, W0, KITTI_CROP
        # weak scaling: every rank evaluates its own set of 102 images (different synthetic depth per rank)
        depths, gts = kitti_like_set(n_img, seed + 1000 * rank)
    d_dev, g_dev = torch.from_numpy(depths).to(device), torch.from_numpy(gts).to(device)
    px_per_step = world * n_img * KITTI_T * H * W  # whole job

    def step(d=d_dev, g=g_dev, c=crop):
        cc = sweep_counts(d, g, rng, c, 0.0, 80.0, max_dist=0.002)
        if world > 1:
            dist.all_reduce(cc, op=dist.ReduceOp.SUM)
        return cc

    for _ in range(warmup):
        step()
    sampler = ClockSampler(torch.cuda.current_device())
    if rank == 0:
        sampler.start()
        sampler.settle(lambda: sweep_counts(d_dev, g_dev, rng, crop, 0.0, 80.0, max_dist=0.002))

    def timed():
        for _ in range(steps):
            c = step()
        return c
    ms, counts = time_region(timed, world, device)
    clocks = sampler.stop() if rank == 0 else None
    ms /= steps
    value = px_per_step / (ms * 1e-3) / 1e6

    # ---- strong scaling + rank-count independence on hardware: the SAME n_img images (rank 0's set) sharded
    # i -> rank i mod R, one all-reduce; the summed counts must equal the single-rank counts of the whole set
    strong = None
    if world > 1:
        d0, g0 = (kitti_like_set(n_img, seed) if not ddad else ddad_like_set(n_img, 300))
        mine = list(range(rank, n_img, world))
        ds, gs = torch.from_numpy(d0[mine]).to(device), torch.from_numpy(g0[mine]).to(device)
        for _ in range(2):
            step(ds, gs)
        ms_s, c_sharded = time_region(lambda: [step(ds, gs) for _ in range(steps)][-1], world, device)
        ms_s /= steps
        same = None
        if rank == 0:
            c_single = sweep_counts(torch.from_numpy(d0).to(device), torch.from_numpy(g0).to(device), rng, crop, 0.0,
                                    80.0, max_dist=0.002)
            same = bool(torch.equal(c_single, c_sharded))
        strong = {"value": round(n_img * KITTI_T * H * W / (ms_s * 1e-3) / 1e6, 1), "unit": "Mpixel/s",
                  "ms_per_step": round(ms_s, 4), "scaling": "strong",
                  "images_total": n_img, "counts_equal_single_rank": same}

    # ---- e2e: host depth + GT in (pinned, double-buffered), counts -> P/R vectors + AUC out on the host
    hb = []
    for k in range(2):
        h = torch.empty(depths.nbytes + gts.nbytes, dtype=torch.uint8).pin_memory()
        h[:depths.nbytes].copy_(torch.from_numpy(depths).view(torch.uint8).reshape(-1))
        h[depths.nbytes:].copy_(torch.from_numpy(gts).reshape(-1))
        hb.append(h)
    db = DoubleBuffer(hb, device)
    aucs = []
    counts_host = torch.empty((len(rng), 4), dtype=torch.int64).pin_memory()

    def compute(slot, dbuf):
        dd = dbuf[:depths.nbytes].view(torch.float32).view(depths.shape)
        gd = dbuf[depths.nbytes:].view(gts.shape)
        cc = step(dd, gd)
        counts_host.copy_(cc, non_blocking=True)

    def e2e_run(n):
        db.run(n, compute)
        torch.cuda.current_stream().synchronize()
        return _auc_of(counts_host)

    e2e_run(2)
    n_e2e = max(2, min(steps, 5))
    ms_e2e, auc = time_region(lambda: e2e_run(n_e2e), world, device)
    ms_e2e /= n_e2e
    h2d_gbs = h2d_probe(world, device)
    peak, peak_src = measured_peak_gbs()
    achieved = AUC_BYTES_PER_PX * px_per_step / world / (ms * 1e-3) / 1e9
    name = "DDAD-DE" if ddad else "KITTI-DE"
    wl = (f"DDAD-size depth-edge AUC eval (BASELINE.json config 5): per GPU {n_img} synthetic {H}x{W} images, 12 Canny "
          f"settings (t/2,t) t=20..240, the reference's default crop [153:371,44:1197] (applied to every dataset, "
          f"eval_depth_edges.py:235), max_dist 0.002, exact matcher; pixel = image x threshold x H x W") if ddad else \
         ("KITTI-DE depth-edge AUC eval (BASELINE.json config 2, shipped wiring): per GPU the 102 bundled "
          "KITTI-DE GT edge maps vs synthetic 384x1280 predicted depth, 12 Canny settings (t/2,t) t=20..240, crop "
          "[153:371,44:1197], max_dist 0.002, exact matcher; pixel = image x threshold x H x W")
    out = {
        "metric": "auc_eval_throughput", "value": round(value, 1), "unit": "Mpixel/s", "ms_per_step": round(ms, 4),
        "steps": steps, "scaling": "weak",
        "config": {"workload": wl,
                   "l2_policy": f"inputs {depths.nbytes / 1e6:.0f} MB + per-CTA matcher arenas > L2",
                   "parallelism": f"images sharded over {world} rank(s) ({n_img} each), one int64[12,4] all-reduce"},
        "e2e": {"value": round(px_per_step / (ms_e2e * 1e-3) / 1e6, 1), "unit": "Mpixel/s",
                "h2d_bytes_per_step": int(depths.nbytes + gts.nbytes), "d2h_bytes_per_step": 12 * 4 * 8,
                "ms_per_step": round(ms_e2e, 3), "auc": round(float(auc), 6), "h2d_probe_gbs": h2d_gbs,
                "api": "eval_depth_edges.sweep_counts (mte::canny_from_depth + mte::pr_counts) on pinned host planes, "
                       "H2D double-buffered on a copy stream, counts -> compute_rec_prec_f1 -> AUC on the host"},
        "counts": counts.cpu().numpy().tolist(),
        # canny_lut, canny_nms, canny_uf_hyst_smem, canny_uf_hyst (overflow images, exits at once when there are none),
        # match_sweep, match (overflow problems, likewise)
        "gpu_launches_per_step": 6,
        "roofline": {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                     "frac": round(achieved / peak, 4),
                     "traffic": recorded_traffic("ddad_eval" if ddad else "auc_eval"),
                     "kernel": "match_sweep_kernel (dominant) + canny_uf_hyst_smem_kernel + canny_nms_kernel",
                     "algorithmic_bytes_per_px": AUC_BYTES_PER_PX, "peak_source": peak_src,
                     "note": "matcher and hysteresis are latency-bound graph work in shared memory: the step lasts as "
                             "long as its slowest image, it is not an HBM stream"},
        "clocks": clocks,
    }
    if strong:
        out["strong_scaling"] = strong
    if ddad:
        # the same set without any crop (SURVEY.md 8d "crop scaled or disabled"): radius 4.57 px, ~25 k + 25 k vertices
        # per window
        n_unc = 2
        du, gu = d_dev[:n_unc], g_dev[:n_unc]
        sweep_counts(du, gu, rng, None, 0.0, 80.0, max_dist=0.002)
        ms_u, cu = time_region(lambda: sweep_counts(du, gu, rng, None, 0.0, 80.0, max_dist=0.002), 1, device)
        out["uncropped"] = {"images": n_unc, "ms": round(ms_u, 3),
                            "value": round(n_unc * KITTI_T * H * W / (ms_u * 1e-3) / 1e6, 1), "unit": "Mpixel/s",
                            "counts_t0": cu.cpu().numpy()[0].tolist()}
    return out


# ---------------------------------------------------------------------------
# DEE annotation post-process (config 4)
# ---------------------------------------------------------------------------
def bench_dee(args, rank, world, device, outputs=None):
    from mindtheedge_b200.tools import dee_postprocess
    n = DEE_FRAMES
    frames = dee_frames(n, 100 + 1000 * rank)      # frame i of the job -> rank i mod R: every rank has its own frames
    p_dev = torch.from_numpy(frames).to(device)
    px = n * H0 * W0

    def step(p=p_dev):
        return dee_postprocess(p, out_dtype=torch.float32)

    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(torch.cuda.current_device())
    if rank == 0:
        sampler.start()
        sampler.settle(step)
    def timed():
        for _ in range(args.steps - 1):   # outputs are dropped at once: the allocator reuses the same blocks every step
            step()
        return step()
    ms, (nrm_last, edges_last) = time_region(timed, world, device)
    clocks = sampler.stop() if rank == 0 else None
    if outputs is not None:
        outputs["normals"] = nrm_last.cpu().numpy()
        outputs["edges"] = edges_last.cpu().numpy()
    del nrm_last, edges_last
    ms /= args.steps
    value = world * px / (ms * 1e-3) / 1e6
    parts = {}
    for name, kw in (("normals_only", {"nms": False, "hysteresis": False}), ("normals_nms", {"hysteresis": False})):
        for _ in range(3):
            dee_postprocess(p_dev, out_dtype=torch.float32, **kw)
        torch.cuda.synchronize()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(10):
            dee_postprocess(p_dev, out_dtype=torch.float32, **kw)
        a1.record()
        torch.cuda.synchronize()
        parts[name + "_ms"] = round(a0.elapsed_time(a1) / 10, 4)

    # e2e: prob maps from pinned host memory, normals u8 + edges fp32 back to pinned host memory, every step
    hb = [torch.from_numpy(frames).pin_memory(), torch.from_numpy(frames.copy()).pin_memory()]
    db = DoubleBuffer(hb, device)
    nrm_h = torch.empty((n, H0, W0), dtype=torch.uint8).pin_memory()
    edg_h = torch.empty((n, H0, W0), dtype=torch.float32).pin_memory()

    def compute(slot, dbuf):
        # the results go back on the compute stream: PCIe already runs both directions (the next step's H2D is on the
        # copy stream); a third stream for the D2H was measured slower (9.3 vs 8.6 ms: 70 GB/s combined is the host's limit)
        nrm, out = dee_postprocess(dbuf, out_dtype=torch.float32)
        nrm_h.copy_(nrm, non_blocking=True)
        edg_h.copy_(out, non_blocking=True)

    db.run(2, compute)
    n_e2e = max(2, min(args.steps, 10))
    ms_e2e, _ = time_region(lambda: db.run(n_e2e, compute), world, device)
    ms_e2e /= n_e2e
    peak, peak_src = measured_peak_gbs()
    achieved = DEE_BYTES_PER_PX * px / (ms * 1e-3) / 1e9
    return {
        "metric": "dee_postprocess_throughput", "value": round(value, 1), "unit": "Mpixel/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 4), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"DEE annotation post-process (BASELINE.json config 4): {n} KITTI-size (384x1280) "
                               "probability maps per GPU per step -> u8 edge normals (Sobel5 + atan2) + NMS + "
                               "hysteresis(0.3, 0.7) edges; frames sharded over ranks, no collective",
                   "l2_policy": f"inputs + outputs {n * H0 * W0 * 9 / 1e6:.0f} MB > L2",
                   "parallelism": f"frame-sharded over {world} rank(s), no collective"},
        "e2e": {"value": round(world * px / (ms_e2e * 1e-3) / 1e6, 1), "unit": "Mpixel/s",
                "h2d_bytes_per_step": int(frames.nbytes), "d2h_bytes_per_step": int(n * H0 * W0 * 5),
                "ms_per_step": round(ms_e2e, 3),
                "api": "tools.dee_postprocess (mte::dee_postprocess) on pinned host frames, H2D double-buffered on a copy "
                       "stream, normals u8 + edges fp32 copied back"},
        "gpu_launches": 5 * args.steps,   # tables, front, hysteresis (+ its empty fallback), finish
        "roofline": {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                     "frac": round(achieved / peak, 4), "traffic": recorded_traffic("dee_postprocess"),
                     "kernel": "dee_front_tma_kernel (Sobel5 + normals + NMS + labels; dominant) + canny_uf_hyst_smem_kernel "
                               "(hysteresis flood) + dee_finish_kernel (img * labels / max)",
                     "algorithmic_bytes_per_px": DEE_BYTES_PER_PX, "peak_source": peak_src, **parts},
        "clocks": clocks,
    }


# ---------------------------------------------------------------------------
# config 3: train step (stock trunk under DDP + this loss)
# ---------------------------------------------------------------------------
def make_trunk():
    """A small stock-PyTorch encoder/decoder emitting 4 inverse-depth scales (full, 1/2, 1/4, 1/8 resolution), in the
    shape of the PackNet heads (conv + sigmoid / min_depth, networks/layers/packnet/layers01.py InvDepth).  Random
    init; only stock cuDNN ops -- the trunk is out of scope, it is here so that DDP has gradient buckets to all-reduce
    while the edge loss runs in its real position."""
    import torch.nn as nn

    class Block(nn.Module):
        def __init__(self, ci, co, stride):
            super().__init__()
            self.c = nn.Conv2d(ci, co, 3, stride, 1)
            self.g = nn.GroupNorm(8, co)
            self.a = nn.ELU(inplace=True)

        def forward(self, x):
            return self.a(self.g(self.c(x)))

    class Trunk(nn.Module):
        def __init__(self):
            super().__init__()
            self.e0 = Block(3, 16, 1)
            self.e1 = Block(16, 32, 2)
            self.e2 = Block(32, 64, 2)
            self.e3 = Block(64, 128, 2)
            self.d2 = Block(128 + 64, 64, 1)
            self.d1 = Block(64 + 32, 32, 1)
            self.d0 = Block(32 + 16, 16, 1)
            self.h = nn.ModuleList([nn.Conv2d(c, 1, 3, 1, 1) for c in (16, 32, 64, 128)])
            self.up = nn.Upsample(scale_factor=2, mode="nearest")

        def forward(self, rgb):
            x0 = self.e0(rgb); x1 = self.e1(x0); x2 = self.e2(x1); x3 = self.e3(x2)
            y2 = self.d2(torch.cat([self.up(x3), x2], 1))
            y1 = self.d1(torch.cat([self.up(y2), x1], 1))
            y0 = self.d0(torch.cat([self.up(y1), x0], 1))
            feats = (y0, y1, y2, x3)
            return [torch.sigmoid(h(f)) / 0.5 for h, f in zip(self.h, feats)]   # inverse depth in (0, 2)

    return Trunk()


def bench_train(args, rank, world, device, outputs=None):
    """models/SemiSupEdgeModel.py:98-162 in miniature: trunk -> 4 inverse-depth scales -> edge loss over all scales
    (compute_edge_loss_with_all_scales :164-198: inv2depth, GradLoss per scale, sum, / 4) -> backward -> optimizer
    step (trainers/common_trainer.py:111-143); DDP all-reduces the trunk's gradient buckets over NCCL."""
    from mindtheedge_b200.losses import multiscale_edge_loss
    from oracle.edge_loss import edge_loss_torch   # the eager baseline arm only
    from torch.nn.parallel import DistributedDataParallel as DDP
    torch.manual_seed(0)
    trunk = make_trunk().to(device)
    model = DDP(trunk, device_ids=[device.index]) if world > 1 else trunk
    opt = torch.optim.SGD(model.parameters(), lr=1e-4, momentum=0.9)
    B = B_PER_GPU
    g = torch.Generator().manual_seed(100 + rank)
    rgb = torch.rand(B, 3, H0, W0, generator=g).to(device)
    tg = loss_inputs(B, 200 + rank, device)
    edges, normals = [t[1] for t in tg], [t[2] for t in tg]
    px_per_step = sum(B * (H0 >> s) * (W0 >> s) for s in range(SCALES))

    def loss_mte(inv):
        total, _, _ = multiscale_edge_loss(inv, edges, None, normals, weight=10.0, pred_is_inverse=True)
        return total

    def loss_eager(inv):
        total = 0
        for s in range(SCALES):
            depth = 1.0 / inv[s].clamp(min=1e-6)
            l, _ = edge_loss_torch(depth, edges[s], None, True, True, 4, normals[s], weight=10.0)
            total = total + l
        return total / SCALES

    def step(loss_fn, ev=None):
        opt.zero_grad(set_to_none=True)
        inv = model(rgb)
        if ev:
            ev[0].record()
        loss = loss_fn(inv)
        if ev:
            ev[1].record()
        loss.backward()
        opt.step()
        return loss

    # gradient parity of the two arms on the same parameters (no optimizer step)
    def grads(loss_fn):
        opt.zero_grad(set_to_none=True)
        loss_fn(model(rgb)).backward()
        return torch.cat([p.grad.reshape(-1) for p in model.parameters()]), None
    ga, _ = grads(loss_mte)
    gb, _ = grads(loss_eager)
    grad_rel = float((ga - gb).abs().max() / gb.abs().max())
    opt.zero_grad(set_to_none=True)

    res = {}
    for name, fn in (("mte", loss_mte), ("eager", loss_eager)):
        for _ in range(max(3, args.warmup)):
            step(fn)
        steps = args.steps if name == "mte" else max(3, min(args.steps, 20))   # the eager arm is a side number
        sampler = ClockSampler(torch.cuda.current_device())
        if rank == 0 and name == "mte":
            sampler.start()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        ms, last = time_region(lambda: [step(fn, ev[i]) for i in range(steps)][-1], world, device)
        if rank == 0 and name == "mte":
            res["clocks"] = sampler.stop()
        if outputs is not None and name == "mte":
            outputs["loss"] = last.detach().cpu().numpy().reshape(1)
            outputs["trunk_params"] = torch.cat([p.detach().reshape(-1) for p in trunk.parameters()]).cpu().numpy()
        res[name] = {"ms_per_step": round(ms / steps, 3), "steps": steps,
                     "loss_fwd_ms": round(float(np.median([a.elapsed_time(b) for a, b in ev])), 4),
                     "loss": float(last.item())}
    ms_step = res["mte"]["ms_per_step"]
    value = world * px_per_step / (ms_step * 1e-3) / 1e6
    n_par = sum(p.numel() for p in trunk.parameters())
    return {
        "metric": "train_step_throughput", "value": round(value, 1), "unit": "Mpixel/s", "n_gpus": world,
        "steps": res["mte"]["steps"], "warmup": max(3, args.warmup), "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "train step (BASELINE.json config 3): stock conv trunk (random init, 4 inverse-depth "
                               "scales) + edge loss over all scales + backward + SGD step, batch 8/GPU 384x1280 fp32; "
                               "pixel = loss pixel (5.22 Mpx per GPU per step)",
                   "trunk_parameters": n_par, "l2_policy": "activations of the step >> L2",
                   "parallelism": f"DistributedDataParallel over {world} rank(s): NCCL all-reduce of the trunk's "
                                  "gradient buckets, no collective in the loss"},
        "with_mte_loss": res["mte"], "with_eager_loss": res["eager"],
        "step_speedup_vs_eager_loss": round(res["eager"]["ms_per_step"] / ms_step, 3),
        "grad_max_rel_diff_vs_eager_loss": grad_rel,
        "e2e": {"value": round(value, 1), "unit": "Mpixel/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "note": "inputs resident (the trunk dominates the step); see the loss workload for host-buffer e2e"},
        "gpu_launches": 3 * res["mte"]["steps"],
        "clocks": res.get("clocks"),
    }


# ---------------------------------------------------------------------------
# CPU reference arm: the reference's own code from oracle/_ref (staged by oracle/make_ref.py), else the oracle port
# ---------------------------------------------------------------------------
def _write_eval_files(tmp, depths, gts):
    import cv2
    gl, pl = [], []
    for i in range(len(depths)):
        gp, dp = os.path.join(tmp, f"gt{i:04d}.png"), os.path.join(tmp, f"pred{i:04d}.npy")
        cv2.imwrite(gp, gts[i] * 255)
        np.save(dp, depths[i])
        gl.append(gp)
        pl.append(dp)
    return gl, pl


def _dee_ref_frame(args_):
    tools_path, frame = args_
    import importlib.util
    spec = importlib.util.spec_from_file_location("ref_tools_worker", tools_path)
    tools = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(tools)
    import cv2
    sx = cv2.Sobel(frame, cv2.CV_64F, 1, 0, ksize=5)
    sy = cv2.Sobel(frame, cv2.CV_64F, 0, 1, ksize=5)
    ang = (((np.arctan2(-sy, sx) * (180 / np.pi) + 180) / 360) * 255).astype("uint8")   # infer_edge_estimation.py:244-250
    out = tools.hysteresis(tools.non_max_suppression(frame))
    return int(ang.sum()) + int(out.sum() > 0)


def _dee_port_frame(frame):
    from oracle import dee as odee
    return int(odee.normals_u8(frame).sum()) + int(odee.hysteresis(odee.non_max_suppression(frame)).sum() > 0)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import ref_loader
    cores = os.cpu_count() or 1
    have_ref = ref_loader.available()
    kind = "reference" if have_ref else "port"
    steps = max(1, args.steps)
    warm = max(1, min(args.warmup, 3))
    base = {"impl": "reference", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "data": "synthetic"}

    if args.workload in ("loss", "train"):
        torch.set_num_threads(cores)
        B = B_PER_GPU
        data = loss_inputs(B, 1000, None)
        px = sum(B * (H0 >> s) * (W0 >> s) for s in range(SCALES))
        if have_ref:
            import warnings
            warnings.filterwarnings("ignore")
            head = ref_loader.load_gradloss_cpu()("cross_entropy", True, [], 10.0, 1.0)
            what = ("UNMODIFIED reference GradLoss (oracle/_ref: losses/grad_loss.py) on CPU torch, the per-scale loop of "
                    "SemiSupEdgeModel.py:164-198 incl. inv2depth")
        else:
            from oracle.edge_loss import edge_loss_torch
            head = lambda d, e, m, ig, isg, t, n: edge_loss_torch(d, e, m, ig, isg, t, n, weight=10.0)  # noqa: E731
            what = "oracle port of GradLoss (oracle/edge_loss.py) on CPU torch"

        def step():
            total = 0
            for inv, edge, normal in data:
                x = inv.clone().requires_grad_(True)
                depth = 1.0 / x.clamp(min=1e-6)
                l, _ = head(depth, edge, None, True, True, 4, normal)
                total = total + l
            (total / SCALES).backward()

        n_t = min(steps, 20)
        for _ in range(warm):
            step()
        t0 = time.perf_counter()
        for _ in range(n_t):
            step()
        dt = (time.perf_counter() - t0) / n_t
        v = px / dt / 1e6
        line = dict(base, metric="edge_loss_fwd_bwd_throughput", value=round(v, 3), unit="Mpixel/s",
                    ms_per_step=round(dt * 1e3, 2), dtype="f32",
                    config={"workload": "edge loss fwd+bwd, batch 8 x 4-scale pyramid 384x1280..48x160 fp32, DEE "
                                        "normals, no mask (BASELINE.json config 3 loss shape) -- the same batch as the "
                                        "GPU arm; " + what, "pixels_per_step_per_gpu": px},
                    cpu_baseline={"value": round(v, 3), "unit": "Mpixel/s", "cores": cores, "kind": kind,
                                  "sample": f"batch {B} x 4 scales ({px / 1e6:.2f} Mpx) per step, {n_t} timed steps, "
                                            f"torch CPU {torch.get_num_threads()} threads"})
    elif args.workload in ("auc", "ddad"):
        ddad = args.workload == "ddad"
        n_img = 16 if not ddad else 4
        depths, gts = (ddad_like_set(n_img, 300) if ddad else kitti_like_set(n_img, 7000))
        H, W = depths.shape[1:]
        workers = min(cores, n_img)
        px = n_img * KITTI_T * H * W
        with tempfile.TemporaryDirectory() as tmp:
            gl, pl = _write_eval_files(tmp, depths, gts)
            if have_ref:
                ede = ref_loader.load_eval_depth_edges()
                what = (f"UNMODIFIED reference pr_evaluation (oracle/_ref: eval_depth_edges.py + edge.py, files + JPEG "
                        f"round trip, Pool({workers}); reference default is 4) with the oracle's C matcher standing "
                        f"in for py-bsds500")

                def run():
                    import contextlib
                    import io
                    with contextlib.redirect_stdout(io.StringIO()):
                        return ede.pr_evaluation(gl, pl, save_folder=os.path.join(tmp, "out"), num_workers=workers)
            else:
                from oracle import pr_counts as opr
                what = "oracle port of pr_evaluation (NumPy Canny + C Hopcroft-Karp), single core"
                workers = 1

                def run():
                    return opr.pr_sweep_counts(list(depths), [g * 255 for g in gts], gt_crop=tuple(KITTI_CROP))
            n_t = max(1, min(steps, 3))
            run()
            t0 = time.perf_counter()
            for _ in range(n_t):
                run()
            dt = (time.perf_counter() - t0) / n_t
        v = px / dt / 1e6
        line = dict(base, metric="auc_eval_throughput", value=round(v, 3), unit="Mpixel/s",
                    ms_per_step=round(dt * 1e3, 2), dtype="u8",
                    config={"workload": f"{'DDAD-size' if ddad else 'KITTI-DE'} depth-edge AUC eval, {n_img} images x 12 "
                                        f"Canny settings per step (bounded sample of the GPU arm's set); " + what},
                    cpu_baseline={"value": round(v, 3), "unit": "Mpixel/s", "cores": workers, "kind": kind,
                                  "sample": f"{n_img} images x 12 settings per step, {n_t} timed steps of {dt:.1f} s"})
    else:  # dee
        import multiprocessing as mp
        n_fr = min(cores, 16)
        frames = dee_frames(n_fr, 100)
        px = n_fr * H0 * W0
        if have_ref:
            tools_path = os.path.join(ROOT, "oracle", "_ref", "packnet_code", "packnet_sfm", "utils", "tools.py")
            jobs, fn = [(tools_path, f) for f in frames], _dee_ref_frame
            what = ("UNMODIFIED reference tools.non_max_suppression + hysteresis (oracle/_ref) + the normals block of "
                    f"infer_edge_estimation.py:244-250, one frame per process, Pool({n_fr}); the reference runs frames "
                    "sequentially in one process")
        else:
            jobs, fn = list(frames), _dee_port_frame
            what = f"oracle port (vectorised NumPy restatement), Pool({n_fr})"
        with mp.Pool(n_fr) as pool:
            t0 = time.perf_counter()
            pool.map(fn, jobs)
            dt = time.perf_counter() - t0
        v = px / dt / 1e6
        line = dict(base, metric="dee_postprocess_throughput", value=round(v, 3), unit="Mpixel/s",
                    ms_per_step=round(dt * 1e3, 2), dtype="f64",
                    config={"workload": f"DEE annotation post-process, {n_fr} KITTI-size frames per step (bounded sample); "
                                        + what},
                    cpu_baseline={"value": round(v, 3), "unit": "Mpixel/s", "cores": n_fr, "kind": kind,
                                  "sample": f"{n_fr} frames, one pass of {dt:.1f} s"})
    line["e2e"] = {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    print(json.dumps(line), flush=True)


def cpu_baseline_subprocess(workload, steps=3, warmup=1, timeout=900):
    """Run the CPU arm in a process of its own (its `.cuda()` shim is process-global) and return its cpu_baseline."""
    try:
        env = dict(os.environ)
        for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT", "CUDA_VISIBLE_DEVICES"):
            env.pop(k, None)
        env["CUDA_VISIBLE_DEVICES"] = ""
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", workload,
                            "--steps", str(steps), "--warmup", str(warmup)], capture_output=True, text=True,
                           timeout=timeout, env=env)
        for l in reversed(r.stdout.strip().splitlines()):
            if l.startswith("{"):
                return json.loads(l)["cpu_baseline"]
        return {"value": None, "error": (r.stderr or "no output")[-300:]}
    except Exception as exc:  # noqa: BLE001
        return {"value": None, "error": repr(exc)[:300]}


def eager_gpu_loss_baseline(device, iters=10, warm=3):
    """The reference's algorithm as plain eager PyTorch ON THE GPU (oracle port of GradLoss + autograd, the per-scale
    loop of SemiSupEdgeModel.py:164-198, inv2depth included) at the headline shape: the like-for-like GPU baseline
    SURVEY.md 8(d) asks for next to the CPU one.  Reported only; nothing of it is on the product path."""
    from oracle.edge_loss import edge_loss_torch
    data = loss_inputs(B_PER_GPU, 4242, device)
    px = sum(B_PER_GPU * (H0 >> s) * (W0 >> s) for s in range(SCALES))

    def step():
        total = 0
        for inv, edge, normal in data:
            x = inv.clone().requires_grad_(True)
            depth = 1.0 / x.clamp(min=1e-6)
            l, _ = edge_loss_torch(depth, edge, None, True, True, 4, normal, weight=10.0)
            total = total + l
        (total / SCALES).backward()

    for _ in range(warm):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    return px / (ms * 1e-3) / 1e6, ms


# ---------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5000)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="mte", choices=["mte", "reference"])
    ap.add_argument("--workload", default="loss", choices=["loss", "auc", "dee", "ddad", "train"])
    ap.add_argument("--no-secondary", action="store_true", help="skip the second workload and the CPU baselines")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32/float64, <= 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl mte)")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: mindtheedge_b200 has no CPU path (use --impl reference for the CPU arm)")
    rank, world, local = dist_setup(args.gpus)
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    host_cores = bind_to_gpu_cores(local, world)
    from mindtheedge_b200 import _lib  # noqa: F401  (fails at once when libmte.so has not been built)
    outputs = {} if args.dump_outputs and rank == 0 else None

    def finish_auc(a):
        return {"metric": a["metric"], "value": a["value"], "unit": a["unit"], "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": a["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": a["config"], "e2e": a["e2e"],
                "gpu_launches": a["gpu_launches_per_step"] * args.steps, "roofline": a["roofline"],
                "counts": a["counts"], "clocks": a["clocks"],
                **({"strong_scaling": a["strong_scaling"]} if "strong_scaling" in a else {}),
                **({"uncropped": a["uncropped"]} if "uncropped" in a else {})}

    if args.workload == "loss":
        line = bench_loss(args, rank, world, device, outputs)
        if not args.no_secondary:
            a = bench_auc(args, rank, world, device, steps=max(2, min(args.steps, 5)), warmup=3)
            a.pop("clocks", None)
            line["auc_eval"] = a
            if outputs is not None:
                outputs["auc_eval_counts"] = np.array(a["counts"])
    elif args.workload in ("auc", "ddad"):
        line = finish_auc(bench_auc(args, rank, world, device, ddad=args.workload == "ddad"))
        if outputs is not None:
            outputs["counts"] = np.array(line["counts"])
    elif args.workload == "dee":
        line = bench_dee(args, rank, world, device, outputs)
    else:
        line = bench_train(args, rank, world, device, outputs)
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    line["host_cores_bound"] = host_cores
    if rank == 0 and not args.no_secondary:
        line["cpu_baseline"] = cpu_baseline_subprocess(args.workload)
        if args.workload == "loss":
            ve, mse = eager_gpu_loss_baseline(device)
            line["eager_gpu_baseline"] = {"value": round(ve, 1), "unit": "Mpixel/s", "ms_per_step": round(mse, 3),
                                          "kind": "port", "sample": "oracle port of GradLoss (eager PyTorch ops + autograd) "
                                          "on the same B200, same shape as the headline, 10 timed steps"}
            if "auc_eval" in line:
                line["auc_eval"]["cpu_baseline"] = cpu_baseline_subprocess("auc", steps=1)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
