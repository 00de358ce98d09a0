"""CPU suite, part 2: the C ABI surface, the host-side logic and the multi-rank reduction
(gloo, world_size 2).  No kernel is launched here."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import GOLDEN, ROOT


def _declared_symbols():
    hdr = open(os.path.join(ROOT, "include", "mte.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return sorted(set(re.findall(r"\b(mte_[a-z0-9_]+)\s*\(", hdr)))


def test_library_exports_every_declared_symbol():
    from mindtheedge_b200 import _lib
    names = _declared_symbols()
    assert len(names) >= 19
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(l.split()[-1] for l in out.splitlines() if l.strip())
    for n in names:
        assert n in exported, f"{n} declared in include/mte.h but not exported by libmte.so"
        assert n in _lib.EXPORTED_SYMBOLS, f"{n} has no ctypes signature"
    assert _lib.lib.mte_version() == 200
    assert _lib.lib.mte_error_string(0) == b"ok"
    assert b"workspace" in _lib.lib.mte_error_string(-3)


def test_library_is_sm100a_and_in_tree():
    from mindtheedge_b200 import _lib
    assert _lib.LIB_PATH.startswith(ROOT)
    out = subprocess.run(["cuobjdump", "-lelf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out


def test_host_side_argument_checks_without_a_gpu():
    """Workspace queries and argument validation are pure host code."""
    import ctypes as C
    from mindtheedge_b200 import _lib
    L = _lib.lib
    sc = (_lib.LossScale * 1)()
    sc[0].pred = 256; sc[0].edge = 512; sc[0].B, sc[0].h, sc[0].w, sc[0].H, sc[0].W = 4, 384, 1280, 384, 1280
    n = L.mte_edge_loss_workspace_bytes(sc, 1)
    assert 256 < n < (1 << 22)
    assert L.mte_edge_loss_ctx_bytes(sc, 1) >= 4 * 4
    sc[0].B = 0
    assert L.mte_edge_loss_workspace_bytes(sc, 1) == 0
    at = _lib.LossAttrs(1, 1, 0, 4.0, 1.0, 1.0)
    assert L.mte_edge_loss_fwd(sc, 1, C.byref(at), None, None, None, 0, None) == -1       # NULL
    assert L.mte_edge_loss_fwd(sc, 1, C.byref(at), 256, 256, 256, 1 << 20, None) == -2    # shape
    sc[0].B = 4
    assert L.mte_edge_loss_fwd(sc, 5, C.byref(at), 256, 256, 256, 1 << 20, None) == -4    # n_scales
    assert L.mte_edge_loss_fwd(sc, 1, C.byref(at), 256, 256, 256, 16, None) == -3         # workspace
    assert L.mte_canny_workspace_bytes(102, 384, 1280, 12) > 2 * 102 * 384 * 1280
    assert L.mte_canny_workspace_bytes(0, 384, 1280, 12) == 0
    lows, highs = (C.c_int32 * 1)(10), (C.c_int32 * 1)(20)
    assert L.mte_canny_from_depth(256, 0, 1, 8, 8, 0.0, 80.0, lows, highs, 1, None, None, 256, 1 << 20, None) == -1
    assert L.mte_canny_from_depth(256, 7, 1, 8, 8, 0.0, 80.0, lows, highs, 1, 256, None, 256, 1 << 20, None) == -4
    assert L.mte_pr_workspace_bytes(4, 384, 1280, 12, 0.002) > 0
    assert L.mte_pr_counts(256, 2, 256, 1, 8, 8, None, None, 300, 0.002, 0, 256, 256, 1 << 30, None) == -4
    assert L.mte_dee_workspace_bytes(2, 384, 1280) > 0 and L.mte_thin_workspace_bytes(2, 10, 10) > 0
    assert L.mte_dee_postprocess(None, 0, 1, 8, 8, 1, 1, 0.3, 0.7, None, None, 1, None, 0, None) == -1
    assert L.mte_edge_loss_alt_workspace_bytes(2, 48, 64) > 2 * 2 * 48 * 64 * 4
    assert L.mte_edge_loss_alt_fwd(256, 256, None, 1, 8, 8, 8, 1, 4.0, 1.0, None, 256, 256, 256, 1 << 20, None) == -4   # dice alone
    assert L.mte_edge_loss_alt_fwd(256, 256, None, 1, 8, 8, 1, 1, 4.0, 1.0, None, 256, 256, 256, 1 << 20, None) == -4   # CE without its loss
    assert L.mte_edge_resize_workspace_bytes(4) > 0 and L.mte_edge_resize_workspace_bytes(0) == 0
    assert L.mte_decode_normals(None, None, 16, None) == -1
    assert L.mte_edge_resize_preserve(256, 1, 8, 8, 256, 4, 4, 256, 16, None) == -3
    assert L.mte_chamfer_workspace_bytes(3, 384, 1280) > 3 * 384 * 1280 * 2 and L.mte_chamfer_workspace_bytes(0, 4, 4) == 0
    assert L.mte_chamfer_counts(None, None, 1, 8, 8, 5.0, None, None, None, 0, None) == -1
    assert L.mte_chamfer_counts(256, 256, 1, 8, 8, 5.0, 256, None, 256, 16, None) == -3


def test_no_cpu_fallback():
    from mindtheedge_b200 import _lib
    from mindtheedge_b200.edge import canny_from_depth
    from mindtheedge_b200.eval_depth_edges import pr_counts
    from mindtheedge_b200.losses import GradLoss
    from mindtheedge_b200.tools import dee_postprocess
    x = torch.rand(1, 1, 8, 8)
    with pytest.raises(_lib.MteError):
        GradLoss("cross_entropy")(x, x)
    with pytest.raises(_lib.MteError):
        canny_from_depth(x[0, 0], [(10, 20)])
    with pytest.raises(_lib.MteError):
        pr_counts(x[0], x[0].to(torch.uint8), [0.5])
    with pytest.raises(_lib.MteError):
        dee_postprocess(x[0, 0])
    with pytest.raises(ValueError):
        GradLoss("dice")                      # no base loss: NameError in the reference (grad_loss.py:150-156)
    with pytest.raises(_lib.MteError):
        GradLoss("attention_loss_dice")(x, x, None, False, False)   # CPU tensors: no fallback for any loss type
    src = open(os.path.join(ROOT, "mindtheedge_b200", "losses.py")).read() + \
        open(os.path.join(ROOT, "mindtheedge_b200", "eval_depth_edges.py")).read()
    assert "import oracle" not in src and "from oracle" not in src


def test_pr_host_arithmetic_vs_reference_golden():
    from mindtheedge_b200.eval_depth_edges import (_threshold_grid, compute_rec_prec_f1,
                                                   mean_recall_at_precision_range)
    z = np.load(os.path.join(GOLDEN, "pr.npz"))
    assert np.array_equal(_threshold_grid(9), z["soft_thr"])
    c = z["soft_counts_thin0"].astype(np.float64)
    rec, prec, f1 = compute_rec_prec_f1(c[:, 0], c[:, 1], c[:, 2], c[:, 3])
    assert (rec <= 1).all() and (prec <= 1).all() and np.isfinite(f1).all()
    r0, p0, f0 = compute_rec_prec_f1(np.zeros(2), np.zeros(2), np.zeros(2), np.zeros(2))
    assert (r0 == 0).all() and (p0 == 0).all() and (f0 == 0).all()
    pr = np.vstack((z["pr_precision"], z["pr_recall"])).transpose()
    assert mean_recall_at_precision_range(pr) == z["pr_auc_full"]
    assert mean_recall_at_precision_range(pr, 0.12, 0.65) == z["pr_auc_part"]
    with pytest.raises(ValueError):
        _threshold_grid([0.5])


def test_shard_indices_cover_every_image_once():
    from mindtheedge_b200.eval_depth_edges import shard_indices
    for n, world in [(102, 8), (49, 8), (3, 4), (0, 2), (102, 1)]:
        seen = sorted(i for r in range(world) for i in shard_indices(n, r, world))
        assert seen == list(range(n))


_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r}); sys.path.insert(0, os.path.join({root!r}, "tests"))
import numpy as np, torch, torch.distributed as dist
from synth import scene_with_gt
from oracle import pr_counts as opr
from mindtheedge_b200.eval_depth_edges import shard_indices, all_reduce_counts
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=int(sys.argv[1]), world_size=2)
gts, depths = zip(*[scene_with_gt(64, 160, 900 + k, n_rect=8) for k in range(5)])
rng, crop = [40, 120], (4, 150, 4, 60)
mine = shard_indices(5)
local = opr.pr_sweep_counts([depths[i] for i in mine], [gts[i] for i in mine], rng, crop) if mine else np.zeros((2, 4), np.int64)
t = all_reduce_counts(torch.from_numpy(local.astype(np.int64)))
full = opr.pr_sweep_counts(depths, gts, rng, crop)
assert np.array_equal(t.numpy(), full), (t, full)
dist.destroy_process_group()
print("rank", sys.argv[1], "ok", mine)
"""


def test_two_rank_count_reduction_gloo(tmp_path):
    """N>1 path on CPU: images sharded i -> rank i mod 2, ONE integer all-reduce, result identical to the
    single-process sum (SURVEY.md 8e)."""
    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(root=ROOT, port=29500 + os.getpid() % 500))
    procs = [subprocess.Popen([sys.executable, str(script), str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                              text=True) for r in range(2)]
    outs = [p.communicate(timeout=300)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o
        assert "ok" in o


def test_reference_arm_prints_one_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours): one JSON line with the contract's keys, the
    same metric / unit as our arm, and no GPU needed."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "edge_loss_fwd_bwd_throughput" and d["unit"] == "Mpixel/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["n_gpus"] == 1
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]


def test_bench_dump_outputs_types_and_budget(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float64 for float64 / int64 data and float32 for u8 / fp32, whole arrays while the set
    fits the budget; over it, every array of one size is sampled at the same seeded positions in every run."""
    import bench
    small = {"counts": np.arange(12, dtype=np.int64).reshape(3, 4), "edges": np.arange(6, dtype=np.uint8).reshape(2, 3)}
    bench.dump_outputs(str(tmp_path / "small"), small)
    c, e = np.load(tmp_path / "small" / "counts.npy"), np.load(tmp_path / "small" / "edges.npy")
    assert c.dtype == np.float64 and np.array_equal(c, small["counts"])
    assert e.dtype == np.float32 and np.array_equal(e, small["edges"])
    monkeypatch.setattr(bench, "DUMP_BYTES", 6000)
    big = {"a": np.arange(1000, dtype=np.float32).reshape(10, 100), "b": np.arange(1000, dtype=np.float64) * 2}
    for run in ("r1", "r2"):
        bench.dump_outputs(str(tmp_path / run), big)
    a, b = np.load(tmp_path / "r1" / "a.npy"), np.load(tmp_path / "r1" / "b.npy")
    assert a.nbytes + b.nbytes <= 6000 and a.size == b.size == 500
    assert (np.diff(a) > 0).all() and np.array_equal(b, 2 * a.astype(np.float64))
    assert np.array_equal(a, np.load(tmp_path / "r2" / "a.npy"))


def test_atan2_candidate_error_bound():
    """dee_front_tma_kernel (csrc/dee.cu: atan2_candidate) lets an fp32 angle candidate decide the u8 normal level and
    the NMS bin ALONE when it is >= 1e-3 levels / 5e-5 bin units away from every boundary.  That needs a hard bound
    on the candidate's error: the same polynomial, emulated here in fp32 (with a deliberately sloppy division: the
    kernel's rcp.approx is good to 1 ulp), must stay within 3e-6 rad of atan2 -- 1.2e-4 levels, 3.8e-6 bin units."""
    f = np.float32

    def fma(a, b, c):
        return (a.astype(np.float64) * b.astype(np.float64) + np.float64(c)).astype(f)

    def cand(y, x, sloppy):
        ax, ay = np.abs(x), np.abs(y)
        mx, mn = np.maximum(ax, ay), np.minimum(ax, ay)
        t = (mn * ((f(1) / mx) * f(sloppy)).astype(f)).astype(f)
        t2 = (t * t).astype(f)
        p = fma(t2, np.full_like(t2, f(-0.0117212)), f(0.05265332))
        for c in (-0.11643287, 0.19354346, -0.33262347, 0.99997726):
            p = fma(p, t2, f(c))
        p = (p.astype(np.float64) * t.astype(np.float64)).astype(f)
        p = np.where(ay > ax, f(1.57079637) - p, p).astype(f)
        p = np.where(x < 0, f(3.14159274) - p, p).astype(f)
        return np.where(y < 0, -p, p).astype(f)

    rng = np.random.default_rng(0)
    n = 2_000_000
    ang = rng.uniform(-np.pi, np.pi, n)
    r = np.exp(rng.uniform(np.log(1e-30), np.log(1e30), n))
    X, Y = r * np.cos(ang), r * np.sin(ang)
    for sloppy in (1.0, 1.0 + 3e-7, 1.0 - 3e-7):
        a = cand(Y.astype(f), X.astype(f), sloppy).astype(np.float64)
        err = np.abs(a - np.arctan2(Y, X))
        err = np.minimum(err, 2 * np.pi - err)
        assert err.max() < 3e-6, err.max()
    t = np.linspace(0, 1, 1_000_001).astype(f)
    a = cand(t, np.ones_like(t), 1.0).astype(np.float64)
    assert np.abs(a - np.arctan(t.astype(np.float64))).max() < 3e-6
