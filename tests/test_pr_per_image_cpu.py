"""Per-image PR counts without a GPU: the host-side checks of mte_pr_counts_per_image and the multi-rank assembly of
per-image rows (gloo, world_size 2)."""
import ctypes as C
import os
import subprocess
import sys

from conftest import ROOT


def test_per_image_entry_point_argument_checks_without_a_gpu():
    """The argument checks of mte_pr_counts, in the same order, before anything touches a device."""
    from mindtheedge_b200 import _lib
    L = _lib.lib
    thr = (C.c_double * 1)(0.5)
    small = L.mte_pr_workspace_bytes(1, 8, 8, 1, 0.0075)
    f = L.mte_pr_counts_per_image
    assert f(256, 0, 256, 1, 8, 8, None, thr, 1, 0.0075, 0, None, 256, 1 << 30, None) == -1            # NULL counts
    assert f(256, 0, 256, 1, 8, 8, None, None, 1, 0.0075, 0, 256, 256, 1 << 30, None) == -1            # NULL thresholds
    assert f(256, 0, 256, 0, 8, 8, None, thr, 1, 0.0075, 0, 256, 256, 1 << 30, None) == -2            # no image
    assert f(256, 2, 256, 1, 8, 8, None, None, 255, 0.002, 0, 256, 256, 1 << 30, None) == -4           # T > 254
    assert f(256, 2, 256, 1, 8, 8, None, None, 0, 0.002, 0, 256, 256, 1 << 30, None) == -4
    assert f(256, 0, 256, 1, 8, 8, None, thr, 1, 0.0075, 2, 256, 256, 1 << 30, None) == -4            # apply_thinning
    assert f(256, 0, 256, 1, 8, 8, None, thr, 1, -1.0, 0, 256, 256, 1 << 30, None) == -4               # max_dist
    assert f(256, 0, 256, 1, 8, 8, None, thr, 1, 0.0075, 0, 256, 256, small - 1, None) == -3           # workspace
    assert f(256, 0, 256, 1, 8, 8, None, thr, 1, 0.0075, 1, 256, 256, small, None) == -3              # thinned workspace
    for args in [(256, 0, 256, 1, 8, 8, None, thr, 1, 0.0075, 0, None, 256, 1 << 30, None),
                 (256, 2, 256, 1, 8, 8, None, None, 300, 0.002, 1, 256, 256, 1 << 30, None),
                 (256, 0, 256, 1, 8, 8, None, thr, 1, 0.0075, 2, 256, 256, 1 << 30, None)]:
        assert f(*args) == L.mte_pr_counts(*args)


_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r}); sys.path.insert(0, os.path.join({root!r}, "tests"))
import numpy as np, torch, torch.distributed as dist
from synth import scene_with_gt
from oracle import pr_counts as opr
from mindtheedge_b200.eval_depth_edges import shard_indices, all_reduce_counts
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=int(sys.argv[1]), world_size=2)
gts, depths = zip(*[scene_with_gt(64, 160, 900 + k, n_rect=8) for k in range(5)])
rng, crop = [40, 120, 80], (4, 150, 4, 60)
# what pr_evaluation_arrays(per_image=True) does: each rank fills its own rows of a zero [N,T,4], one integer
# all-reduce assembles them
rows = torch.zeros((5, len(rng), 4), dtype=torch.int64)
for i in shard_indices(5):
    rows[i] = torch.from_numpy(opr.pr_sweep_counts([depths[i]], [gts[i]], rng, crop))
all_reduce_counts(rows)
single = np.stack([opr.pr_sweep_counts([d], [g], rng, crop) for d, g in zip(depths, gts)])
assert np.array_equal(rows.numpy(), single), (rows, single)
assert np.array_equal(rows.numpy().sum(0), opr.pr_sweep_counts(depths, gts, rng, crop))
# the fractional per-image sum_r of the mask branch: one writer per entry, the other rank adds 0.0
s = torch.zeros(5, dtype=torch.float64)
for i in shard_indices(5):
    s[i] = float(np.float64(gts[i] > 127).sum()) / 3.0
all_reduce_counts(s)
assert np.array_equal(s.numpy(), np.array([float(np.float64(g > 127).sum()) / 3.0 for g in gts]))
dist.destroy_process_group()
print("rank", sys.argv[1], "ok", shard_indices(5))
"""


def test_two_rank_per_image_rows_gloo(tmp_path):
    """Images sharded i -> rank i mod 2; the rows gathered by one all-reduce equal the single-process rows."""
    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(root=ROOT, port=29000 + os.getpid() % 500))
    procs = [subprocess.Popen([sys.executable, str(script), str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                              text=True) for r in range(2)]
    outs = [p.communicate(timeout=300)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o
        assert "ok" in o
