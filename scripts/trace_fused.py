"""Phase timeline of the one-pass loss kernel (-DMTE_FUSED_TRACE build selected with MTE_LIB): %globaltimer stamps
folded over all CTAs.  Config-3 loss shape, rotating input sets.  Prints the table and one JSON line of medians.
Builds from before the split grid barrier fill eight slots only: their two extra events print as n/a."""
import ctypes as C, json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np, torch
import bench
from mindtheedge_b200 import _lib
from mindtheedge_b200.losses import _attrs, _scales_struct
dev = torch.device("cuda", 0)
sets = [bench.loss_inputs(8, 1000 + i, dev) for i in range(4)]
at = _attrs(True, True, True, 4.0, 10.0, 1.0)
w = [0.25] * 4
keep = []
for sc in sets:
    pred = [t[0] for t in sc]; edge = [t[1] for t in sc]; normal = [t[2] for t in sc]
    gmap = [torch.empty_like(e) for e in edge]; gpred = [torch.empty_like(p) for p in pred]
    b = _scales_struct(pred, edge, normal, None, gmap, gpred, w)
    losses = torch.zeros(5, device=dev); ctx = torch.zeros(_lib.lib.mte_edge_loss_ctx_bytes(b, 4) // 4, device=dev)
    ws = torch.zeros(_lib.lib.mte_edge_loss_workspace_bytes(b, 4), dtype=torch.uint8, device=dev)
    keep.append((b, gmap, gpred, losses, ctx, ws))
st = torch.cuda.current_stream().cuda_stream
NSLOT = 10
SLOTS = slice(1032, 1032 + 8 * NSLOT)   # byte 1024 past the barrier counter (ticket[2])
rows = []
for it in range(24):
    b, _, _, losses, ctx, ws = keep[it % 4]
    ws[SLOTS].zero_()
    torch.cuda.synchronize()
    _lib.check(_lib.lib.mte_edge_loss_fwd_grad(b, 4, C.byref(at), None, losses.data_ptr(), ctx.data_ptr(), ws.data_ptr(), ws.numel(), st))
    torch.cuda.synchronize()
    t = ws[SLOTS].cpu().numpy().view(np.uint64).astype(np.uint64)
    inv = lambda v: np.uint64(~np.uint64(v))
    base = int(inv(t[0]))
    rel = lambda v: float(int(v) - base) if v else float("nan")
    first_out = rel(inv(t[8])) if t[8] else float("nan")
    ev = [rel(t[1]), rel(inv(t[2])), rel(t[3]), first_out, rel(t[4]), rel(inv(t[5])), rel(t[6]), rel(t[9]), rel(t[7])]
    if it >= 8:
        rows.append(ev)
r = np.array(rows, dtype=np.float64) / 1e3
names = ["last CTA starts", "first CTA ends phase 1", "last CTA ends phase 1 (last arrival)",
         "first CTA leaves the barrier", "last CTA leaves the barrier", "first CTA ends phase 2", "last CTA ends phase 2",
         "last CTA elected", "loss written"]
med = np.median(r, 0)
for n, m, lo, hi in zip(names, med, r.min(0), r.max(0)):
    if np.isnan(m):
        print("%-38s n/a" % n)
    else:
        print("%-38s median %6.2f us  (min %6.2f max %6.2f) after the first CTA's start" % (n, m, lo, hi))
d = lambda a, b_: None if np.isnan(med[b_] - med[a]) else round(float(np.median(r[:, b_] - r[:, a])), 3)
out = {"lib": os.path.basename(_lib.LIB_PATH), "launches": len(rows),
       "median_us": {n: (None if np.isnan(m) else round(float(m), 3)) for n, m in zip(names, med)},
       "last_arrival_to_first_out_us": d(2, 3), "last_arrival_to_last_out_us": d(2, 4),
       "last_p2_end_to_elected_us": d(6, 7), "elected_to_loss_us": d(7, 8), "last_p2_end_to_loss_us": d(6, 8)}
print(json.dumps(out), flush=True)
