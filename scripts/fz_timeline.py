"""Debug: phase timeline of the fused tile kernels (build with ADER_B200_DEFINES=-DADER_TC_TIMELINE)."""
import ctypes as C, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import bench
from ader_b200 import _lib
from ader_b200.model import Ader
WL = bench.WL
dev = torch.device("cuda", 0)
B, Me, V, Vp = WL["B"], WL["M_e"], WL["V"], WL["V_prev"]
M = B + Me
model = Ader(WL["item_num"], bench.make_args(), device=dev, init_seed=0)
model.update_loss(WL["lam"])
rng = np.random.RandomState(100)
ids, lab, lens = bench.synth_rows(rng, M, V)
teacher = torch.randn((WL["exemplars"], (Vp + 3) // 4 * 4), device=dev)[:, :Vp] * 2
rows = torch.from_numpy(rng.randint(0, WL["exemplars"], Me).astype(np.int32)).to(dev)
for _ in range(5):
    model.train_step(ids, lab[:B], V, WL["lr"], 0.3, exemplar_logits=teacher, teacher_rows=rows, n_tokens=int(lens.sum()))
torch.cuda.synchronize()
lib = _lib.load()
buf = np.zeros((8, 160, 16), np.int64)
lib.ader_debug_fz_timeline.argtypes = [C.c_void_p]
lib.ader_debug_fz_timeline(buf.ctypes.data_as(C.c_void_p))
names = {0: ("k_qkv_fwd (last = block 1)", ["entry", "setup", "prologue", "weights", "gemmQ", "end"]),
         1: ("k_ffn_bwd (last = block 0)", ["entry", "setup", "stage", "weights", "gemm1+epi", "gemm2+epi", "end"])}
fine = {0: ("qkv_fwd_tile (last tile of block 1)", [6, 7, 2, 3, 4, 8, 5], ["start", "rows loaded+reduced", "LN+tiles+sync", "wait Wq", "gemmQ+epi", "gemmK+epi", "gemmV+epi+sync"]),
        4: ("attn_fwd_group (last group)", [0, 1, 2, 3], ["start", "staged+sync", "keys done", "LN2 done"]),
        5: ("ffn_fwd_tile (last tile)", [0, 1, 2, 5, 3, 4], ["start", "rows+tile+sync", "wait W", "gemm1", "epi1+sync", "gemm2+epi+sync"])}
for k, (nm, slots, labels) in fine.items():
    t = buf[k]
    used = np.nonzero(t[:, slots[0]])[0]
    if len(used) == 0:
        continue
    ts = t[used][:, slots]
    dur = np.diff(ts, axis=1) / 1e3
    print("== %s: %d CTAs" % (nm, len(used)))
    print("   step durations (us) median: " + ", ".join("%s %.2f" % (l, v) for l, v in zip(labels[1:], np.median(dur, axis=0))))
    print("   p90:                        " + ", ".join("%s %.2f" % (l, v) for l, v in zip(labels[1:], np.percentile(dur, 90, axis=0))))
for k, (nm, labels) in names.items():
    if not np.any(buf[k][:, 0]):
        continue
    t = buf[k]
    used = np.nonzero(t[:, 0])[0]
    g0 = t[used, 0].min()
    rel = (t[used][:, :len(labels)] - t[used, 0:1]) / 1e3
    print("== %s: %d CTAs, start spread %.1f us" % (nm, len(used), (t[used, 0].max() - g0) / 1e3))
    print("   phase end times (us from CTA entry), median over CTAs: " + ", ".join("%s %.1f" % (l, v) for l, v in zip(labels, np.median(rel, axis=0))))
    print("   max over CTAs:                                        " + ", ".join("%s %.1f" % (l, v) for l, v in zip(labels, rel.max(axis=0))))
