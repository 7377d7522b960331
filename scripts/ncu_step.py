"""Target for ncu: eager bench-shape train steps with cudaProfilerStart/Stop around the last STEPS of them.

    ncu --profile-from-start off --metrics gpu__time_duration.sum --clock-control none --csv \
        --log-file gpurun_out/launches.csv python scripts/ncu_step.py 2
    ncu --profile-from-start off --set full --clock-control none --import-source on -k regex:k_tc2 \
        -o gpurun_out/tc_full python scripts/ncu_step.py 1

Same shapes / dropout as bench.py (YOOCHOOSE ADER period-4 step), the same C-ABI calls the captured graph holds."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import bench
from ader_b200 import ops
from ader_b200.model import Ader

steps = int(sys.argv[1]) if len(sys.argv) > 1 else 2
WL = bench.WL
dev = torch.device("cuda", 0)
B, Me, V, Vp = WL["B"], WL["M_e"], WL["V"], WL["V_prev"]
M = B + Me
model = Ader(WL["item_num"], bench.make_args(), device=dev, init_seed=0)
model.update_loss(WL["lam"])
rng = np.random.RandomState(100)
t_ids, t_lab, t_len = bench.synth_rows(rng, 32768, V)
e_ids, e_lab, e_len = bench.synth_rows(rng, WL["exemplars"], Vp)
d_t_ids, d_t_lab, d_e_ids = torch.from_numpy(t_ids).to(dev), torch.from_numpy(t_lab).to(dev), torch.from_numpy(e_ids).to(dev)
teacher = torch.randn((WL["exemplars"], (Vp + 3) // 4 * 4), device=dev)[:, :Vp] * 2
ids_buf = torch.empty((M, 50), dtype=torch.int32, device=dev)


def step():
    ti = rng.randint(0, 32768, B).astype(np.int32); ei = rng.randint(0, WL["exemplars"], Me).astype(np.int32)
    dti, dei = torch.from_numpy(ti).to(dev), torch.from_numpy(ei).to(dev)
    pos = d_t_lab[dti.long()]
    ntok = int(t_len[ti].sum() + e_len[ei].sum())
    torch.cuda.synchronize()
    if step.on:
        torch.cuda.profiler.start()
    ops.gather_rows_i32(d_t_ids, dti, ids_buf[:B]); ops.gather_rows_i32(d_e_ids, dei, ids_buf[B:])
    model.train_step(ids_buf, pos, V, WL["lr"], WL["dropout"], exemplar_logits=teacher, teacher_rows=dei, n_tokens=ntok)
    torch.cuda.synchronize()
    if step.on:
        torch.cuda.profiler.stop()


step.on = False
for _ in range(5):
    step()
step.on = True
for _ in range(steps):
    step()
print("profiled %d steps" % steps)
