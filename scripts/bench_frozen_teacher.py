"""Stored teacher logits vs a frozen teacher snapshot (data.FrozenTeacher): step time, loss-group time and peak device memory.

    python scripts/bench_frozen_teacher.py [--out profiles/frozen_teacher.json] [--steps 200] [--warmup 20]

Configurations (bench.py's two workloads, plus the exemplar budget the reference uses by default):
  yoochoose_p4  M = 512 + 138 rows, V = 18 661, V_prev = 17 421, 30 000 exemplars (stored and frozen)
  synthetic1m   M = 4096 + 1024 rows, V = 1 000 000, V_prev = 900 000, 2 048 exemplars (stored and frozen)
  synthetic1m_30k  the same with 30 000 exemplars, frozen only (the stored matrix would be 108 GB)
Times: CUDA events around `steps` replays of the captured training step (GraphStep, index-fed as the driver runs a period:
batch gather + fused encoder + tcgen05 loss + Adam, dropout 0.3) after `warmup` replays, and around `steps` eager calls of
the tcgen05 loss group alone (ader_loss_fwd_bwd_tc) on a fixed rep.  Peak memory: torch.cuda.max_memory_allocated from
the moment the teacher (stored matrix or snapshot) exists, through capture and all timed calls -- model, teacher and step
workspaces; the set-up that builds the teacher is not included.  FLOPs: algorithmic work of the
teacher passes, 2 * M_e * V_prev * d per pass (the frozen form runs two; the stored form none).  The card's name and power
limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CONFIGS = {
    "yoochoose_p4": dict(item_num=25958, B=512, M_e=138, V=18661, V_prev=17421, E=30000, forms=("logits", "frozen")),
    "synthetic1m": dict(item_num=1000000, B=4096, M_e=1024, V=1000000, V_prev=900000, E=2048, forms=("logits", "frozen")),
    "synthetic1m_30k": dict(item_num=1000000, B=4096, M_e=1024, V=1000000, V_prev=900000, E=30000, forms=("frozen",)),
}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = [x.strip() for x in q.split(",")]
        return dict(name=name, power_limit=plim, max_sm_clock=clk)
    except Exception as e:                     # still report what torch knows
        return dict(name=torch.cuda.get_device_name(0), power_limit="unread (%s)" % type(e).__name__)


def ids_rows(rng, n, V):
    ids = np.zeros((n, 50), np.int32)
    lens = np.minimum(50, rng.geometric(0.25, n))
    for r in range(n):
        ids[r, 50 - lens[r]:] = rng.randint(1, V + 1, lens[r])
    return ids, int(lens.sum())


def run_form(cfg, form, steps, warmup):
    from ader_b200 import ops
    from ader_b200.data import FrozenTeacher
    from ader_b200.model import Ader
    torch.cuda.empty_cache()
    args = type("Args", (), dict(hidden_units=150, maxlen=50, num_blocks=2, num_heads=1, random_seed=0, lr=5e-4,
                                 dropout_rate=0.3, disable_distillation=False, loss_impl="tc"))()
    m = Ader(cfg["item_num"], args, init_seed=0)
    rng = np.random.RandomState(0)
    B, Me, V, Vp, E = cfg["B"], cfg["M_e"], cfg["V"], cfg["V_prev"], cfg["E"]
    dev = m.device
    # exemplar sessions and their reps under the "previous model" (the live weights stand in for it), in chunks like
    # ExemplarGenerator; the stored form is the [E, V_prev] matrix this snapshot stands for (built, then the snapshot dropped)
    ex_ids, reps = [], []
    for lo in range(0, E, 8192):
        ex, ntok = ids_rows(rng, min(8192, E - lo), Vp)
        ex_ids.append(ex)
        reps.append(m.rep(ex, n_tokens=ntok).clone())
    ft = FrozenTeacher(m, torch.cat(reps), Vp)
    del reps
    teacher = ft if form == "frozen" else ft.logits()
    del ft
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()     # peak = model + teacher + what the steps allocate (not the set-up above)
    teacher_bytes = teacher.nbytes() if form == "frozen" else teacher.numel() * 4
    m.update_loss(1.0)
    # GPU-resident row sources and per-step indices, as the driver feeds a period (main.py: index-fed graph replays)
    n_pool = 4 * B
    pool, _ = ids_rows(rng, n_pool, V)
    lab = rng.randint(1, V + 1, n_pool).astype(np.int32)
    src = (torch.from_numpy(pool).to(dev), torch.from_numpy(lab).to(dev),
           torch.from_numpy(np.concatenate(ex_ids)).to(dev), torch.arange(E, dtype=torch.int32, device=dev))
    ex_all = np.concatenate(ex_ids)
    n_in_pool, n_in_ex = (pool != 0).sum(1), (ex_all != 0).sum(1)
    plan = []
    for _ in range(8):
        ti, ei = rng.randint(0, n_pool, B).astype(np.int32), rng.randint(0, E, Me).astype(np.int32)
        plan.append((torch.from_numpy(ti).to(dev), torch.from_numpy(ei).to(dev), int(n_in_pool[ti].sum() + n_in_ex[ei].sum())))
    cap = max(p[2] for p in plan)
    gs = m.graph_step(B, Me, V, 5e-4, 0.3, teacher=teacher, sources=src, tcaps=[cap])
    gs.precapture(indexed=True)
    step = lambda i: gs.run_indices(plan[i % 8][0], plan[i % 8][1], plan[i % 8][2])
    for i in range(warmup):
        step(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        step(i)
    e1.record()
    torch.cuda.synchronize()
    step_ms = e0.elapsed_time(e1) / steps
    # the loss group alone (eager ader_loss_fwd_bwd_tc calls) on a fixed rep
    ti, ei, _ = plan[0]
    pos = src[1][ti.long()].contiguous()
    rep_fixed = torch.randn(B + Me, 150, device=dev) * 0.3
    fz = (teacher.rep, teacher.table, teacher.table16) if form == "frozen" else ()
    a = ops.make_loss_args(B + Me, B, Me, V, Vp, 1, 1.0, pos, None, None if form == "frozen" else teacher, ei, 0, 0, *fz)
    ws = torch.empty(ops.loss_tc_ws_bytes(m.ms, a), dtype=torch.uint8, device=dev)
    loss = torch.zeros(1, device=dev); row_loss = torch.empty(B + Me, device=dev); d_rep = torch.empty_like(rep_fixed)
    call = lambda: ops.loss_fwd_bwd_tc(m.ms, m.theta, rep_fixed, a, ws, loss, row_loss, d_rep, m.grad)
    for _ in range(warmup):
        call()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        call()
    e1.record()
    torch.cuda.synchronize()
    loss_ms = e0.elapsed_time(e1) / steps
    peak = torch.cuda.max_memory_allocated()
    n_et = (B + Me - 1) // 128 - B // 128 + 1
    out = dict(form=form, step_ms_graph_replay=step_ms, loss_group_ms_eager=loss_ms, steps=steps, warmup=warmup,
               peak_mem_bytes=int(peak), teacher_bytes=int(teacher_bytes),
               stored_matrix_bytes_would_be=int(E * Vp * 4),
               teacher_pass_flop_algorithmic=(2 * 2 * Me * Vp * 150) if form == "frozen" else 0,
               teacher_pass_flop_issued=(2 * 2 * n_et * 128 * ((Vp + 127) // 128 * 128) * 160) if form == "frozen" else 0,
               loss=float(loss.item()), step_loss=float(m._loss.item()))
    del gs, m, teacher, ws, src
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "frozen_teacher.json"))
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--configs", default=",".join(CONFIGS))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_frozen_teacher needs a CUDA device")
    res = dict(card=card(), torch=torch.__version__, when=time.strftime("%Y-%m-%d %H:%M:%S"), configs={})
    for name in a.configs.split(","):
        cfg = CONFIGS[name]
        res["configs"][name] = dict(shape={k: v for k, v in cfg.items() if k != "forms"}, forms=[])
        for form in cfg["forms"]:
            r = run_form(cfg, form, a.steps, a.warmup)
            print(name, json.dumps(r), flush=True)
            res["configs"][name]["forms"].append(r)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["card"]))


if __name__ == "__main__":
    main()
