#!/usr/bin/env python
"""bench.py -- train sessions/sec of the ADER hot path on B200 (BASELINE.json metric).

A "step" is one pass of the hot path over one batch: encoder forward, full-vocabulary logits +
CE + adaptive distillation, backward (incl. embedding scatter) and the TF1-Adam update, on the
shape of BASELINE.json configs[1] (YOOCHOOSE ADER, --batch_size=512): 512 train rows + 138
exemplar rows per step, V = 18 661 items, V_prev = 17 421, table 25 959 rows (period 4 of the
shipped split, SURVEY A.4), synthetic sessions with the YOOCHOOSE length histogram.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

N > 1 (under torchrun): data parallel, one rank per GPU, per-rank batch fixed (weak scaling); the gradients
are summed and Adam applied by one kernel over NVLink peer memory (csrc/dp.cu; ADER_B200_DP=nccl selects the
NCCL all-reduce + replicated Adam instead).  The same run also times the reference's global batch split over
the ranks (strong scaling, `strong_scaling` in the JSON line).  `--impl reference` times the reference's own
CPU implementation of the same step (its torch-CPU restatement under oracle/, TensorFlow is not
installable here) on the host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# ---- workload: YOOCHOOSE ADER, period-4 shape (SURVEY A.4; measured with the reference loaders) ----
WL = dict(name="yoochoose_ader_train_step(period4 shape)", item_num=25958, B=512, M_e=138, V=18661, V_prev=17421,
          lam=1.0, lr=5e-4, pool_rows=110699, exemplars=30000, dropout=0.3)   # dropout 0.3: main.py:106,141 (ADER runs train with it)
# BASELINE configs[4]: synthetic 1M-item vocabulary, seq len 50, batch 4096 (+ 1024 exemplar rows distilled against 900k
# previous-period items); selected with --config synthetic1m.  At N > 1 the step is data parallel like configs[1]: per-rank
# rows fixed, table gradient reduce-scattered / parameters all-gathered by the peer-memory (or NVLS) optimiser kernel.
WL_SYNTH1M = dict(name="synthetic_1M_items_train_step(batch 4096 + 1024 exemplar rows, seq len 50)", item_num=1000000, B=4096,
                  M_e=1024, V=1000000, V_prev=900000, lam=1.0, lr=5e-4, pool_rows=32768, exemplars=2048, dropout=0.3)
# P(input length = k), k = 0..50, of YOOCHOOSE period-5 training rows (reference Sampler, seed 0)
LEN_HIST = [0.0001, 0.3048, 0.1778, 0.1171, 0.0812, 0.0597, 0.0449, 0.0352, 0.0279, 0.0221, 0.018, 0.0148, 0.0124,
            0.0102, 0.0086, 0.0072, 0.0063, 0.0053, 0.0046, 0.0041, 0.0036, 0.0031, 0.0028, 0.0024, 0.0022, 0.0018,
            0.0017, 0.0016, 0.0014, 0.0012, 0.0011, 0.001, 0.0009, 0.0008, 0.0008, 0.0007, 0.0007, 0.0006, 0.0005,
            0.0005, 0.0005, 0.0005, 0.0004, 0.0004, 0.0003, 0.0003, 0.0003, 0.0003, 0.0003, 0.0003, 0.0047]


def make_args():
    return type("Args", (), dict(hidden_units=150, maxlen=50, num_blocks=2, num_heads=1, random_seed=0, lr=WL["lr"],
                                 dropout_rate=0.0, disable_distillation=False))()


def synth_rows(rng, n, vmax, L=50):
    p = np.array(LEN_HIST[1:], np.float64)
    p /= p.sum()
    lens = rng.choice(np.arange(1, L + 1), size=n, p=p)
    if WL.get("full_len"):          # SURVEY 8(d) "seq len 50" variant: every slot of every row filled
        lens = np.full(n, L, dtype=lens.dtype)
    ids = np.zeros((n, L), np.int32)
    # item popularity ~ Zipf-like over 1..vmax (hot rows exercise the scatter)
    u = rng.random_sample((n, L))
    items = np.minimum(vmax, np.floor(vmax ** u).astype(np.int64)).astype(np.int32)
    items = np.maximum(items, 1)
    mask = np.arange(L)[None, :] >= (L - lens)[:, None]
    ids[mask] = items[mask]
    label = np.maximum(1, np.minimum(vmax, np.floor(vmax ** rng.random_sample(n)).astype(np.int64))).astype(np.int32)
    return ids, label, lens.astype(np.int32)


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.samples = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.time(), line.strip()))

    def stop(self, windows):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        rows = []
        for ts, line in self.samples:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                rows.append((ts, float(f[0]), float(f[1]), f[3:7]))
            except ValueError:
                continue
        inwin = [r for r in rows if any(a - 0.05 <= r[0] <= b + 0.05 for a, b in windows)] or rows
        if not inwin:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in inwin for i in range(4) if r[3][i].lower().startswith("active")})
        return {"sm_mhz": float(np.median([r[1] for r in inwin])), "sm_max_mhz": inwin[0][2], "reasons": reasons,
                "samples": len(inwin)}


# --------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's algorithm on the host cores (oracle restatement)
# --------------------------------------------------------------------------------------------------
def cpu_step_fn():
    import torch
    from oracle import sasrec as S
    # torchrun exports OMP_NUM_THREADS=1 to its workers: the CPU arm must still use every host core it can
    try:
        torch.set_num_threads(max(1, len(os.sched_getaffinity(0))))
    except Exception:
        torch.set_num_threads(max(1, os.cpu_count() or 1))
    hp = S.Hyper(WL["item_num"])
    params = S.init_params(hp, 0)
    rng = np.random.RandomState(1)
    M = WL["B"] + WL["M_e"]
    ids, label, _ = synth_rows(rng, M, WL["V"])
    ids_t = torch.tensor(ids).long()
    pos = torch.tensor(label[:WL["B"]])
    teacher = torch.tensor(rng.standard_normal((WL["M_e"], WL["V_prev"])).astype(np.float32))
    opt = S.AdamTF1(params)
    state = {"params": params}

    def step():
        fn = lambda ps: S.loss_ader(ps, ids_t, pos, WL["V"], hp, WL["lam"], exemplar_logits=teacher)
        loss, grads = S.grads_of(fn, state["params"])
        state["params"] = opt.step(state["params"], grads, WL["lr"])
        return loss

    return step, M, torch.get_num_threads()


def run_cpu(steps: int, warmup: int):
    step, M, cores = cpu_step_fn()
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    return M * steps / dt, dt / steps * 1e3, cores, M


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if WL["V"] > 200000:     # [M, V] fp32 logits + the one-hot of the restated graph: ~40 GB of host memory per step at 1M items
        print(json.dumps({"impl": "reference", "unavailable": "CPU restatement not run at the 1M-item shape (materialises [5120, 1M] fp32 twice)"}))
        return
    val, ms, cores, M = run_cpu(args.steps, args.warmup)
    sample = ("%d full steps after %d warm-up steps of %d rows, dense over 50 slots, [M,V] logits "
              "materialised, torch-CPU fp32 restatement of the reference graph" % (args.steps, args.warmup, M))
    line = {"impl": "reference", "metric": "train sessions/sec", "value": val, "unit": "sessions/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(1),
            "cpu_baseline": {"value": val, "unit": "sessions/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "sessions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------------
# the metric as BASELINE.json words it: train sessions/sec PER PERIOD on the shipped split + eval rows/sec
# --------------------------------------------------------------------------------------------------
def find_data_root():
    for root in (os.environ.get("ADER_DATA_ROOT"), os.path.join(ROOT, "data_cache"), os.path.join(ROOT, "data")):
        if root and os.path.isdir(os.path.join(root, "YOOCHOOSE")):
            return root
    return None


def real_period_run(n_periods=2, num_epochs=4):
    """YOOCHOOSE ADER (BASELINE configs[1]: --lambda_=1.0 --batch_size=512 --test_batch=64) through the product driver
    (ader_b200.main.run: real samplers, epoch-resident index queue, early stopping, evaluation, herding), bounded to the
    first periods / epochs; returns the driver's own per-period throughput records."""
    import io, tempfile, contextlib
    from ader_b200.main import build_parser, run
    root = find_data_root()
    if root is None:
        return {"unavailable": "no YOOCHOOSE period files (ADER_DATA_ROOT / data_cache are not tracked in git)"}
    a = build_parser().parse_args([])
    a.dataset, a.data_root, a.lambda_, a.batch_size, a.test_batch = "YOOCHOOSE", root, 1.0, 512, 64
    a.max_periods, a.num_epochs, a.checkpoint = n_periods, num_epochs, False
    tmp = tempfile.mkdtemp(prefix="ader_bench_")
    a.results_root, a.cache_dir = tmp, os.path.join(tmp, "cache")
    t0 = time.time()
    with contextlib.redirect_stdout(io.StringIO()):
        out = run(a)
    wall = time.time() - t0
    recs = [{k: (round(v, 4) if isinstance(v, float) else ([round(x, 4) for x in v] if isinstance(v, list) and v and isinstance(v[0], float) else v))
             for k, v in r.items()} for r in out["throughput"]]
    return {"dataset": "YOOCHOOSE (shipped split)", "periods": recs, "wall_s": round(wall, 2), "epochs_cap": num_epochs,
            "note": "train_s = epoch loops only (valid eval excluded), eval_s = validation passes + test pass incl. the rank D2H; "
                    "dropout 0.3, herding exemplars, adaptive distillation from period 2"}


def gpu_components(dev):
    """Kernel-group throughputs beside the train step (BASELINE.md section 3, C4-C6 counterparts): evaluation ranking at the
    DIGINETICA period-10 shape, segmented herding, EWC Fisher."""
    import torch
    from ader_b200 import ops
    from ader_b200.model import Ader, Ewc
    out = {}
    rng = np.random.RandomState(7)
    # evaluation: R rows, V = 40 135 (SURVEY A.4 period 10), fused tcgen05 ranking vs the exact fp32 path
    a = make_args()
    m = Ader(43136, a, device=dev, init_seed=0)
    R, V = 16384, 40135
    ids, lab, lens = synth_rows(rng, R, V)
    gt = torch.from_numpy(lab).to(dev)
    ids_d = torch.from_numpy(ids).to(dev)
    for impl in ("tc", "exact"):
        m.eval_impl = impl
        m.rank_topk(ids_d, gt, V, 0, n_tokens=int(lens.sum()))
        torch.cuda.synchronize()
        t0 = time.time()
        for _ in range(3):
            m.rank_topk(ids_d, gt, V, 0, n_tokens=int(lens.sum()))
        torch.cuda.synchronize()
        out["eval_rows_per_s_" + impl] = R * 3 / (time.time() - t0)
    out["eval_shape"] = {"rows": R, "max_item": V, "includes": "encoder pass (exact fp32) + ranking"}
    out["eval_fallbacks"] = m.eval_fallbacks
    # herding: N candidate rows in segments with the YOOCHOOSE-like size mix (median 3, a few large)
    sizes = np.minimum(3000, np.maximum(1, (rng.pareto(1.1, 12000) * 2).astype(np.int64) + 1))
    N = int(sizes.sum())
    rep = torch.randn(N, 150, device=dev)
    seg_off = np.zeros(len(sizes) + 1, np.int32); np.cumsum(sizes, out=seg_off[1:])
    quota = np.minimum(sizes, np.maximum(1, sizes // 2)).astype(np.int32)
    steps = np.ceil(1.1 * quota).astype(np.int32)
    t = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev)
    cand = torch.arange(N, dtype=torch.int32, device=dev)
    picks = torch.zeros(N, dtype=torch.int32, device=dev); n_p = torch.zeros(len(sizes), dtype=torch.int32, device=dev)
    ws = torch.empty(ops.herding_ws_bytes(m.ms, N), dtype=torch.uint8, device=dev)
    args_h = (m.ms, rep, cand, t(seg_off), t(quota), t(steps), ws, picks, n_p)
    ops.herding_segmented(*args_h); torch.cuda.synchronize()
    t0 = time.time(); ops.herding_segmented(*args_h); torch.cuda.synchronize()
    dt = time.time() - t0
    out["herding"] = {"candidate_rows": N, "segments": int(len(sizes)), "largest": int(sizes.max()), "seconds": dt, "rows_per_s": N / dt,
                      "gbs_compulsory": N * 150 * 4 / dt / 1e9}
    # EWC Fisher (EWC.py:126-164): S sessions at batch-1 semantics, V_tab = 43 137
    e = Ewc(43136, a, device=dev, init_seed=0)
    S_ = 4096
    sess = [list(rng.randint(1, V + 1, int(n) + 1)) for n in np.minimum(50, rng.geometric(0.22, S_) + 1)]
    import random
    random.seed(0)
    e.compute_fisher(None, sess[:256], 50, V)                        # warm-up (workspace allocation, first launches)
    torch.cuda.synchronize(); t0 = time.time()
    e.compute_fisher(None, sess, 50, V)
    torch.cuda.synchronize()
    out["fisher_samples_per_s"] = S_ / (time.time() - t0)
    out["fisher_shape"] = {"samples": S_, "v_tab": 43137, "includes": "host session sampling + batched exact backward + fp64 accumulation"}
    del m, e
    torch.cuda.empty_cache()
    return out


def cpu_components(budget_s=6.0):
    """CPU baselines C4-C7 of BASELINE.md section 3 on bounded samples (oracle restatement, all host cores)."""
    import torch
    from oracle import protocol as P
    from oracle import sasrec as S
    try:
        torch.set_num_threads(max(1, len(os.sched_getaffinity(0))))
    except Exception:
        pass
    out = {"cores": torch.get_num_threads()}
    rng = np.random.RandomState(11)
    hp = S.Hyper(43136)
    params = S.init_params(hp, 0)
    V = 40135
    # C4: evaluation at test_batch = 64 with argsort(argsort(-logits)) semantics (ADER.py:99-103, util.py:323-339)
    ids, lab, _ = synth_rows(rng, 64, V)
    n, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < budget_s:
        with torch.no_grad():
            lg = S.logits_of(S.forward_rep(params, torch.tensor(ids).long(), hp), params[0], V)
            ranks = torch.argsort(torch.argsort(-lg, dim=1), dim=1)          # the reference's double argsort
            _ = ranks[torch.arange(64), torch.tensor(lab).long() - 1]
        n += 64
    out["C4_eval_rows_per_s"] = n / (time.perf_counter() - t0)
    # C5: herding, the reference's per-item NumPy loop (util.py:419-434)
    sizes = np.minimum(3000, np.maximum(1, (rng.pareto(1.1, 4000) * 2).astype(np.int64) + 1))
    reps = [rng.randn(int(k), 150).astype(np.float32) for k in sizes]
    n, t0 = 0, time.perf_counter()
    for r in reps:
        P.herding_picks(r, max(1, len(r) // 2))
        n += len(r)
        if time.perf_counter() - t0 > budget_s:
            break
    out["C5_herding_rows_per_s"] = n / (time.perf_counter() - t0)
    # C6: Fisher, one full forward + backward per sample (EWC.py:142-161)
    ids, lab, _ = synth_rows(rng, 8, V)
    n, t0 = 0, time.perf_counter()
    for i in range(8):
        S.fisher_diag(params, torch.tensor(ids[i:i + 1]).long(), torch.tensor(lab[i:i + 1]), V, hp, 1)
        n += 1
        if time.perf_counter() - t0 > budget_s:
            break
    out["C6_fisher_samples_per_s"] = n / (time.perf_counter() - t0)
    # C7: logits + CE forward / backward at the synthetic 1 M-item vocabulary, row-chunked (16 GB of logits otherwise)
    E = torch.randn(1000001, 150) * 0.05
    rep = torch.randn(64, 150, requires_grad=True)
    Et = E[1:].clone().requires_grad_(True)
    pos = torch.randint(0, 1000000, (64,))
    n, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < budget_s:
        loss = torch.nn.functional.cross_entropy(rep @ Et.t(), pos)
        loss.backward()
        rep.grad = None; Et.grad = None
        n += 64
    out["C7_synthetic1m_logits_sessions_per_s"] = n / (time.perf_counter() - t0)
    out["sample"] = "each figure: as many units as fit in ~%.0f s on the host cores (64-row eval batches at V=40135; herding items of the YOOCHOOSE size mix; single-sample Fisher passes at V_tab=43137; 64-row chunks of the 1M-item logits+CE fwd/bwd)" % budget_s
    return out


GROUP = int(os.environ.get("ADER_B200_GRAPH_STEPS", "1"))      # steps per graph replay of the resident region (the product default: 1)
DUMP_MAX_ELEMS = 1 << 22       # per dumped array (16 MiB in fp32): the 1M-item table is sampled, the YOOCHOOSE one is not


def step_outputs(model, loss):
    """What a train step hands its caller, on the host: the step's loss, the parameters it leaves and the gradient it
    computed.  Arrays longer than DUMP_MAX_ELEMS keep one element of each of DUMP_MAX_ELEMS equal strata of their index
    range, at an offset drawn from np.random.default_rng(0): the same sample in every run and every build."""
    import torch
    n = model.theta.numel()
    idx = None
    if n > DUMP_MAX_ELEMS:
        edges = np.arange(DUMP_MAX_ELEMS + 1, dtype=np.int64) * n // DUMP_MAX_ELEMS
        offs = (np.random.default_rng(0).random(DUMP_MAX_ELEMS) * np.diff(edges)).astype(np.int64)
        idx = torch.from_numpy(edges[:-1] + offs).to(model.device)
    out = {"loss": loss.detach().reshape(-1).cpu().numpy()}
    for name, t in (("theta", model.theta), ("grad", model.grad)):
        out[name] = (t if idx is None else t[idx]).detach().cpu().numpy()
    return out


def workload_config(n):
    return {"workload": WL["name"], "batch_size": WL["B"], "exemplar_rows": WL["M_e"], "max_item": WL["V"],
            "prev_max_item": WL["V_prev"], "table_rows": WL["item_num"] + 1, "lambda": WL["lam"], "maxlen": 50,
            "hidden_units": 150, "num_blocks": 2, "dropout_rate": WL["dropout"], "global_batch": (WL["B"] + WL["M_e"]) * n,
            "parallelism": "dp%d" % n if n > 1 else "single",
            "l2": "per-step working set (theta+m+v+grad of %d rows, logits workspace) exceeds the 126 MB L2; "
                  "inputs change every step" % (WL["V"] + 1)}


# --------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------
def gpu_arm(args):
    import torch
    import torch.distributed as dist
    from ader_b200 import ops
    from ader_b200.model import Ader

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    t_boot = time.time()

    def crumb(stage):                  # per-rank breadcrumbs: a wedged multi-GPU run shows where every rank stopped
        sys.stderr.write("[bench rank %d/%d +%.1fs] %s\n" % (rank, world, time.time() - t_boot, stage))
        sys.stderr.flush()

    def on_timeout():
        crumb("WATCHDOG: no result after 600 s, leaving")
        os._exit(3)

    wd = threading.Timer(600.0, on_timeout)     # a wedged collective must not hold the box (the driver's own limit is 870 s)
    wd.daemon = True
    wd.start()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        crumb("process group up")
    K, W = args.steps, max(args.warmup, 3)
    B, Me, V, Vp = WL["B"], WL["M_e"], WL["V"], WL["V_prev"]
    M = B + Me

    model = Ader(WL["item_num"], make_args(), device=dev, init_seed=0)
    model.update_loss(WL["lam"])
    dp_kind = None
    if world > 1:       # data parallel: global-mean denominators, gradients summed over the ranks (ader_b200/dist.py)
        from ader_b200.dist import make_comm, shard_rows
        model.dp = make_comm(model)
        dp_kind = model.dp.kind
        crumb("data-parallel back end: %s" % dp_kind)
    # every rank builds the SAME row pools and the index streams of ALL ranks (host integers): the graph buckets below are
    # then identical on every rank, so all ranks capture the same graphs in the same order (a rank-dependent bucket set
    # left ranks inside NCCL graph capture while the others were already replaying: the round-1 hang at N = 8)
    rng = np.random.RandomState(100)
    pool = 32768
    t_ids, t_lab, t_len = synth_rows(rng, pool, V)
    e_ids, e_lab, e_len = synth_rows(rng, WL["exemplars"], Vp)
    d_t_ids, d_t_lab = torch.from_numpy(t_ids).to(dev), torch.from_numpy(t_lab).to(dev)
    d_e_ids = torch.from_numpy(e_ids).to(dev)
    gen = torch.Generator(device=dev); gen.manual_seed(5)
    ld_t = (Vp + 3) // 4 * 4     # rows 16-byte aligned, as ExemplarGenerator stores them
    teacher = (torch.randn((WL["exemplars"], ld_t), device=dev, generator=gen) * 2.0)[:, :Vp]   # stored exemplar logits, HBM resident

    nsteps = W + K
    ntok_all = []
    for r in range(world):
        rr = np.random.RandomState(1000 + r)
        ti_r = [rr.randint(0, pool, B).astype(np.int32) for _ in range(nsteps)]
        ei_r = [rr.randint(0, WL["exemplars"], Me).astype(np.int32) for _ in range(nsteps)]
        ntok_all += [int(t_len[a].sum() + e_len[b].sum()) for a, b in zip(ti_r, ei_r)]
        if r == rank:
            ti_all, ei_all = ti_r, ei_r
    ntok = [int(t_len[a].sum() + e_len[b].sum()) for a, b in zip(ti_all, ei_all)]
    d_ti = [torch.from_numpy(a).to(dev) for a in ti_all]
    d_ei = [torch.from_numpy(a).to(dev) for a in ei_all]
    ids_buf = torch.empty((M, 50), dtype=torch.int32, device=dev)

    P = WL["dropout"]
    gs = None
    d_e_row = torch.arange(WL["exemplars"], dtype=torch.int32, device=dev)      # stored teacher row of each exemplar
    if world > 1:
        model.global_counts = (B * world, Me * world)
    if not args.no_graph:       # the step as CUDA graphs (one per token-capacity bucket); same C-ABI calls as the eager step
        caps = sorted({int(-(-q // 256) * 256) for q in np.quantile(ntok_all, [0.5, 0.9, 0.99, 1.0])})
        # epoch-resident index queue (ader_b200/main.py PeriodTrainer.run_epoch): the row indices of every step of the
        # resident region live in HBM, a step graph gathers its batch from the queue, GROUP consecutive steps are one replay
        q_host = np.concatenate([np.concatenate([a, b]) for a, b in zip(ti_all, ei_all)]).astype(np.int32)
        queue = (torch.from_numpy(q_host).to(dev), torch.arange(nsteps, dtype=torch.int64, device=dev) * (B + Me),
                 torch.zeros(1, dtype=torch.int32, device=dev))
        gs = model.graph_step(B, Me, V, WL["lr"], P, teacher=teacher, sources=(d_t_ids, d_t_lab, d_e_ids, d_e_row), tcaps=caps,
                              queue=queue)
        crumb("graph step built, buckets %s" % (gs.tcaps,))
        gs.precapture()          # graphs are captured on first use otherwise: keep that out of the timed regions
        for cap in gs.tcaps:
            gs._graph_for(cap, "q")
            if GROUP > 1:
                gs._graph_for(cap, "q", GROUP)
        crumb("graphs captured")

    def resident_step(i):
        if gs is not None:
            return gs.run_indices(d_ti[i], d_ei[i], ntok[i])
        ops.gather_rows_i32(d_t_ids, d_ti[i], ids_buf[:B])
        ops.gather_rows_i32(d_e_ids, d_ei[i], ids_buf[B:])
        pos = d_t_lab[d_ti[i].long()]
        return model.train_step(ids_buf, pos, V, WL["lr"], P, exemplar_logits=teacher, teacher_rows=d_ei[i],
                                n_tokens=ntok[i])

    def e2e_step(i):
        if gs is not None:
            return gs.run_rows(h_ids[i], h_pos[i], ei_all[i], ntok[i])
        return model.train_step(h_ids[i], h_pos[i], V, WL["lr"], P, exemplar_logits=teacher, teacher_rows=ei_all[i],
                                n_tokens=ntok[i])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    clocks = ClockSampler(local) if rank == 0 else None
    windows = []

    # ---- value: inputs resident in HBM -----------------------------------------------------------
    def resident_run(lo, hi):
        """Steps [lo, hi) of the resident region: the queued epoch loop of the product (GROUP steps per graph replay).
        Returns the device loss of the last step."""
        loss = None
        if gs is None:
            for i in range(lo, hi):
                loss = resident_step(i)
            return loss
        i = lo
        while i < hi:
            n = GROUP if (GROUP > 1 and i + GROUP <= hi) else 1
            loss = gs.run_queued(max(ntok[i:i + n]), nsteps=n)
            i += n
        return loss

    resident_run(0, W)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.time()
    e0.record()
    last_step_loss = resident_run(W, W + K)
    e1.record()
    barrier()
    windows.append((w0, time.time()))
    # the later regions keep training the same model: take the outputs of the timed region's last step now
    outputs = step_outputs(model, last_step_loss) if args.dump_outputs and rank == 0 else None
    ms_total = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms_total], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    value = M * K * world / (ms_total / 1e3)

    # ---- e2e: public API with HOST buffers, H2D of the step inputs + D2H of the loss every step ---
    h_ids = [np.concatenate([t_ids[a], e_ids[b]]) for a, b in zip(ti_all, ei_all)]
    h_pos = [t_lab[a] for a in ti_all]
    for i in range(min(W, 3)):
        float(e2e_step(i).item())
    barrier()
    w0 = time.time()
    e0.record()
    if gs is not None:
        # every step: host batch -> pinned staging -> ONE H2D copy -> graph replay -> pinned D2H of its loss; the host
        # reads the loss of step i after it has fed step i+1 (one step in flight), all K losses inside the timed region
        pend = None
        for i in range(W, W + K):
            e2e_step(i)
            nxt = gs.fetch_loss()
            if pend is not None:
                last_loss = pend.result()
            pend = nxt
        last_loss = pend.result()
    else:
        for i in range(W, W + K):
            last_loss = float(e2e_step(i).item())
    e1.record()
    barrier()
    windows.append((w0, time.time()))
    ms_e2e = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms_e2e], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_e2e = float(t.item())
    e2e_value = M * K * world / (ms_e2e / 1e3)
    h2d = M * 50 * 4 + B * 4 + Me * 4
    clock_info = clocks.stop(windows) if clocks else None

    crumb("weak-scaling + e2e regions timed")

    # ---- strong scaling (N > 1): the REFERENCE's global batch (B + M_e rows, the parity configuration of SURVEY 8e) split
    # over the ranks -- train rows and exemplar rows separately, global-mean denominators -- reported beside the weak line
    strong = None
    if world > 1 and gs is not None:
        (tl, th), (el, eh) = shard_rows(B, Me, rank, world)
        rg = np.random.RandomState(999)
        ti_g = [rg.randint(0, pool, B).astype(np.int32) for _ in range(nsteps)]
        ei_g = [rg.randint(0, WL["exemplars"], Me).astype(np.int32) for _ in range(nsteps)]
        nt_rank = [[int(t_len[a[slice(*shard_rows(B, Me, r, world)[0])]].sum() + e_len[b[slice(*shard_rows(B, Me, r, world)[1])]].sum())
                    for a, b in zip(ti_g, ei_g)] for r in range(world)]
        caps_s = sorted({int(-(-q // 128) * 128) for q in np.quantile(np.concatenate(nt_rank), [0.5, 0.9, 1.0])})
        model.global_counts = (B, Me)
        gss = model.graph_step(th - tl, eh - el, V, WL["lr"], P, teacher=teacher, sources=(d_t_ids, d_t_lab, d_e_ids, d_e_row), tcaps=caps_s)
        gss.precapture(indexed=True)
        crumb("strong-scaling graphs captured (%d + %d rows per rank)" % (th - tl, eh - el))
        d_tis = [torch.from_numpy(a[tl:th].copy()).to(dev) for a in ti_g]
        d_eis = [torch.from_numpy(b[el:eh].copy()).to(dev) for b in ei_g]
        for i in range(W):
            gss.run_indices(d_tis[i], d_eis[i], nt_rank[rank][i])
        barrier()
        e0.record()
        for i in range(W, W + K):
            gss.run_indices(d_tis[i], d_eis[i], nt_rank[rank][i])
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_s = float(t.item())
        strong = {"value": M * K / (ms_s / 1e3), "unit": "sessions/s", "ms_per_step": ms_s / K, "global_batch": M,
                  "rows_per_rank": [th - tl, eh - el], "scaling": "strong",
                  "note": "reference batch size kept (parity configuration): latency-bound, the all-gather of theta is on the chain"}
        model.global_counts = (B * world, Me * world)
        crumb("strong-scaling region timed")
    if model.dp is not None:
        model.dp.check()        # a timed-out peer wait would have produced garbage: fail loudly

    # ---- per-phase device times (CUDA events on the launching stream), averaged over the timed inputs
    phases = {}
    reps = min(K, 50) if world == 1 else 0      # eager single-rank launches (a lone rank must not enter the collective)
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(5)] for _ in range(reps)]
    for r in range(reps):
        i = W + r
        ops.gather_rows_i32(d_t_ids, d_ti[i], ids_buf[:B])
        ops.gather_rows_i32(d_e_ids, d_ei[i], ids_buf[B:])
        pos = d_t_lab[d_ti[i].long()]
        evs[r][0].record()
        model.loss_and_grad(ids_buf, pos, V, exemplar_logits=teacher, teacher_rows=d_ei[i], n_tokens=ntok[i],
                            dropout_rate=P, _events=evs[r][1:4])
        model.apply_gradients(V, WL["lr"])
        evs[r][4].record()
    torch.cuda.synchronize()
    for name, a, b in (("encoder_fwd", 0, 1), ("logits_ce_kd_fwd_bwd", 1, 2), ("encoder_bwd_scatter", 2, 3), ("adam", 3, 4)):
        phases[name] = float(np.mean([evs[r][a].elapsed_time(evs[r][b]) for r in range(reps)])) if reps else None

    # ---- kernel launch count + in-pipeline kernel durations (CUPTI via torch.profiler, outside the timed regions)
    launches_per_step = None
    kernels_us = {}
    try:
        from torch.profiler import ProfilerActivity, profile
        nprof = 10
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for r in range(nprof):
                resident_step(W + r)
            torch.cuda.synchronize()
        cnt = 0
        for e in prof.events():
            if e.device_type.name != "CUDA":
                continue
            n = e.name.split("(")[0].replace("void ", "")
            if "ader" in n or n.startswith("k_"):
                cnt += 1
                kernels_us[n] = kernels_us.get(n, 0.0) + e.device_time / nprof
        launches_per_step = cnt // nprof
        if os.environ.get("ADER_B200_TRACE") and rank == 0:      # kernel timeline of the replayed steps (critical-path analysis)
            prof.export_chrome_trace(os.environ["ADER_B200_TRACE"])
    except Exception:
        pass

    # ---- the north-star kernel group alone: logits + CE + KD forward/backward (ader_loss_fwd_bwd_tc), captured as its
    # own CUDA graph and timed with CUDA events over back-to-back replays (fresh teacher rows every replay) -----------
    loss_group_ms = None
    tc_kernels_ms = None
    try:
        rep_in = torch.randn((M, 150), device=dev) * 0.5
        pos_in = d_t_lab[d_ti[W].long()].contiguous()
        rows_in = d_ei[W].clone()
        la = ops.make_loss_args(M, B, Me, V, Vp, model.KD, WL["lam"], pos_in, None, teacher, rows_in)
        lws = torch.empty(ops.loss_tc_ws_bytes(model.ms, la), dtype=torch.uint8, device=dev)
        rl, dr, ls = torch.empty(M, device=dev), torch.empty((M, 150), device=dev), torch.zeros(1, device=dev)
        gsave = model.grad.clone()
        run_loss = lambda: ops.loss_fwd_bwd_tc(model.ms, model.theta, rep_in, la, lws, ls, rl, dr, model.grad)
        side = torch.cuda.Stream(); side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            run_loss()
        torch.cuda.current_stream().wait_stream(side); torch.cuda.synchronize()
        gl = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gl):
            run_loss()
        nrep = 50
        for r in range(5):
            rows_in.copy_(d_ei[W + r]); gl.replay()
        torch.cuda.synchronize()
        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ea.record()
        for r in range(nrep):
            rows_in.copy_(d_ei[W + (r % K)]); gl.replay()
        eb.record(); torch.cuda.synchronize()
        loss_group_ms = ea.elapsed_time(eb) / nrep
        # ... and the three tcgen05 kernels of that group alone (k_tc_logits<FWD>, <DREP>, <DE>) on the workspace the
        # group just prepared: the launches the roofline is quoted on
        run_k = lambda: ops.debug_loss_tc_kernels(model.ms, model.theta, la, lws, model.grad)
        with torch.cuda.stream(side):
            run_k()
        torch.cuda.current_stream().wait_stream(side); torch.cuda.synchronize()
        gk = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gk):
            run_k()
        for r in range(5):
            gk.replay()
        torch.cuda.synchronize()
        ea.record()
        for r in range(nrep):
            gk.replay()
        eb.record(); torch.cuda.synchronize()
        tc_kernels_ms = ea.elapsed_time(eb) / nrep
        model.grad.copy_(gsave)
    except Exception as ex:      # noqa: BLE001
        sys.stderr.write("loss-group timing failed: %r\n" % (ex,))

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
        peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained" if peaks else "fallback"
        flops = 6.0 * M * 150 * V                      # SURVEY 8d: fwd + bwd of the output projection, d counted as 150
        dom_ms = tc_kernels_ms or loss_group_ms or phases["logits_ce_kd_fwd_bwd"]
        if not dom_ms:
            raise RuntimeError("the tcgen05 loss kernels could not be timed")
        achieved = flops / (dom_ms * 1e-3) / 1e12
        traffic = None          # dram__bytes_read.sum + dram__bytes_write.sum of the three launches (ncu --set full, profiles/)
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "tc_traffic.json")))
            if tr.get("workload") == WL["name"]:
                traffic = tr["dram_bytes_per_step"]
        except Exception:
            pass
        # the kernel that dominates the step BY TIME is not the north-star kernel: the weight-gradient launches (TF32 legacy
        # mma.sync).  Algorithmic work 2 * T * d * d per matrix, 5 matrices per block; in-pipeline durations from the CUPTI pass
        # above; peak = the probe-measured mma.sync rate (profiles/r2/hmma_probe.txt: 0.45 m16n8k8 per cycle per SM)
        dominant = None
        try:
            wname = max((k for k in kernels_us if "k_wgrad" in k), key=lambda k: kernels_us[k])
            t_mean = float(np.mean(ntok[W:W + 10]))
            wflops = 2.0 * t_mean * 150 * 150 * 5 * 2
            sm_mhz = (clock_info or {}).get("sm_mhz") or 1965.0
            wpeak = 0.45 * 2048 * 148 * sm_mhz * 1e6 / 1e12
            wach = wflops / (kernels_us[wname] * 1e-6) / 1e12
            dominant = {"kernel": wname + " (all launches of a step, in-pipeline durations)", "bound": "tensor (legacy mma.sync tf32)",
                        "achieved": wach, "peak": wpeak, "unit": "TFLOP/s", "frac": wach / wpeak,
                        "us_per_step": kernels_us[wname], "algorithmic_flops_per_step": wflops,
                        "peak_source": "hmma_probe: 0.45 mma.m16n8k8 per cycle per SM x 148 SMs x sm clock"}
        except Exception:
            pass
        big = WL["V"] > 200000        # the CPU restatement materialises [M, V] fp32 logits + a one-hot: 40 GB at 1M items
        cpu_val, cpu_ms, cores, _ = (None, None, None, None) if big else run_cpu(2, 1)
        period = components = cpu_comp = None
        if world == 1 and not args.no_period and not big:
            try:
                period = real_period_run()
            except Exception as ex:      # noqa: BLE001
                period = {"error": repr(ex)}
            try:
                components = gpu_components(dev)
                cpu_comp = cpu_components()
            except Exception as ex:      # noqa: BLE001
                components = {"error": repr(ex)}
        line = {"metric": "train sessions/sec", "value": value, "unit": "sessions/s", "n_gpus": world, "steps": K,
                "warmup": W, "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "bf16 operands / f32 accumulate (logits+CE+KD on tcgen05), f32 elsewhere", "data": "synthetic", "config": workload_config(world),
                "e2e": {"value": e2e_value, "unit": "sessions/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                        "ms_per_step": ms_e2e / K, "last_loss": last_loss,
                        "loss_read": "sync .item() per step" if gs is None else "pinned D2H per step, read one step behind"},
                "gpu_launches": (launches_per_step or 0) * K,
                "gpu_launches_per_step": launches_per_step,
                "clocks": clock_info,
                "phases_ms_eager": phases,
                "step_mode": "eager launches" if gs is None else "CUDA graph per token-capacity bucket %s; resident region: epoch-resident index queue, %d steps per graph replay" % (gs.tcaps, GROUP),
                "kernels_us_per_step": dict(sorted(((k, round(v, 2)) for k, v in kernels_us.items()), key=lambda kv: -kv[1])[:12]),
                "loss_group_ms": loss_group_ms,
                "tc_kernels_ms": tc_kernels_ms,
                "step_impl": model.step_impl,
                "dp_backend": dp_kind,
                "strong_scaling": strong,
                "period_metric": period,
                "components": components,
                "cpu_components": cpu_comp,
                "roofline": {"kernel": "k_tc2<FWD> + <DREP> + <DE> (the three tcgen05 launches of logits+CE+KD fwd+bwd; CUDA-event "
                                       "timed graph replays of exactly these launches; the whole 13-launch group is loss_group_ms)",
                             "bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                             "traffic": traffic, "peak_source": peak_src,
                             "algorithmic_flops_per_launch": flops,
                             "group_achieved": flops / (loss_group_ms * 1e-3) / 1e12 if loss_group_ms else None},
                "roofline_step_dominant": dominant,
                "cpu_baseline": None if big else
                                {"value": cpu_val, "unit": "sessions/s", "cores": cores, "kind": "port",
                                 "sample": "2 full steps of %d rows after 1 warm-up, torch-CPU fp32 restatement" % M}}
        if outputs is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, arr in outputs.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
        print(json.dumps(line))
        sys.stdout.flush()
    if world > 1:
        # Leave without tearing NCCL down: destroy_process_group() with captured graphs that hold NCCL kernels alive
        # deadlocked at exit (measured at N=2); every rank has finished its work and rank 0 has printed the line.
        try:
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush(); sys.stderr.flush()
            os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200, help="timed steps, after --warmup untimed ones (with --impl reference too)")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ader_b200")
    ap.add_argument("--no-graph", dest="no_graph", action="store_true", help="issue the step's launches eagerly")
    ap.add_argument("--no-period", dest="no_period", action="store_true",
                    help="skip the real-period run on the shipped split and the component figures (N = 1 only)")
    ap.add_argument("--config", default="yoochoose_p4", choices=["yoochoose_p4", "synthetic1m", "synthetic1m_full"],
                    help="workload: BASELINE configs[1] shape (default, the headline) or configs[4] (1M-item vocabulary; session "
                         "lengths from the YOOCHOOSE histogram, or _full: all 50 slots of every row filled)")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR", default=None,
                    help="write the loss, parameters and gradient of the last timed step as DIR/<name>.npy (float32; at most "
                         "%d elements per array, a fixed seeded sample beyond that) to compare two builds output for output"
                    % DUMP_MAX_ELEMS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU step's outputs: it does not apply to --impl reference")
    if args.config.startswith("synthetic1m"):
        WL.update(WL_SYNTH1M)
        if args.config.endswith("_full"):
            WL.update(full_len=True, name=WL_SYNTH1M["name"] + ", all 50 slots filled")
    if args.impl == "reference":
        reference_arm(args)
    else:
        gpu_arm(args)


if __name__ == "__main__":
    main()
