"""Outputs and times of the filter-and-refine top-k entries, for comparing two builds of the library bit for bit.

    ADER_B200_LIB=<lib A> python scripts/compare_topk_libs.py run --out a1.json [--reps 7]
    ADER_B200_LIB=<lib B> python scripts/compare_topk_libs.py run --out b1.json
    ... (alternate the two libraries, several runs each)
    python scripts/compare_topk_libs.py compare --a a1.json a2.json ... --b b1.json b2.json ...

`run` computes, with whichever library is loaded, on seeded inputs:
- evaluation at R = 16 384, V = 40 135 (the shape of bench.py's component measurement), k = 0 and k = 20:
  ader_eval_rank_tc / ader_eval_rank_topk_tc, and the exact ader_eval_rank_topk;
- recommendation at the shapes of scripts/bench_recommend.py (R in {4 096, 65 536}, V in {18 661, 43 105, 1 000 000},
  k in {20, 100}), with and without the sessions' own items excluded: ader_recommend_topk_tc, and the exact
  ader_recommend_topk at R = 4 096, V = 43 105.
rep comes from the exact encoder on seeded sessions (hidden_units 150, maxlen 50, 2 blocks, the layout's seeded weights).
Every output, and rep itself (so that `compare` can check both libraries saw the same input), is stored as the SHA-256 of
its dtype, shape and bytes.  Each tensor-core call is run once untimed,
then `reps` times between CUDA events; the median is kept.  The card's name and power limit are read in the same run.

`compare` checks rank, top-k items, top-k scores and the overflow word bit for bit between every run of A and every run of B
(the lists of a call whose overflow word is set are not defined, so there only the word is compared), and prints, per
tensor-core call, the median times of each library over its runs, their range, and the spread (max - min) / mean.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

EVAL = (16384, 40135)
REC_R = (4096, 65536)
REC_V = (18661, 43105, 1000000)
REC_EXACT = (4096, 43105)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    return q


def sessions(rng, n, V, L=50):
    ids = np.zeros((n, L), np.int32)
    lens = np.minimum(L, rng.geometric(0.25, n))
    for r in range(n):
        ids[r, L - lens[r]:] = rng.randint(1, V + 1, lens[r])
    return ids, int(lens.sum())


def run(a):
    import torch
    from ader_b200 import _lib, ops
    from ader_b200.model import Ader
    if not torch.cuda.is_available():
        raise SystemExit("compare_topk_libs needs a CUDA device")
    args = type("Args", (), dict(hidden_units=150, maxlen=50, num_blocks=2, num_heads=1, random_seed=0, lr=5e-4, dropout_rate=0.0))()
    out, times = {}, {}

    def timed(name, call, over):
        call()
        ts = []
        for _ in range(a.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            call()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        times[name] = ts
        out[name + "/overflow"] = int(over.item())

    def keep(name, **tensors):
        for key, t in tensors.items():
            x = t.contiguous().cpu().numpy()
            out[name + "/" + key] = hashlib.sha256(("%s %s" % (x.dtype, x.shape)).encode() + x.tobytes()).hexdigest()

    for V in sorted(set(REC_V) | {EVAL[1]}):
        m = Ader(V, args, init_seed=0)
        for R in sorted(set(REC_R) | {EVAL[0]}):
            if (R, V) != EVAL and not (R in REC_R and V in REC_V):
                continue
            rng = np.random.RandomState(R + V)
            ids_np, n_tok = sessions(rng, R, V)
            ids = torch.from_numpy(ids_np).cuda()
            rep = m.encode(ids, n_tok)[0].clone()
            keep("%dx%d" % (R, V), rep=rep)
            over = torch.zeros(1, dtype=torch.int32, device="cuda")
            if (R, V) == EVAL:
                gt = torch.from_numpy(rng.randint(1, V + 1, R).astype(np.int32)).cuda()
                for k in (0, 20):
                    name = "eval %dx%d k=%d" % (R, V, k)
                    rank = torch.empty(R, dtype=torch.int32, device="cuda")
                    items = torch.empty((R, max(k, 1)), dtype=torch.int32, device="cuda")
                    scores = torch.empty((R, max(k, 1)), dtype=torch.float32, device="cuda")
                    ws = m._eval_ws.get(ops.eval_rank_tc_ws_bytes(m.ms, R, V))
                    if k == 0:
                        timed(name, lambda: ops.eval_rank_tc(m.ms, m.theta, rep, gt, V, ws, rank, over), over)
                        keep(name, rank=rank)
                    else:
                        timed(name, lambda: ops.eval_rank_topk_tc(m.ms, m.theta, rep, gt, V, k, ws, rank, items, scores, over), over)
                        keep(name, rank=rank, items=items, scores=scores)
                    ws = m._eval_ws.get(ops.eval_ws_bytes(m.ms, R, V))
                    ops.eval_rank_topk(m.ms, m.theta, rep, gt, V, k, ws, rank, items, scores)
                    keep("exact " + name, rank=rank, **(dict(items=items, scores=scores) if k else {}))
            else:
                for k in (20, 100):
                    items = torch.empty((R, k), dtype=torch.int32, device="cuda")
                    scores = torch.empty((R, k), dtype=torch.float32, device="cuda")
                    for seen in (ids, None):
                        name = "rec %dx%d k=%d excl=%d" % (R, V, k, seen is not None)
                        ws = m._eval_ws.get(ops.recommend_tc_ws_bytes(m.ms, R, V))
                        try:
                            timed(name, lambda: ops.recommend_topk_tc(m.ms, m.theta, rep, seen, V, k, ws, items, scores, over), over)
                            keep(name, items=items, scores=scores)
                        except _lib.AderError as e:      # too few chunks for k: the entry refuses
                            out[name + "/refused"] = str(e)
                        if (R, V) == REC_EXACT:
                            ws = m._eval_ws.get(ops.eval_ws_bytes(m.ms, R, V))
                            ops.recommend_topk(m.ms, m.theta, rep, seen, V, k, ws, items, scores)
                            keep("exact " + name, items=items, scores=scores)
            del ids, rep
        del m
        torch.cuda.empty_cache()
    with open(a.out, "w") as f:
        json.dump(dict(card=card(), lib=os.environ.get("ADER_B200_LIB", ""), reps=a.reps, times=times, out=out), f, indent=1)
    print("wrote", a.out, flush=True)


def compare(a):
    runs = [("A%d" % (i + 1), json.load(open(p))) for i, p in enumerate(a.a)]
    runs += [("B%d" % (i + 1), json.load(open(p))) for i, p in enumerate(a.b)]
    ref_name, ref = runs[-len(a.b)]
    ok = True
    for name, run_ in runs:
        x, y = run_["out"], ref["out"]
        if sorted(x) != sorted(y):
            print("%s: different outputs from %s: %s" % (name, ref_name, sorted(set(x) ^ set(y))))
            ok = False
            continue
        for key in sorted(x):
            call = key.rsplit("/", 1)[0]
            if key.endswith(("/items", "/scores")) and (x.get(call + "/overflow") or y.get(call + "/overflow")):
                continue
            if x[key] != y[key]:
                print("%s: %s differs from %s" % (name, key, ref_name))
                ok = False
    print("%d runs against %s over %d outputs: %s" % (len(runs), ref_name, len(ref["out"]), "all bit-identical" if ok else "DIFFERENCES"))
    print("card:", ref["card"], "| A:", runs[0][1]["lib"], "| B:", ref["lib"], "| reps per run:", ref["reps"])
    print("%-34s %4s %24s %24s %7s %7s %7s" % ("call", "over", "A ms: median (min-max)", "B ms: median (min-max)", "B/A-1",
                                              "A sprd", "B sprd"))
    for call in sorted(ref["times"]):
        ma = [float(np.median(r["times"][call])) for n, r in runs if n[0] == "A"]
        mb = [float(np.median(r["times"][call])) for n, r in runs if n[0] == "B"]
        print("%-34s %4d %8.3f (%6.3f-%6.3f) %8.3f (%6.3f-%6.3f) %+6.1f%% %6.1f%% %6.1f%%" % (
            call, ref["out"][call + "/overflow"], np.median(ma), min(ma), max(ma), np.median(mb), min(mb), max(mb),
            100 * (np.mean(mb) / np.mean(ma) - 1), 100 * (max(ma) - min(ma)) / np.mean(ma), 100 * (max(mb) - min(mb)) / np.mean(mb)))
    refused = sorted(k.rsplit("/", 1)[0] for k in ref["out"] if k.endswith("/refused"))
    if refused:
        print("refused by the tensor-core entry (too few chunks for k):", ", ".join(refused))
    return 0 if ok else 1


def main():
    p = argparse.ArgumentParser()
    sub = p.add_subparsers(dest="cmd", required=True)
    r = sub.add_parser("run")
    r.add_argument("--out", required=True)
    r.add_argument("--reps", type=int, default=7)
    c = sub.add_parser("compare")
    c.add_argument("--a", nargs="+", required=True)
    c.add_argument("--b", nargs="+", required=True)
    a = p.parse_args()
    sys.exit(run(a) if a.cmd == "run" else compare(a))


if __name__ == "__main__":
    main()
