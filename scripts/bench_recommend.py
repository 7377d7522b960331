"""Recommendation throughput: the encoder pass and the top-k pass of Ader.recommend, tensor-core entry against the exact one.

    python scripts/bench_recommend.py [--out profiles/recommend.json] [--reps 3]

Shapes: R in {4 096, 65 536} sessions per call, V in {18 661, 43 105, 1 000 000} items, k in {20, 100}, the sessions' own
items excluded; hidden_units 150, maxlen 50, 2 blocks, weights from the layout's seeded initialisation, session lengths
geometric (p = 0.25, at most 50), items uniform in 1..V.
Times: CUDA events around the exact-fp32 encoder pass (the one recommend uses) and around the top-k call alone, on a rep
computed once; every shape is run once untimed first.  The tc entry (ader_recommend_topk_tc) gets all R rows in one call,
`reps` times; a call whose candidate list overflows counts as a fallback.  The exact entry (ader_recommend_topk) writes the
[rows, V] fp32 scores and walks each row k times, so it is timed once on the first `rows_timed` rows, as many as keep
rows * V * k <= 1e10 (its time grows linearly in rows); rows/s is over the rows each entry was given.  The lists of the two
entries are compared on the rows both computed, for tc calls that did not overflow; where a call overflowed, Ader.recommend
reruns the batch on the exact entry, and `recommend_rows_per_s` adds the exact entry's time per row (measured on
`rows_timed` rows) to the tc call's.  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

RS = (4096, 65536)
VS = (18661, 43105, 1000000)
KS = (20, 100)
EXACT_WORK = 1e10          # rows * V * k of one timed exact call


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = [x.strip() for x in q.split(",")]
        return dict(name=name, power_limit=plim, max_sm_clock=clk)
    except Exception as e:
        return dict(name=torch.cuda.get_device_name(0), power_limit="unread (%s)" % type(e).__name__)


def sessions(rng, n, V, L=50):
    ids = np.zeros((n, L), np.int32)
    lens = np.minimum(L, rng.geometric(0.25, n))
    for r in range(n):
        ids[r, L - lens[r]:] = rng.randint(1, V + 1, lens[r])
    return ids, int(lens.sum())


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), out


def run_vocab(V, reps, rng):
    from ader_b200 import ops
    from ader_b200.model import Ader
    args = type("Args", (), dict(hidden_units=150, maxlen=50, num_blocks=2, num_heads=1, random_seed=0, lr=5e-4, dropout_rate=0.0))()
    m = Ader(V, args, init_seed=0)
    rows = []
    for R in RS:
        ids_np, n_tok = sessions(rng, R, V)
        ids = torch.from_numpy(ids_np).cuda()
        m.encode(ids, n_tok)
        enc_ms, (rep, _) = timed(lambda: m.encode(ids, n_tok))
        rep = rep.clone()
        for k in KS:
            row = dict(R=R, V=V, k=k, encoder_ms=enc_ms, encoder_rows_per_s=R / enc_ms * 1e3)
            nc = ops.eval_topk_chunks(m.ms, R, V)
            if 16 * nc >= k:
                ws = m._eval_ws.get(ops.recommend_tc_ws_bytes(m.ms, R, V))
                items = torch.empty((R, k), dtype=torch.int32, device="cuda")
                scores = torch.empty((R, k), dtype=torch.float32, device="cuda")
                over = torch.zeros(1, dtype=torch.int32, device="cuda")
                call = lambda: ops.recommend_topk_tc(m.ms, m.theta, rep, ids, V, k, ws, items, scores, over)
                call()
                ts, falls = [], 0
                for _ in range(reps):
                    t, _ = timed(call)
                    ts.append(t)
                    falls += int(over.item() != 0)
                row["tc"] = dict(chunks=nc, topk_ms=float(np.median(ts)), topk_ms_all=ts,
                                 rows_per_s=R / float(np.median(ts)) * 1e3, fallback_fraction=falls / reps)
                tc_items, tc_scores = items.cpu().numpy(), scores.cpu().numpy()
            else:
                row["tc"] = None
            n = int(min(R, max(148, EXACT_WORK // (V * k))))
            ws = m._eval_ws.get(ops.eval_ws_bytes(m.ms, n, V))
            items = torch.empty((n, k), dtype=torch.int32, device="cuda")
            scores = torch.empty((n, k), dtype=torch.float32, device="cuda")
            call = lambda: ops.recommend_topk(m.ms, m.theta, rep[:n], ids[:n], V, k, ws, items, scores)
            call()
            t, _ = timed(call)
            row["exact"] = dict(rows_timed=n, topk_ms=t, rows_per_s=n / t * 1e3)
            if row["tc"] is not None and row["tc"]["fallback_fraction"] == 0:
                row["tc"]["same_lists_as_exact"] = bool(np.array_equal(tc_items[:n], items.cpu().numpy())
                                                        and np.array_equal(tc_scores[:n].view(np.int32),
                                                                           scores.cpu().numpy().view(np.int32)))
                row["tc_speedup_rows_per_s"] = row["tc"]["rows_per_s"] / row["exact"]["rows_per_s"]
            elif row["tc"] is not None:
                # an overflowed call's lists are not used: Ader.recommend reruns the batch on the exact entry
                row["tc"]["same_lists_as_exact"] = None
                row["tc"]["recommend_rows_per_s"] = R / (R / row["tc"]["rows_per_s"] + R / row["exact"]["rows_per_s"])
            print(json.dumps(row), flush=True)
            rows.append(row)
        del rep, ids
        torch.cuda.empty_cache()
    del m
    torch.cuda.empty_cache()
    return rows


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--out", default=os.path.join(ROOT, "profiles", "recommend.json"))
    p.add_argument("--reps", default=3, type=int)
    a = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_recommend needs a CUDA device")
    rng = np.random.RandomState(0)
    res = dict(card=card(), hidden_units=150, maxlen=50, num_blocks=2, exclude_seen=True, reps=a.reps, configs=[])
    for V in VS:
        res["configs"] += run_vocab(V, a.reps, rng)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
