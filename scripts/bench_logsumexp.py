"""Log-sum-exp throughput and accuracy: ader_logsumexp_tc against ader_logsumexp, and an evaluation pass with and without
the held-out NLL.

    python scripts/bench_logsumexp.py [--out profiles/logsumexp.json] [--reps 5]

Entries: R in {4 096, 65 536} rows, V in {18 661, 43 105, 1 000 000} items, with a ground truth per row (lse and nll);
hidden_units 150, reps N(0, 1/d) * 3 (scores of a few units), item table N(0, 0.25).  CUDA events around the call alone, on
inputs made once; every shape is run once untimed first.  The tc entry gets all R rows, `reps` times.  The exact entry writes
the [rows, V] fp32 scores, so it is timed on as many rows as keep rows * V <= 4.3e9 (17 GB of scores), `reps` times; the
rows used are recorded.  Accuracy: the largest |lse_tc - lse_fp64| over the first min(4 096, 1e9 / V) rows of each shape against an
fp64 product of the same fp32 rep and table, and the largest and mean bound eps_i = 2^-12 ||rep_i|| max_j ||E_j|| there.
Evaluation: Evaluator.evaluate at the DIGINETICA shape (43 136 items, max_item 43 105, hidden_units 150, maxlen 50, 2 blocks)
over 60 000 synthetic validation rows (session lengths geometric, p = 0.25, at most 50), with and without nll=True, rows/s
end to end (host clock, the pass ends with the ranks on the host), alternated `reps` times after one untimed pass each.
The card's name and power limit are read in the same run."""
import argparse
import json
import os
import random
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

RS = (4096, 65536)
VS = (18661, 43105, 1000000)
EXACT_WORK = 4.3e9         # rows * V of one exact call (its [rows, V] fp32 workspace)
D = 150


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = [x.strip() for x in q.split(",")]
        return dict(name=name, power_limit=plim, max_sm_clock=clk)
    except Exception as e:
        return dict(name=torch.cuda.get_device_name(0), power_limit="unread (%s)" % type(e).__name__)


def event_ms(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def entries(reps):
    from ader_b200 import ops
    from ader_b200.params import Hyper, ParamLayout
    out = []
    g = torch.Generator().manual_seed(0)
    for V in VS:
        hp = Hyper(V + 31, D)
        ms = ops.model_struct(hp)
        theta = (torch.randn(ParamLayout(hp).total, generator=g) * 0.5).cuda()
        theta[:D] = 0.0
        table = theta[D:(V + 1) * D].view(V, D)
        for R in RS:
            rep = (torch.randn(R, D, generator=g) * (3.0 / D ** 0.5)).cuda()
            gt = torch.randint(1, V + 1, (R,), generator=g, dtype=torch.int32).cuda()
            lse, nll = torch.empty(R, device="cuda"), torch.empty(R, device="cuda")
            ws = torch.empty(ops.logsumexp_tc_ws_bytes(ms, R, V), dtype=torch.uint8, device="cuda")
            tc = lambda: ops.logsumexp_tc(ms, theta, rep, gt, V, ws, lse, nll)
            tc()
            t_tc = event_ms(tc, reps)
            n = int(min(4096, R, 1e9 // V))
            ref = torch.logsumexp(rep[:n].double() @ table.double().t(), dim=1)
            eps = 2.0 ** -12 * rep[:n].double().norm(dim=1) * table.double().norm(dim=1).max()
            err = (lse[:n].double() - ref).abs()
            del ws
            rows = int(min(R, EXACT_WORK // V))
            ws = torch.empty(ops.eval_ws_bytes(ms, rows, V), dtype=torch.uint8, device="cuda")
            ex = lambda: ops.logsumexp(ms, theta, rep[:rows], gt[:rows], V, ws, lse[:rows], nll[:rows])
            ex()
            t_ex = event_ms(ex, reps)
            del ws
            rec = dict(R=R, V=V, tc_ms=t_tc, tc_rows_per_s=R / t_tc * 1e3, exact_rows=rows, exact_ms=t_ex,
                       exact_rows_per_s=rows / t_ex * 1e3, max_abs_err_tc=float(err.max()), max_eps=float(eps.max()),
                       mean_eps=float(eps.mean()), max_err_over_eps=float((err / eps).max()))
            print(json.dumps(rec), flush=True)
            out.append(rec)
        del theta
        torch.cuda.empty_cache()
    return out


def evaluation(reps):
    from ader_b200.data import Evaluator
    from ader_b200.model import Ader
    args = type("Args", (), dict(hidden_units=D, maxlen=50, num_blocks=2, num_heads=1, random_seed=0, lr=5e-4,
                                 dropout_rate=0.0, disable_distillation=False))()
    m = Ader(43136, args, init_seed=0)
    V = 43105
    rng = np.random.RandomState(0)
    lens = np.minimum(51, rng.geometric(0.25, 60000) + 1)
    rows = [list(rng.randint(1, V + 1, n)) for n in lens]
    cache = {}

    def one(nll):
        random.seed(0)
        ev = Evaluator(rows, True, 50, 64, V, "valid", m, None, cache=cache, nll=nll)
        torch.cuda.synchronize()
        t0 = time.time()
        ev.evaluate(1)
        return time.time() - t0, len(ev.ranks), ev.mean_nll()

    one(False), one(True)
    t = {False: [], True: []}
    for _ in range(reps):
        for nll in (False, True):
            s, n, mean = one(nll)
            t[nll].append(s)
    rec = dict(rows=n, rows_per_s=n / float(np.median(t[False])), rows_per_s_nll=n / float(np.median(t[True])),
               s=t[False], s_nll=t[True], mean_nll=mean, eval_impl=m.eval_impl)
    print(json.dumps(rec), flush=True)
    return rec


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--out", default=os.path.join(ROOT, "profiles", "logsumexp.json"))
    p.add_argument("--reps", default=5, type=int)
    a = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    res = dict(card=card(), entries=entries(a.reps), evaluation=evaluation(a.reps))
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
