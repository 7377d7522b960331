"""First calls on a second device and from several host threads at once.  A kernel is opted in to its shared memory, and
its module loaded, on its first call on each device (kernel_ready, csrc/common.cuh).  Each case runs in a fresh
interpreter, so no earlier test has prepared a kernel; the work covers every kernel that needs such an opt-in."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SCRIPT = r"""
import sys, threading
import numpy as np, torch
from ader_b200 import ops
from ader_b200.model import Ader
from ader_b200.params import Hyper

V = 2990


def args(loss_impl):
    return type("Args", (), dict(hidden_units=150, maxlen=50, num_blocks=2, num_heads=1, random_seed=0, lr=5e-4,
                                 dropout_rate=0.0, disable_distillation=False, loss_impl=loss_impl))()


def batch():
    rng = np.random.RandomState(3)
    ids = np.zeros((37, 50), np.int32)
    for r in range(37):
        n = int(rng.randint(1, 20)); ids[r, 50 - n:] = rng.randint(1, V + 1, n)
    return ids, rng.randint(1, V + 1, 37).astype(np.int32)


# each returns a closure that launches its work on the current device; building it launches no library kernel
def train(dev):        # the default tc step (fused encoder, k_tc2, k_wgrad2, the DAG), then the tc log-sum-exp
    m, (ids, pos) = Ader(3000, args("tc"), device=dev, init_seed=0), batch()
    def run():
        m.train_step(ids, pos, V)
        lse, nll = m.logsumexp(m.rep(ids), V, pos)
        return [m.theta, lse, nll]
    return run


def exact(dev):        # exact loss_and_grad (k_attn_fwd / k_attn_bwd, the SGEMM), then k_eval_tc ranks and top-k
    m, (ids, pos) = Ader(3000, args("exact"), device=dev, init_seed=0), batch()
    def run():
        m.loss_and_grad(ids, pos, V)
        return [m.grad, *m.rank_topk(ids, pos, V, k=2), *m.recommend(ids, V, k=10)]
    return run


def herding(dev):      # on-chip herding with segments of the mid (17..350) and big (> 350) classes
    sizes = [20, 100, 349, 351, 700]
    N = sum(sizes)
    t = lambda a: torch.tensor(a, dtype=torch.int32, device=dev)
    rep = torch.from_numpy(np.random.RandomState(5).randn(N, 150).astype(np.float32)).to(dev)
    seg_off, quota = t(np.concatenate([[0], np.cumsum(sizes)])), t([n // 2 for n in sizes])
    steps, cand = (quota * 11 + 9) // 10, torch.arange(N, dtype=torch.int32, device=dev)
    ms = ops.model_struct(Hyper(100))
    ws = torch.empty(ops.herding_ws_bytes(ms, N), dtype=torch.uint8, device=dev)
    picks, n_picked = t([-1] * N), t([0] * len(sizes))
    def run():
        ops.herding_segmented(ms, rep, cand, seg_off, quota, steps, ws, picks, n_picked)
        return [picks, n_picked]
    return run


WORK = [train, exact, herding]


def collect(dev):
    with torch.cuda.device(dev):
        return [[x.cpu().numpy() for x in make(torch.device("cuda", dev))()] for make in WORK]


def same(a, b):
    for i, (x, y) in enumerate(zip(a, b)):
        for j, (u, v) in enumerate(zip(x, y)):
            assert u.dtype == v.dtype and u.shape == v.shape and u.tobytes() == v.tobytes(), (WORK[i].__name__, j)


if sys.argv[1] == "devices":       # the same seeded work on device 0, then on device 1
    same(collect(0), collect(1))
else:                              # first calls from one thread per workload at the same moment, then one thread alone
    runs = [make(torch.device("cuda", 0)) for make in WORK]
    start, got, errors = threading.Barrier(len(runs)), [None] * len(runs), []
    def go(i):
        try:
            start.wait()
            got[i] = [x.cpu().numpy() for x in runs[i]()]
        except BaseException as e:
            errors.append(e)
    threads = [threading.Thread(target=go, args=(i,)) for i in range(len(runs))]
    for th in threads: th.start()
    for th in threads: th.join()
    if errors:
        raise errors[0]
    same(got, collect(0))
"""


def _run(mode):
    subprocess.run([sys.executable, "-c", SCRIPT, mode], check=True, cwd=ROOT, timeout=600)


def test_two_devices_one_process_match():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _run("devices")


def test_first_calls_from_threads_match_one_thread():
    _run("threads")
