"""Log-sum-exp of the next-item softmax on the GPU: ader_logsumexp (exact fp32 scores, fp64 sums) and ader_logsumexp_tc
(tcgen05, [R, V] never written) against an fp64 oracle (oracle/sasrec.py logits_of / ce_rows in float64 on the same fp32
rep and table), their determinism, the torch ops, the cross-check with the training loss, ``Ader.recommend(probs=True)``,
the NLL of ``Ader.rank_topk`` / ``Evaluator`` / ``main.run --eval_nll`` and ``python -m ader_b200.recommend --probs``."""
import os
import random
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import sasrec as S

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
C_ERR = 2.0 ** -12
ITEMS = 43200


def _ms(d, item_num=ITEMS):
    from ader_b200 import ops
    from ader_b200.params import Hyper
    return ops.model_struct(Hyper(item_num, d, 50, 1, 1))


def _theta(d, item_num=ITEMS, seed=0):
    """a flat parameter vector whose item table is random (the entries read nothing else)"""
    from ader_b200.params import Hyper, ParamLayout
    n = ParamLayout(Hyper(item_num, d, 50, 1, 1)).total
    g = torch.Generator().manual_seed(seed)
    th = torch.randn(n, generator=g) * 0.5
    th[:d] = 0.0                                              # item 0 (padding) is the zero row
    return th.cuda()


def _reps(R, d, seed=1):
    """scores of a few units; row 0 is zero (lse = log V), every 5th row is scaled x50 (running-max rescale)"""
    g = torch.Generator().manual_seed(seed)
    rep = torch.randn(R, d, generator=g) * (3.0 / d ** 0.5)
    rep[0] = 0.0
    rep[3::5] *= 50.0
    return rep.cuda().contiguous()


def _gt(R, V, seed=2):
    rng = np.random.RandomState(seed)
    gt = rng.randint(1, V + 1, R).astype(np.int32)
    gt[0] = 1
    gt[-1] = V
    if R > 2:
        gt[1] = V
        gt[2] = 1
    return torch.from_numpy(gt).cuda()


def _oracle(theta, rep, gt, d, V):
    table = theta[:(V + 1) * d].view(V + 1, d).double()
    lg = S.logits_of(rep.double(), table, V)
    lse = torch.logsumexp(lg, dim=1)
    nll = S.ce_rows(lg, gt)
    return lse.cpu().numpy(), nll.cpu().numpy()


def _eps(theta, rep, d, V):
    table = theta[d:(V + 1) * d].view(V, d).double()
    return (C_ERR * rep.double().norm(dim=1) * table.norm(dim=1).max()).cpu().numpy()


def _fp32_dot(theta, rep, d, V):
    """rounding bound of an fp32 dot product of length d: gamma_d sum |a_k b_k| <= d 2^-24 ||rep_i|| max_j ||E_j||.  The exact
    entry's scores are fp32 products, so where a score is a cancellation of large terms (the x50 rows) its lse carries
    that much on top of the summation rounding."""
    return _eps(theta, rep, d, V) * d * 2.0 ** -12


def _run(d, theta, rep, gt, V, tc):
    from ader_b200 import ops
    ms, R = _ms(d), rep.shape[0]
    lse = torch.full((R,), float("nan"), device="cuda")
    nll = torch.full((R,), float("nan"), device="cuda") if gt is not None else None
    if tc:
        ws = torch.empty(ops.logsumexp_tc_ws_bytes(ms, R, V), dtype=torch.uint8, device="cuda")
        ops.logsumexp_tc(ms, theta, rep, gt, V, ws, lse, nll)
    else:
        ws = torch.empty(ops.eval_ws_bytes(ms, R, V), dtype=torch.uint8, device="cuda")
        ops.logsumexp(ms, theta, rep, gt, V, ws, lse, nll)
    return lse.cpu().numpy(), (nll.cpu().numpy() if nll is not None else None)


# ---- 1. bounds against the fp64 oracle -----------------------------------------------------------------------------------
VS = [1, 33, 64, 127, 129, 18661, 43105]
RS = [1, 127, 129, 4096]


@pytest.mark.parametrize("d", [2, 64, 150, 160, 192, 256])
def test_both_entries_within_their_bounds(d):
    from ader_b200 import _lib, ops
    theta = _theta(d)
    for V in VS:
        for R in RS:
            rep, gt = _reps(R, d), _gt(R, V)
            want_lse, want_nll = _oracle(theta, rep, gt, d, V)
            lse, nll = _run(d, theta, rep, gt, V, tc=False)
            tol = 1e-5 * (1 + np.abs(want_lse)) + _fp32_dot(theta, rep, d, V)
            assert (np.abs(lse - want_lse) <= tol).all(), ("exact lse", d, V, R, np.abs(lse - want_lse).max())
            assert (np.abs(nll - want_nll) <= tol).all(), ("exact nll", d, V, R, np.abs(nll - want_nll).max())
            assert abs(lse[0] - np.log(V)) <= 1e-6 * (1 + np.log(V))
            lse2, nll2 = _run(d, theta, rep, None, V, tc=False)
            assert np.array_equal(lse2, lse) and nll2 is None
            if d > 160:                                   # the tc entry refuses, before it writes anything
                ms = _ms(d)
                assert ops.path_check(ms, ops.PATH_EVAL_TC) is not None
                with pytest.raises(_lib.AderError, match="logsumexp_tc_ws_bytes"):
                    ops.logsumexp_tc_ws_bytes(ms, R, V)
                out = torch.full((R,), 7.0, device="cuda")
                n_out = torch.full((R,), 7.0, device="cuda")
                fake_ws = torch.empty(16, dtype=torch.uint8, device="cuda")
                with pytest.raises(_lib.AderError, match="hidden_units <= 160"):
                    ops.logsumexp_tc(ms, theta, rep, gt, V, fake_ws, out, n_out)
                assert bool((out == 7.0).all()) and bool((n_out == 7.0).all())
                continue
            eps = _eps(theta, rep, d, V)
            lse_t, nll_t = _run(d, theta, rep, gt, V, tc=True)
            assert (np.abs(lse_t - want_lse) <= eps + 1e-5).all(), ("tc lse", d, V, R, np.abs(lse_t - want_lse).max())
            assert (np.abs(nll_t - want_nll) <= eps + 1e-5).all(), ("tc nll", d, V, R, np.abs(nll_t - want_nll).max())
            assert abs(lse_t[0] - np.log(V)) <= 1e-5
            np.testing.assert_array_equal(nll_t, lse_t - _gt_score(theta, rep, gt, d))
            lse_t2, nll_t2 = _run(d, theta, rep, gt, V, tc=True)      # deterministic: same bits on a second call
            assert np.array_equal(lse_t2.view(np.int32), lse_t.view(np.int32))
            assert np.array_equal(nll_t2.view(np.int32), nll_t.view(np.int32))
            lse_t3, _ = _run(d, theta, rep, None, V, tc=True)         # without gt: the same normaliser
            assert np.array_equal(lse_t3.view(np.int32), lse_t.view(np.int32))


def _gt_score(theta, rep, gt, d):
    """the exact fp32 ground-truth score (ader_logits, the fmaf chain the tc entry's anchor uses)"""
    from ader_b200 import ops
    R = rep.shape[0]
    V = int(gt.max().item())
    out = torch.empty((R, (V + 3) // 4 * 4), device="cuda")
    ops.logits(_ms(d), theta, rep, V, out)
    return out.gather(1, (gt.long() - 1)[:, None])[:, 0].cpu().numpy()


def test_exact_nll_equals_the_training_row_loss():
    """dropout 0, mode 0, pos = gt: ader_loss_fwd_bwd's row_loss is the same cross-entropy"""
    from ader_b200 import ops
    d, V, R = 150, 18661, 300
    theta, rep, gt = _theta(d), _reps(R, d), _gt(R, V)
    _, nll = _run(d, theta, rep, gt, V, tc=False)
    ms = _ms(d)
    a = ops.make_loss_args(R, R, 0, V, pos=gt)
    ws = torch.empty(ops.loss_ws_bytes(ms, a), dtype=torch.uint8, device="cuda")
    loss = torch.empty(1, device="cuda")
    row_loss = torch.empty(R, device="cuda")
    ops.loss_fwd_bwd(ms, theta, rep, a, ws, loss, row_loss, None, None)
    np.testing.assert_allclose(nll, row_loss.cpu().numpy(), rtol=1e-5, atol=1e-6)


def test_torch_ops_give_the_same_bits():
    from ader_b200 import ops
    ops.register_torch_ops()
    d, V, R = 150, 18661, 200
    theta, rep, gt = _theta(d), _reps(R, d), _gt(R, V)
    model = [ITEMS + 1, d, 50, 1, 1]
    for name, tc in (("logsumexp", False), ("logsumexp_tc", True)):
        ws_n = ops.logsumexp_tc_ws_bytes(_ms(d), R, V) if tc else ops.eval_ws_bytes(_ms(d), R, V)
        ws = torch.empty(ws_n, dtype=torch.uint8, device="cuda")
        lse, nll = torch.empty(R, device="cuda"), torch.empty(R, device="cuda")
        getattr(torch.ops.ader_b200, name)(model, theta, rep, gt, V, ws, lse, nll)
        want = _run(d, theta, rep, gt, V, tc)
        assert np.array_equal(lse.cpu().numpy().view(np.int32), want[0].view(np.int32))
        assert np.array_equal(nll.cpu().numpy().view(np.int32), want[1].view(np.int32))
        getattr(torch.ops.ader_b200, name)(model, theta, rep, None, V, ws, lse, None)
        assert np.array_equal(lse.cpu().numpy().view(np.int32), want[0].view(np.int32))


# ---- 2. the model surface ------------------------------------------------------------------------------------------------
def _args(**kw):
    base = dict(hidden_units=150, maxlen=50, num_blocks=2, num_heads=1, random_seed=0, lr=5e-4,
                dropout_rate=0.0, disable_distillation=False, loss_impl="exact")
    base.update(kw)
    return type("Args", (), base)()


def _model(item_num, seed=1, scale=0.05, **kw):
    from ader_b200.model import Ader
    args = _args(**kw)
    m = Ader(item_num, args, init_seed=0)
    hp = S.Hyper(item_num, args.hidden_units, args.maxlen, args.num_blocks, args.num_heads)
    params = S.randomize_params(S.init_params(hp, 0), seed, scale)
    m.theta.copy_(torch.cat([p.reshape(-1) for p in params]))
    return m


def _sessions(rng, R, L, item_max):
    ids = np.zeros((R, L), np.int32)
    for r in range(R):
        n = int(rng.randint(1, L + 1))
        ids[r, L - n:] = rng.randint(1, item_max + 1, n)
    return ids


def test_rank_topk_nll_leaves_ranks_and_lists_unchanged():
    m = _model(3000)
    V, R = 2900, 700
    rng = np.random.RandomState(5)
    ids, gt = _sessions(rng, R, 50, V), rng.randint(1, V + 1, R).astype(np.int32)
    for force in (False, True):
        r0, i0, s0 = m.rank_topk(ids, gt, V, 20, force_exact=force)
        nll = torch.full((R,), float("nan"), device="cuda")
        r1, i1, s1 = m.rank_topk(ids, gt, V, 20, force_exact=force, nll=nll)
        assert torch.equal(r0, r1) and torch.equal(i0, i1) and torch.equal(s0, s1)
        rep = m.rep(ids)
        lse, want = m.logsumexp(rep, V, gt, force_exact=force)
        assert torch.equal(nll, want)
        o_lse, o_nll = _oracle(m.theta, rep, torch.from_numpy(gt).cuda(), 150, V)
        eps = _eps(m.theta, rep, 150, V)
        assert (np.abs(nll.cpu().numpy() - o_nll) <= eps + 1e-5).all()


def test_recommend_probabilities():
    m = _model(3000)
    V, R, k = 2900, 300, 50
    rng = np.random.RandomState(6)
    ids = _sessions(rng, R, 50, V)
    ids[7, :] = 0
    ids[7, -1] = 5
    rep = m.rep(ids)
    lg = m.logits(rep, V)
    out = {}
    for force in (False, True):
        items, scores = m.recommend(ids, V, k, force_exact=force)
        items_p, probs = m.recommend(ids, V, k, force_exact=force, probs=True)
        assert torch.equal(items, items_p)
        lse = m.logsumexp(rep, V, force_exact=force)[0]
        assert torch.equal(probs, torch.exp(scores - lse[:, None]))
        total = torch.exp(lg.double() - lse.double()[:, None]).sum(dim=1)
        tol = 1e-5 + (0 if force else 1.01 * float(np.max(_eps(m.theta, rep, 150, V))))
        assert float((total - 1).abs().max()) <= tol
        out[force] = (probs.cpu().numpy(), _eps(m.theta, rep, 150, V))
    # tensor-core and exact probabilities: p_tc / p_exact = exp(lse_exact - lse_tc), within exp(+-eps)
    (p_tc, eps), (p_ex, _) = out[False], out[True]
    assert (np.abs(p_tc - p_ex) <= p_ex * (np.expm1(eps[:, None] + 1e-5)) + 1e-12).all()
    # padding (item 0, score -inf) gives 0
    _, probs = m.recommend(ids[:3], 3, 5, exclude_seen=False, probs=True)
    assert torch.equal(probs[:, 3:], torch.zeros_like(probs[:, 3:]))
    assert float((probs[:, :3].sum(dim=1) - 1).abs().max()) <= 1e-5 + 1.01 * float(np.max(eps))


# ---- 3. end to end ------------------------------------------------------------------------------------------------------
def _e2e_args(tmp, **kw):
    from ader_b200.main import build_parser
    a = build_parser().parse_args([])
    a.dataset = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "tiny_data")
    a.results_root = str(tmp)
    a.item_num = 700
    a.batch_size, a.test_batch, a.exemplar_size, a.num_epochs, a.stop = 64, 16, 150, 3, 5
    a.max_periods = 1
    a.dropout_rate = 0.0
    a.loss_impl = "exact"
    a.selection = "random"
    a.trace = True
    for k, v in kw.items():
        setattr(a, k, v)
    return a


def _epoch_lines(path):
    return [l for l in open(path).read().splitlines() if l.startswith("epoch:")]


def test_main_eval_nll_records_the_oracle_cross_entropy(tmp_path):
    from ader_b200.data import DataLoader, Sampler
    from ader_b200.main import CKPT_NAME, run
    a = _e2e_args(tmp_path / "off")
    off = run(a)
    b = _e2e_args(tmp_path / "on", eval_nll=True)
    on = run(b)
    po, pn = off["trace"]["periods"][0], on["trace"]["periods"][0]
    assert po["valid"] == pn["valid"] and po["test"] == pn["test"] and po["test_ranks"] == pn["test_ranks"]
    assert "test_nll" not in po and "valid_nll" not in po and "NLL" not in off["per_period"]
    assert len(pn["valid_nll"]) == len(pn["valid"]) and on["per_period"]["NLL"] == [pn["test_nll"]]
    log_off = _epoch_lines(os.path.join(str(tmp_path / "off"), "tiny_data-ADER", "Training_logs.txt"))
    log_on = _epoch_lines(os.path.join(str(tmp_path / "on"), "tiny_data-ADER", "Training_logs.txt"))
    assert all(" NLL: " not in l for l in log_off)
    assert all(" NLL: " in l for l in log_on)
    assert [l.split(" NLL: ")[0] for l in log_on] == log_off
    # the recorded test NLL is the oracle's mean cross-entropy of the period's test rows at the restored best epoch
    m = on["model"]
    dl = DataLoader(b.dataset)
    dl.train_loader(0)                                    # the items known after period 1's training data, as in main.run
    test_sess, _ = dl.evaluate_loader(1)
    ids, label, n_in = Sampler(test_sess, b.maxlen, b.test_batch).packed()
    keep = n_in > 0
    assert keep.sum() == len(pn["test_ranks"])
    rep = m.rep(ids[keep])
    V = int(off["throughput"][0]["max_item"])
    _, o_nll = _oracle(m.theta, rep, torch.from_numpy(label[keep]).cuda(), b.hidden_units, V)
    eps = _eps(m.theta, rep, b.hidden_units, V)
    assert abs(pn["test_nll"] - o_nll.mean()) <= eps.mean() + 1e-5
    assert abs(float(log_on[-1].split(" NLL: ")[1]) - o_nll.mean()) <= eps.mean() + 1e-4
    # the recommend command writes probabilities from that run's checkpoint
    ckpt = os.path.join(str(tmp_path / "on"), "tiny_data-ADER", CKPT_NAME)
    rng = np.random.RandomState(4)
    sessions = [list(rng.randint(1, 701, int(n))) for n in rng.randint(1, 60, 40)]
    sess_file = tmp_path / "sessions.txt"
    sess_file.write_text("".join(" ".join(map(str, s)) + "\n" for s in sessions))
    out = tmp_path / "probs.txt"
    env = dict(os.environ, PYTHONPATH=ROOT)
    subprocess.run([sys.executable, "-m", "ader_b200.recommend", "--checkpoint", ckpt, "--sessions", str(sess_file),
                    "--out", str(out), "--probs", "--k", "10"], check=True, cwd=ROOT, env=env)
    from ader_b200.recommend import load_model, recommend_sessions
    restored, max_item = load_model(ckpt)
    items, probs = recommend_sessions(restored, sessions, max_item, 10, probs=True)
    lines = out.read_text().splitlines()
    assert len(lines) == len(sessions)
    for r, line in enumerate(lines):
        toks = line.split()
        assert [int(t.split(":")[0]) for t in toks] == items[r].tolist()
        p = np.array([np.float32(t.split(":")[1]) for t in toks])
        assert np.array_equal(p.view(np.int32), probs[r].view(np.int32))
        assert (p > 0).all() and p.sum() <= 1 + 1e-5 and (np.diff(p) <= 0).all()


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def _rows():
    rng = np.random.RandomState(9)
    return [list(rng.randint(1, 381, int(n))) for n in rng.randint(2, 30, 500)]


def _evaluate(m, dp=None):
    from ader_b200.data import Evaluator
    random.seed(0)
    ev = Evaluator(_rows(), True, 50, 64, 380, "test", m, None, dp=dp, nll=True)
    ev.evaluate(1)
    return np.asarray(ev.ranks), ev.nll


def _dp_worker(rank, world, port, out, impl):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from ader_b200.model import Ader
        m = Ader(400, _args(eval_impl=impl), device=torch.device("cuda", rank), init_seed=0)
        m.theta.add_(torch.randn(m.theta.shape, generator=torch.Generator().manual_seed(1)).to(m.device) * 0.05)
        out[rank] = _evaluate(m, dp=(rank, world))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("impl", ["exact", "tc"])
def test_data_parallel_evaluation_gives_the_single_rank_nll(impl):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from ader_b200.model import Ader
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_dp_worker, args=(2, _free_port(), out, impl), nprocs=2, join=True)
    m = Ader(400, _args(eval_impl=impl), init_seed=0)
    m.theta.add_(torch.randn(m.theta.shape, generator=torch.Generator().manual_seed(1)).to(m.device) * 0.05)
    ranks, nll = _evaluate(m)
    for r in range(2):
        assert np.array_equal(out[r][0], ranks)
        if impl == "exact":                    # every row's value is independent of the batch it is in
            assert np.array_equal(out[r][1].view(np.int32), nll.view(np.int32))
        else:                                  # the chunk count follows the shard's row count: within the bound
            np.testing.assert_allclose(out[r][1], nll, rtol=0, atol=1e-3)
