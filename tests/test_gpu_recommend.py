"""Recommendation on the GPU: ader_recommend_topk (exact fp32 scores + row selection) against a stable (-score, id) sort of
``ader_logits``, ader_recommend_topk_tc against the exact entry bit for bit (ids and scores), the overflow fallback of
``Ader.recommend``, padding, agreement with the evaluation top-k lists, the torch ops, and the command end to end."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import sasrec as S

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


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


def _sessions(rng, R, L, item_max, max_len=None):
    """left-padded id rows; lengths 1..max_len (some rows repeat an item)"""
    ids = np.zeros((R, L), np.int32)
    lens = rng.randint(1, (max_len or L) + 1, R)
    for r in range(R):
        n = int(lens[r])
        row = rng.randint(1, item_max + 1, n)
        if n > 2 and r % 3 == 0:
            row[0] = row[-1]
        ids[r, L - n:] = row
    return ids


def _ref_topk(lg, ids, k, exclude):
    """stable sort by (-score, id) of the eligible columns of every row, padded with 0 / -inf"""
    R, V = lg.shape
    items = np.zeros((R, k), np.int32)
    scores = np.full((R, k), -np.inf, np.float32)
    for i in range(R):
        ok = np.ones(V, bool)
        if exclude:
            seen = ids[i][(ids[i] >= 1) & (ids[i] <= V)]
            ok[seen - 1] = False
        cols = np.nonzero(ok)[0]
        s = lg[i, cols]
        top = cols[np.lexsort((cols, -s))][:k]
        items[i, :len(top)] = top + 1
        scores[i, :len(top)] = lg[i, top]
    return items, scores


def _run(m, rep, ids_t, V, k, tc):
    from ader_b200 import ops
    R = rep.shape[0]
    items = torch.empty((R, k), dtype=torch.int32, device=m.device)
    scores = torch.empty((R, k), dtype=torch.float32, device=m.device)
    if tc:
        ws = torch.empty(ops.recommend_tc_ws_bytes(m.ms, R, V), dtype=torch.uint8, device=m.device)
        over = torch.full((1,), -7, dtype=torch.int32, device=m.device)
        ops.recommend_topk_tc(m.ms, m.theta, rep, ids_t, V, k, ws, items, scores, over)
        return items.cpu().numpy(), scores.cpu().numpy(), int(over.item())
    ws = torch.empty(ops.eval_ws_bytes(m.ms, R, V), dtype=torch.uint8, device=m.device)
    ops.recommend_topk(m.ms, m.theta, rep, ids_t, V, k, ws, items, scores)
    return items.cpu().numpy(), scores.cpu().numpy(), 0


def _same(a, b):
    assert np.array_equal(a[0], b[0])
    assert np.array_equal(a[1].view(np.int32), b[1].view(np.int32))      # bitwise, -inf padding included


# ---- 1. the exact entry against ader_logits ----------------------------------------------------------------------------
@pytest.mark.parametrize("exclude", [False, True], ids=["all", "exclude_seen"])
def test_exact_entry_equals_sorted_logits(exclude):
    rng = np.random.RandomState(3)
    m = _model(2000)
    R, V, k = 200, 1900, 100
    ids = _sessions(rng, R, 50, 2000)                      # ids above V are in sessions too: never excluded, never returned
    rep = m.rep(ids)
    lg = m.logits(rep, V).cpu().numpy()
    got = _run(m, rep, torch.from_numpy(ids).cuda() if exclude else None, V, k, tc=False)
    _same(got, _ref_topk(lg, ids, k, exclude))
    if exclude:
        for i in range(R):
            assert not set(got[0][i]) & set(ids[i][ids[i] > 0])


# ---- 2. the tc entry against the exact entry, bit for bit ----------------------------------------------------------------
def _plant_twins(m, rep, ids, V, rows):
    """For each row in `rows`: give its top-1 item and its 5th item a bit-equal twin (a copy of the table row under another
    id), and put the top-1 item into the row's session, so with exclusion on its twin must come first."""
    d = m.hp.hidden_units
    table = m.theta[:m.hp.v_tab * d].view(m.hp.v_tab, d)
    lg = m.logits(rep, V).cpu().numpy()
    rng = np.random.RandomState(5)
    targets = {}
    for i in rows:
        order = np.lexsort((np.arange(V), -lg[i]))
        targets[i] = (int(order[0]) + 1, int(order[4]) + 1)
    used = {t for pair in targets.values() for t in pair}   # a twin never overwrites another row's target
    for i in rows:
        for t in targets[i]:
            while True:
                w = int(rng.randint(1, V + 1))
                if w not in used and w not in ids[i]:
                    break
            used.add(w)
            table[w] = table[t]
        ids[i, 0] = targets[i][0]                          # rows are shorter than maxlen: column 0 is padding
    return {i: targets[i][0] for i in rows}


SHAPES = [(37, 450), (300, 18661), (1500, 40135), (64, 43105)]


@pytest.mark.parametrize("R,V", SHAPES, ids=["%dx%d" % s for s in SHAPES])
def test_tc_entry_equals_exact_entry(R, V, monkeypatch):
    from ader_b200 import ops
    rng = np.random.RandomState(R)
    m = _model(V + 20)
    ids = _sessions(rng, R, 50, V + 20, max_len=40)
    rep = m.rep(ids).clone()
    rows = list(range(0, R, max(1, R // 12)))
    tops = _plant_twins(m, rep, ids, V, rows)
    ids_t = torch.from_numpy(ids).cuda()
    nc = ops.eval_topk_chunks(m.ms, R, V)
    for k in (1, 20, 50, 100):
        for exclude in (False, True):
            seen = ids_t if exclude else None
            want = _run(m, rep, seen, V, k, tc=False)
            if 16 * nc >= k:
                got = _run(m, rep, seen, V, k, tc=True)
                assert got[2] == 0, (k, exclude)           # no overflow at these shapes
                _same(got, want)
            if exclude:
                assert all(tops[i] not in want[0][i] for i in rows)
    # routing of Ader.recommend: the tc entry exactly where 16 * chunks >= k, never a fallback
    calls = []
    real = ops.recommend_topk_tc
    monkeypatch.setattr(ops, "recommend_topk_tc", lambda *a: (calls.append(a[5]), real(*a))[1])
    for k in (1, 20, 50, 100):
        calls.clear()
        items, scores = m.recommend(ids, V, k)
        assert calls == ([k] if 16 * nc >= k else [])
        _same((items.cpu().numpy(), scores.cpu().numpy()), _run(m, m.rep(ids), ids_t, V, k, tc=False))
    assert m.eval_fallbacks == 0
    if R == 37:
        assert nc == 1                                     # k > 16 went to the exact entry above


def test_excluded_top1_twin_is_returned():
    rng = np.random.RandomState(11)
    R, V = 300, 18661
    m = _model(V)
    ids = _sessions(rng, R, 50, V, max_len=30)
    rep = m.rep(ids).clone()
    lg_before = m.logits(rep, V).cpu().numpy()
    rows = list(range(0, R, 7))
    tops = _plant_twins(m, rep, ids, V, rows)
    ids_t = torch.from_numpy(ids).cuda()
    got = _run(m, rep, ids_t, V, 20, tc=True)
    assert got[2] == 0
    _same(got, _run(m, rep, ids_t, V, 20, tc=False))
    for i in rows:
        t = tops[i]
        assert got[0][i, 0] != t and got[1][i, 0] == lg_before[i, t - 1]   # the twin of the excluded top-1 leads the list
        assert t not in got[0][i]


# ---- 3. overflow ---------------------------------------------------------------------------------------------------------
def test_overflow_falls_back_to_the_exact_entry():
    rng = np.random.RandomState(2)
    R, V = 256, 18661
    m = _model(V)
    ids = _sessions(rng, R, 50, V, max_len=20)
    rep = m.rep(ids).clone()
    lg = m.logits(rep, V).cpu().numpy()
    t = int(np.argmax(lg[0])) + 1
    d = m.hp.hidden_units
    table = m.theta[:m.hp.v_tab * d].view(m.hp.v_tab, d)
    # 300 twins outside row 0's session (its rep stays as it is): more than 256 bit-equal items on top of row 0
    twins = rng.choice(np.setdiff1d(np.arange(1, V + 1), np.concatenate([[t], ids[0]])), 300, replace=False)
    table[torch.from_numpy(twins).long().cuda()] = table[t].clone()
    ids_t = torch.from_numpy(ids).cuda()
    got = _run(m, rep, ids_t, V, 50, tc=True)
    assert got[2] != 0
    want = _run(m, rep, ids_t, V, 50, tc=False)
    assert len(set(want[1][0].tolist())) == 1
    items, scores = m.recommend(ids, V, 50)
    assert m.eval_fallbacks == 1
    assert np.array_equal(items[0].cpu().numpy(), want[0][0])
    ex_items, ex_scores = m.recommend(ids, V, 50, force_exact=True)
    _same((items.cpu().numpy(), scores.cpu().numpy()), (ex_items.cpu().numpy(), ex_scores.cpu().numpy()))


# ---- 4. padding ----------------------------------------------------------------------------------------------------------
def test_rows_with_few_eligible_items_are_padded():
    V, k = 40, 10
    m = _model(60)
    ids = np.zeros((3, 50), np.int32)
    ids[0, 50 - V:] = np.arange(1, V + 1)                 # every item seen
    ids[1, 50 - (V - 3):] = np.arange(4, V + 1)           # items 1..3 left
    ids[2, -3:] = [5, 6, 55]                              # an id above V: ignored
    rep = m.rep(ids)
    ids_t = torch.from_numpy(ids).cuda()
    want = _run(m, rep, ids_t, V, k, tc=False)
    got = _run(m, rep, ids_t, V, k, tc=True)
    assert got[2] == 0
    _same(got, want)
    assert (want[0][0] == 0).all() and np.isneginf(want[1][0]).all()
    assert sorted(want[0][1, :3]) == [1, 2, 3] and (want[0][1, 3:] == 0).all() and np.isneginf(want[1][1, 3:]).all()
    assert np.isfinite(want[1][2]).all()
    lg = m.logits(rep, V).cpu().numpy()
    _same(want, _ref_topk(lg, ids, k, True))


# ---- 5. agreement with evaluation ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 20, 32])
def test_lists_equal_rank_topk(k):
    rng = np.random.RandomState(k)
    R, V = 700, 40135
    m = _model(V)
    ids = _sessions(rng, R, 50, V)
    gt = rng.randint(1, V + 1, R).astype(np.int32)
    _, ev_items, ev_scores = m.rank_topk(ids, gt, V, k)
    items, scores = m.recommend(ids, V, k, exclude_seen=False)
    _same((items.cpu().numpy(), scores.cpu().numpy()), (ev_items.cpu().numpy(), ev_scores.cpu().numpy()))


# ---- 6. torch ops --------------------------------------------------------------------------------------------------------
def test_torch_ops_equal_ctypes_calls():
    from ader_b200 import ops
    ops.register_torch_ops()
    rng = np.random.RandomState(9)
    R, V, k = 300, 18661, 40
    m = _model(V)
    ids = _sessions(rng, R, 50, V)
    rep = m.rep(ids)
    ids_t = torch.from_numpy(ids).cuda()
    model = [m.hp.v_tab, m.hp.hidden_units, m.hp.maxlen, m.hp.num_blocks, m.hp.num_heads]
    for seen in (ids_t, None):
        items = torch.empty((R, k), dtype=torch.int32, device="cuda")
        scores = torch.empty((R, k), dtype=torch.float32, device="cuda")
        ws = torch.empty(ops.eval_ws_bytes(m.ms, R, V), dtype=torch.uint8, device="cuda")
        torch.ops.ader_b200.recommend_topk(model, m.theta, rep, seen, V, k, ws, items, scores)
        _same((items.cpu().numpy(), scores.cpu().numpy()), _run(m, rep, seen, V, k, tc=False))
        ws = torch.empty(ops.recommend_tc_ws_bytes(m.ms, R, V), dtype=torch.uint8, device="cuda")
        over = torch.zeros(1, dtype=torch.int32, device="cuda")
        torch.ops.ader_b200.recommend_topk_tc(model, m.theta, rep, seen, V, k, ws, items, scores, over)
        assert int(over.item()) == 0
        _same((items.cpu().numpy(), scores.cpu().numpy()), _run(m, rep, seen, V, k, tc=True))


# ---- 7. the command end to end -------------------------------------------------------------------------------------------
def _e2e_args(tmp, **kw):
    from ader_b200.main import build_parser
    a = build_parser().parse_args([])
    a.dataset = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "tiny_data")
    a.results_root = str(tmp)
    a.item_num = 700
    a.batch_size, a.test_batch, a.exemplar_size, a.num_epochs, a.stop = 64, 16, 150, 3, 5
    a.max_periods = 3
    a.dropout_rate = 0.0
    a.loss_impl = "exact"
    for k, v in kw.items():
        setattr(a, k, v)
    return a


def test_command_writes_the_lists_of_the_restored_model(tmp_path):
    from ader_b200.main import CKPT_NAME, run
    from ader_b200.model import Ader
    from ader_b200.recommend import recommend_sessions
    a = _e2e_args(tmp_path / "run", selection="random")
    run(a)
    ckpt = os.path.join(str(tmp_path / "run"), "tiny_data-" + a.save_dir, CKPT_NAME)
    st = torch.load(ckpt, map_location="cpu", weights_only=False)
    max_item = int(max(st["item_set"]))
    rng = np.random.RandomState(4)
    sessions = [list(rng.randint(1, 701, int(n))) for n in rng.randint(1, 80, 150)]    # some longer than maxlen
    sessions[3] = list(range(1, 51))
    sess_file = tmp_path / "sessions.txt"
    sess_file.write_text("".join(" ".join(map(str, s)) + "\n" for s in sessions))
    restored = Ader(700, _args(), init_seed=0)
    restored.theta.copy_(st["model"]["theta"].cuda())
    env = dict(os.environ, PYTHONPATH=ROOT)
    for extra, k, keep in ((["--scores"], 20, False), (["--keep_seen", "--k", "100", "--batch", "37"], 100, True)):
        out = tmp_path / "topk.txt"
        subprocess.run([sys.executable, "-m", "ader_b200.recommend", "--checkpoint", ckpt, "--sessions", str(sess_file),
                        "--out", str(out), *extra], check=True, cwd=ROOT, env=env)
        items, scores = recommend_sessions(restored, sessions, max_item, k, exclude_seen=not keep)
        lines = out.read_text().splitlines()
        assert len(lines) == len(sessions)
        for r, line in enumerate(lines):
            toks = line.split()
            assert len(toks) == k
            if "--scores" in extra:
                assert [int(t.split(":")[0]) for t in toks] == items[r].tolist()
                assert np.array_equal(np.array([np.float32(t.split(":")[1]) for t in toks]).view(np.int32), scores[r].view(np.int32))
            else:
                assert [int(t) for t in toks] == items[r].tolist()
            if not keep:
                assert not set(items[r]) & set(sessions[r][-50:])
        assert (items <= max_item).all()
