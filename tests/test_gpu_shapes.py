"""Every kernel path at the edges of the model shapes the library accepts, against the fp64 oracle.

Each case below sits on one boundary of a kernel: the 160-column padding of the fused encoder / tcgen05 loss / tcgen05
evaluation / on-chip herding (KP = HALF = 160), the second K chunk of the fp32 GEMM (d > 160), the 8-token tiles of the
fused attention, the head dims of its multi-head branch, the shared-memory tiles of the exact attention kernels (their
thresholds are the formulas of tests/test_shape_contract.py) and the 64-wide exclusion lists of recommendation.  Every
path that ader_path_check says serves the case is compared with oracle/sasrec.py run on the same parameters cast to
float64; every path it refuses must refuse before any launch, and inference must still work afterwards.

Tolerances are those of the rest of the suite: exact fp32 path 3e-5 * max|x| (+1e-6 on representations, 2e-7 on
gradients); fused encoder representations ACT_TOL = 1e-2; default tensor-core training per tensor rel-L2 <= 3e-2 and
max-abs <= 0.15 max|g|; ranks, top-k lists and herding picks exact except at near-ties below 1e-5; Fisher 1e-4 relative.
Training batches have 256 or 320 rows: the bounds of the tensor-core path come from the baseline-shape test (385 and
650 rows), and at 32-40 rows the rounding noise of tensors summed over few tokens (early position-table rows, LayerNorm
gains, W1) alone reached rel-L2 3.3e-2 to 4.2e-2 at four shapes, the control shape not among them.  The oracle stays cheap:
about a second per case.  Each case prints, per check, the share of its tolerance the worst element used (rel-L2 for the fused gradients).
"""
import math
import time

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import protocol as P
from oracle import sasrec as S

ITEMS = 5300            # item table rows - 1
V_TRAIN = 480           # max_item of the training steps
V_PREV = 400            # teacher width of the distillation cases
V_EVAL = 5200           # max_item of evaluation / recommendation: 82 column tiles, 10 vocabulary chunks (top-20 on tcgen05)
ACT_TOL, GRAD_L2_TOL, GRAD_TOL = 1e-2, 3e-2, 0.15

# (hidden_units, maxlen, num_heads, num_blocks, loss mode of the training check, boundary)
CASES = [
    (150, 50, 1, 2, "vanilla", "control"),
    (160, 50, 1, 2, "kd_frozen", "d = KP, no pad column"),
    (160, 64, 10, 1, "kd_stored", "KP at the largest maxlen, head dim 16; exact backward refused"),
    (64, 64, 4, 2, "kd_frozen", "largest maxlen, served by both backwards"),
    (136, 64, 2, 1, "er", "last d the exact backward takes at maxlen 64"),
    (138, 64, 1, 1, "vanilla", "first d the exact backward refuses at maxlen 64"),
    (48, 33, 3, 2, "kd_stored", "maxlen not a multiple of 4 or 8"),
    (150, 63, 6, 1, "er", "odd head dim 25"),
    (152, 9, 19, 1, "vanilla", "head dim 8"),
    (2, 8, 2, 1, "kd_stored", "smallest d, head dim 1"),
    (32, 1, 1, 1, "er", "maxlen 1"),
    (64, 20, 2, 8, "vanilla", "8 blocks"),
    # found here: the LayerNorm-parameter and position-table reductions of the exact backward launched ceil32(d) x 6
    # threads, over 1024 from d = 161 on, so no model wider than 160 could train; above 160 they now use 4 token lanes
    (162, 50, 1, 2, "kd_frozen", "just above KP: a second, 2-wide K chunk of the fp32 GEMM"),
    (190, 50, 2, 1, "er", "last d trainable at maxlen 50"),
    (256, 40, 8, 1, "kd_stored", "widest trainable model"),
    (256, 64, 8, 1, None, "inference only: the exact forward fills its 200 KB exactly"),
]
HERDING_D = (32, 160, 162, 256)          # second-generation form at d <= 160, first-generation form above


def _args(d, L, h, nb, **kw):
    base = dict(hidden_units=d, maxlen=L, num_blocks=nb, num_heads=h, random_seed=0, lr=5e-4, dropout_rate=0.0,
                disable_distillation=False)
    base.update(kw)
    return type("Args", (), base)()


def _model(d, L, h, nb, seed=1, scale=0.02, **kw):
    """Ader at the given shape with default flags (+ kw) and randomised weights; the oracle's fp64 copy of the weights.
    The weight scale is that of test_default_tc_path_matches_oracle_at_baseline_shapes, whose bounds the fused path uses."""
    from ader_b200.model import Ader
    m = Ader(ITEMS, _args(d, L, h, nb, **kw), init_seed=0)
    hp = S.Hyper(ITEMS, d, L, nb, h)
    params = S.randomize_params(S.init_params(hp, 0), seed, scale)
    m.theta.copy_(torch.cat([p.reshape(-1) for p in params]))
    return m, hp, [p.double() for p in params]


def _ids(rng, L, M, item_max, empty=False, full_row=False):
    """Left-padded sessions: rows of length 1, L and L - 1, one row repeating an item, a hot item (item 11) in a third of
    the rows (a long scatter segment), random lengths elsewhere; optionally an empty row and a row of L distinct items."""
    lens = [1, L, max(L - 1, 1)] + list(rng.randint(1, L + 1, M - 3))
    ids = np.zeros((M, L), np.int32)
    for r, n in enumerate(lens):
        ids[r, L - n:] = rng.randint(1, item_max + 1, n)
    if L >= 3:
        ids[3, L - 3:] = [17, 23, 17]
        ids[4, :] = 0
        ids[4, L - min(L, 6):] = 29                                     # one item over a whole session
    hot = rng.rand(M) < 0.35
    ids[hot, -1] = 11
    if full_row:
        ids[5] = np.arange(1, L + 1, dtype=np.int32) * 7                 # L distinct items: fills the exclusion list
    if empty:
        ids[-1] = 0
    return ids


def _close(got, want, rel, abs_, what):
    got, want = torch.as_tensor(got).double(), torch.as_tensor(want).double()
    scale = float(want.abs().max()) if want.numel() else 0.0
    err = float((got - want).abs().max()) if want.numel() else 0.0
    tol = rel * scale + abs_
    assert err <= tol, "%s: max err %.3e (scale %.3e, tol %.3e)" % (what, err, scale, tol)
    return err / tol                 # share of the tolerance used


def _views(m, flat):
    return [v.detach().cpu() for v in m.layout.views(flat)]


def _herding_gap(rep, m, picks, k):
    """top-1/top-2 gap of w.D at the step that produced the k-th unique pick (fp64 replay)."""
    D = (rep.T / np.linalg.norm(rep.T, axis=0)).astype(np.float64)
    mu = D.mean(axis=1); w = mu.copy(); sel = []
    for _ in range(int(math.ceil(1.1 * m))):
        s = w @ D
        i = int(np.argmax(s))
        if len(sel) == k and i not in sel:
            t = np.sort(s)
            return float(t[-1] - t[-2])
        w = w + mu - D[:, i]
        if i not in sel:
            sel.append(i)
    return 0.0


def _ref_topk(lg, ids, k):
    """stable (-score, id) sort of the columns not among the row's own items"""
    R, V = lg.shape
    items = np.zeros((R, k), np.int32)
    scores = np.zeros((R, k), np.float32)
    for i in range(R):
        ok = np.ones(V, bool)
        seen = ids[i][(ids[i] >= 1) & (ids[i] <= V)]
        ok[seen - 1] = False
        cols = np.nonzero(ok)[0]
        top = cols[np.lexsort((cols, -lg[i, cols]))][:k]
        items[i] = top + 1
        scores[i] = lg[i, top]
    return items, scores


def _blocks_behind(name, nb):
    """Encoder blocks the data gradient crosses before it reaches tensor `name`.  The fused backward rounds that gradient
    to row-scaled fp16 operands in every block, so independent rounding errors add up in quadrature over the blocks behind
    a weight: its rel-L2 bound is GRAD_L2_TOL * sqrt(blocks / 2), the bound itself at the 2 blocks it was set for.  Found
    here: at 8 blocks the W1 gradient of block 0 reached rel-L2 3.07e-2 (max-abs 0.07 max|g|, well inside its bound)."""
    if name.startswith("b") and "." in name and name.split(".")[0][1:].isdigit():
        return nb - int(name.split(".")[0][1:])
    return 0 if name.startswith("lnf") else nb


def _served(ms, path):
    from ader_b200 import ops
    return ops.path_check(ms, path) is None


# ---- checks -----------------------------------------------------------------------------------------------------------
def _check_reps(m, hp, params, ids, log):
    """exact encoder vs the oracle (3e-5 * max|rep| + 1e-6); fused encoder (where served) within ACT_TOL"""
    from ader_b200 import ops
    live = ids.any(axis=1)
    want = S.forward_rep(params, torch.tensor(ids[live]).long(), hp)
    ids_t = torch.tensor(ids, device=m.device)
    rep_e = m.encode(ids_t, impl="exact")[0].clone()
    log["rep exact"] = _close(rep_e.cpu()[live], want, 3e-5, 1e-6, "exact rep")
    assert float(rep_e.cpu()[~torch.tensor(live)].abs().max()) == 0.0                 # empty row -> zeros
    if _served(m.ms, ops.PATH_ENCODER_TC):
        rep_t = m.encode(ids_t, impl="tc")[0].clone()
        log["rep fused"] = _close(rep_t.cpu()[live], want, ACT_TOL, 1e-6, "fused rep")
    return rep_e


def _loss_inputs(m, hp, params, mode, rng, L):
    """(ids, pos, loss_and_grad kwargs, oracle loss function) of one training batch in the given mode"""
    from ader_b200.data import FrozenTeacher
    M, n_ex = (256, 0) if mode == "vanilla" else (320, 96)
    ids = _ids(rng, L, M, V_TRAIN)
    n_train = M - n_ex
    pos = rng.randint(1, V_TRAIN + 1, n_train).astype(np.int32)
    pos[0], pos[-1] = 1, V_TRAIN
    ids_o, pos_o = torch.tensor(ids).long(), torch.tensor(pos)
    lam = 0.8
    if mode == "vanilla":
        return ids, pos, {}, lambda ps: S.loss_vanilla(ps, ids_o, pos_o, V_TRAIN, hp)
    m.disable_distillation = mode == "er"
    m.update_loss(lam)
    if mode == "er":
        ex_pos = rng.randint(1, V_TRAIN + 1, n_ex).astype(np.int32)
        return ids, pos, {"exemplar_pos": ex_pos}, \
            lambda ps: S.loss_ader(ps, ids_o, pos_o, V_TRAIN, hp, lam, exemplar_pos=torch.tensor(ex_pos))
    if mode == "kd_stored":
        teacher = (rng.randn(n_ex, V_PREV) * 2).astype(np.float32)
        return ids, pos, {"exemplar_logits": teacher}, \
            lambda ps: S.loss_ader(ps, ids_o, pos_o, V_TRAIN, hp, lam, exemplar_logits=torch.tensor(teacher).double())
    assert mode == "kd_frozen"
    prev, _, _ = _model(hp.hidden_units, L, hp.num_heads, hp.num_blocks, seed=7)          # the previous model
    ft = FrozenTeacher(prev, prev.rep(ids[n_train:]), V_PREV)
    teacher = ft.logits().cpu().double()                                                  # what the snapshot stands for
    return ids, pos, {"exemplar_logits": ft}, \
        lambda ps: S.loss_ader(ps, ids_o, pos_o, V_TRAIN, hp, lam, exemplar_logits=teacher)


def _check_grads(m, hp, params, ids, pos, kw, fn, what, log):
    ref, grads = S.grads_of(fn, params)
    loss = float(m.loss_and_grad(ids, pos, V_TRAIN, **kw).item())
    torch.cuda.synchronize()
    got = _views(m, m.grad)
    assert float(got[0][V_TRAIN + 1:].abs().max()) == 0.0, "%s: table rows > V received gradient" % what
    exact = m.encoder_impl == "exact"
    assert loss == pytest.approx(ref, rel=2e-5 if exact else 1e-3), what
    gscale = max(float(w.abs().max()) for w in grads)
    floor_ = 1e-5 * gscale        # tensors whose true gradient is identically zero (the key bias: softmax is shift invariant)
    worst = 0.0
    for i, (name, _) in enumerate(S.param_shapes(hp)):
        g, w = got[i].double(), grads[i].double()
        if i == 0:
            g, w = g[1:V_TRAIN + 1], w[1:V_TRAIN + 1]
        if exact:
            worst = max(worst, _close(g, w, 3e-5, 2e-7, "%s grad of %s" % (what, name)))
            continue
        rel = float((g - w).norm() / (w.norm() + floor_ * w.numel() ** 0.5))
        mx = float((g - w).abs().max() / (w.abs().max() + floor_))
        tol = GRAD_L2_TOL * math.sqrt(max(_blocks_behind(name, hp.num_blocks), 2) / 2)
        assert rel <= tol and mx <= GRAD_TOL, "%s grad of %s: rel-L2 %.3e, max-abs/max|g| %.3e" % (what, name, rel, mx)
        worst = max(worst, rel)
    log["grad %s" % what] = worst


def _check_eval(m, hp, params, rep_e, ids, log):
    """ranks / top-20 (tcgen05 where served, and exact) == the device logits' own; == the oracle's away from near-ties;
    recommendation with exclusion == the stable sort of the device logits with the session's items masked"""
    from ader_b200 import ops
    rng = np.random.RandomState(5)
    R = ids.shape[0]
    gt = rng.randint(1, V_EVAL + 1, R).astype(np.int32)
    gt[0], gt[1] = 1, V_EVAL
    lg_dev = m.logits(rep_e, V_EVAL).cpu().numpy()
    live = ids.any(axis=1)
    lg = S.logits_of(S.forward_rep(params, torch.tensor(ids[live]).long(), hp), params[0], V_EVAL).numpy()
    sg = lg[np.arange(len(lg)), gt[live] - 1]
    lonely = np.array([np.sum(np.abs(lg[i] - sg[i]) < 1e-5) == 1 for i in range(len(lg))])
    want_oracle = S.rank_of_gt(lg, gt[live])
    ref_items, ref_scores = _ref_topk(lg_dev, ids, 20)
    impls = ["tc", "exact"] if _served(m.ms, ops.PATH_EVAL_TC) else ["exact"]
    for impl in impls:
        m.eval_impl = impl
        fb = m.eval_fallbacks
        rank, items, _ = m.rank_topk(ids, gt, V_EVAL, 20, force_exact=(impl == "exact"))
        rank, items = rank.cpu().numpy(), items.cpu().numpy()
        assert np.array_equal(rank, S.rank_of_gt(lg_dev, gt)), "%s ranks" % impl
        assert np.array_equal(items, S.topk_items(lg_dev, 20)), "%s top-20" % impl
        assert np.array_equal(rank[live][lonely], want_oracle[lonely]), "%s ranks vs oracle" % impl
        r_items, r_scores = m.recommend(ids, V_EVAL, 20, force_exact=(impl == "exact"))
        assert np.array_equal(r_items.cpu().numpy(), ref_items), "%s recommendation" % impl
        assert np.array_equal(r_scores.cpu().numpy(), ref_scores), "%s recommendation scores" % impl
        assert m.eval_fallbacks == fb, "%s: a candidate overflow sent the batch to the exact entry" % impl
    if "tc" in impls:
        assert 2 * ops.eval_topk_chunks(m.ms, R, V_EVAL) >= 20                # the tcgen05 top-20 really ran
    log["eval rows vs oracle"] = float(lonely.mean())


def _check_herding(m, d, log):
    """segments of <= 16, 17..350 and > 350 candidates; picks == the float32 NumPy reference except at near-ties"""
    from ader_b200 import ops
    rng = np.random.RandomState(9)
    sizes = [3, 16, 17, 120, 351, 420]
    quota = np.array([2, 9, 17, 30, 40, 60], np.int32)
    N = sum(sizes)
    ids = _ids(rng, m.hp.maxlen, N, V_EVAL)
    rep = m.rep(ids)
    rep_np = rep.cpu().numpy()
    seg_off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
    quota = np.minimum(quota, sizes).astype(np.int32)
    steps = np.array([int(math.ceil(1.1 * int(q))) for q in quota], np.int32)
    dev = m.device
    t = lambda a: torch.tensor(a, device=dev)
    picks = torch.full((N,), -1, dtype=torch.int32, device=dev)
    n_picked = torch.zeros(len(sizes), dtype=torch.int32, device=dev)
    ws = torch.empty(ops.herding_ws_bytes(m.ms, N), dtype=torch.uint8, device=dev)
    ops.herding_segmented(m.ms, rep, t(np.arange(N, dtype=np.int32)), t(seg_off), t(quota), t(steps), ws, picks, n_picked)
    picks, n_picked = picks.cpu().numpy(), n_picked.cpu().numpy()
    ties = 0
    for c in range(len(sizes)):
        seg = rep_np[seg_off[c]:seg_off[c + 1]]
        want = P.herding_picks(seg, int(quota[c]))
        got = picks[seg_off[c]:seg_off[c] + n_picked[c]].tolist()
        if got != want:
            k = next(i for i, (a, b) in enumerate(zip(got + [-1], want + [-1])) if a != b)
            gap = _herding_gap(seg, int(quota[c]), want, k)
            assert gap < 1e-5, "d=%d segment of %d diverges at pick %d with argmax gap %.3e" % (d, sizes[c], k, gap)
            ties += 1
    log["herding near-tie segments"] = ties


def _check_fisher(m, hp, params, log):
    from ader_b200 import ops
    rng = np.random.RandomState(13)
    n = 6
    ids = _ids(rng, hp.maxlen, n, V_TRAIN)
    pos = rng.randint(1, V_TRAIN + 1, n).astype(np.int32)
    want = S.fisher_diag(params, torch.tensor(ids).long(), torch.tensor(pos), V_TRAIN, hp, n)
    dev = m.device
    acc = torch.zeros(m.layout.total, dtype=torch.float64, device=dev)
    tcap = int((ids != 0).sum())
    ops.fisher_batched(m.ms, m.theta, torch.tensor(ids, device=dev), torch.tensor(pos, device=dev), tcap, V_TRAIN,
                       torch.empty(ops.encoder_ws_bytes(m.ms, n, tcap), dtype=torch.uint8, device=dev),
                       torch.empty(ops.encoder_bwd_ws_bytes(m.ms, n, tcap), dtype=torch.uint8, device=dev),
                       torch.empty(ops.fisher_batched_ws_bytes(m.ms, n, V_TRAIN), dtype=torch.uint8, device=dev), acc)
    got = _views(m, (acc / n).float())
    worst = 0.0
    for i, (name, _) in enumerate(S.param_shapes(hp)):
        g, w = got[i], torch.tensor(want[i])
        if i == 0:
            g, w = g[1:V_TRAIN + 1], w[1:V_TRAIN + 1]
        worst = max(worst, _close(g, w, 1e-4, 1e-12, "batched fisher %s" % name))
    log["fisher"] = worst


def _check_refusals(d, L, h, nb, ids, log):
    """Training through the exact backward and the batched Fisher refuse before any launch where the exact attention
    backward does not fit; the same model keeps serving inference."""
    from ader_b200 import _lib, ops
    mx, _, _ = _model(d, L, h, nb, loss_impl="exact")
    assert mx.encoder_impl == "exact" and mx.train_refusal is not None
    pos = np.ones(ids.shape[0], np.int32)
    theta0, grad0 = mx.theta.clone(), mx.grad.clone()
    for call in (lambda: mx.loss_and_grad(ids, pos, V_TRAIN), lambda: mx.train_step(ids, pos, V_TRAIN)):
        with pytest.raises(_lib.AderError) as e:
            call()
        msg = str(e.value)
        assert "hidden_units=%d" % d in msg and "maxlen=%d" % L in msg and "shared memory" in msg, msg
    assert torch.equal(mx.theta, theta0) and torch.equal(mx.grad, grad0) and mx.global_step == 0
    # the batched Fisher entry: nothing written into the workspaces or the accumulator
    dev = mx.device
    n, tcap = 4, int((ids[:4] != 0).sum())
    enc = torch.full((ops.encoder_ws_bytes(mx.ms, n, tcap),), 0x5A, dtype=torch.uint8, device=dev)
    bwd = torch.full((ops.encoder_bwd_ws_bytes(mx.ms, n, tcap),), 0x5A, dtype=torch.uint8, device=dev)
    fws = torch.full((1 << 16,), 0x5A, dtype=torch.uint8, device=dev)
    acc = torch.zeros(mx.layout.total, dtype=torch.float64, device=dev)
    with pytest.raises(_lib.AderError, match="maxlen=%d" % L):
        ops.fisher_batched(mx.ms, mx.theta, torch.tensor(ids[:4], device=dev), torch.ones(n, dtype=torch.int32, device=dev),
                           tcap, V_TRAIN, enc, bwd, fws, acc)
    torch.cuda.synchronize()
    assert bool((enc == 0x5A).all()) and bool((bwd == 0x5A).all()) and bool((fws == 0x5A).all()) and not bool(acc.any())
    assert mx.rep(ids).shape == (ids.shape[0], d)                           # inference still works
    log["refused"] = 1.0


@pytest.mark.parametrize("d,L,h,nb,mode,why", CASES, ids=["d%d_L%d_h%d_b%d" % c[:4] for c in CASES])
def test_shape_against_fp64_oracle(d, L, h, nb, mode, why):
    from ader_b200 import ops
    t0 = time.time()
    log = {}
    m, hp, params = _model(d, L, h, nb)
    rng = np.random.RandomState(d * 100 + L)
    ids = _ids(rng, L, 44, V_EVAL, empty=True, full_row=(L == 64))
    rep_e = _check_reps(m, hp, params, ids, log)
    # an empty row scores every item 0: no certainty band can hold it, so evaluation takes the sessions only
    _check_eval(m, hp, params, rep_e[:-1], ids[:-1], log)
    if d in HERDING_D:
        _check_herding(m, d, log)
    bwd_ok = _served(m.ms, ops.PATH_ENCODER_BWD)
    if mode is None:                                         # no training path: refused before any launch
        assert m.train_refusal is not None and not bwd_ok
        with pytest.raises(ops._lib.AderError, match="maxlen=%d" % L):
            m.loss_and_grad(ids[:8], np.ones(8, np.int32), V_TRAIN)
        assert m.rep(ids).shape == (ids.shape[0], d)
    else:
        assert m.train_refusal is None
        ids_l, pos, kw, fn = _loss_inputs(m, hp, params, mode, rng, L)
        _check_grads(m, hp, params, ids_l, pos, kw, fn, "default (%s, %s)" % (m.encoder_impl, mode), log)
        if m.encoder_impl == "tc" and bwd_ok:                # the exact training path at the same shape
            mx, _, _ = _model(d, L, h, nb, loss_impl="exact")
            mx.mode, mx.lambda_ = m.mode, m.lambda_
            _check_grads(mx, hp, params, ids_l, pos, kw, fn, "exact (%s)" % mode, log)
    if _served(m.ms, ops.PATH_FISHER_BATCHED):
        _check_fisher(m, hp, params, log)
    if not bwd_ok:
        _check_refusals(d, L, h, nb, ids[:-1], log)
    print("\nshape d=%d maxlen=%d heads=%d blocks=%d (%s): %s; %.1f s" % (
        d, L, h, nb, why, ", ".join("%s %.2e" % kv for kv in log.items()), time.time() - t0))
