"""GPU parity of the fused tensor-core encoder (ader_encoder_fwd_tc / ader_encoder_bwd_tc: row-scaled fp16
operands, fp32 accumulation) against (a) the exact fp32 CUDA path, workspace slot by slot, and (b) the CPU
oracle.

Stated tolerances (measured values in profiles/RESULTS_r1.md):
  * activations / rep: 1e-2 * max|want| element-wise (measured rel-L2 3e-4 .. 7e-4: fp16 unit round-off 2^-12
    per operand over 150-term dot products, two blocks);
  * loss: 1e-3 rel;
  * gradients, per tensor: rel-L2 <= 3e-2 and max-abs <= 0.15 * max|g|.  The backward GEMMs themselves are
    accurate to ~1e-3; what dominates is the ReLU kink: a forward perturbed by 3e-4 flips the sign of ~2e-4
    of the hidden pre-activations, and each flip switches a whole gradient element on or off (the result is
    the exact gradient of the perturbed forward).  Measured: rel-L2 <= 1.8e-2, max-abs <= 0.10 (one w1 element).
  * a tensor whose true gradient is identically zero (the key bias: softmax is shift invariant) is compared
    absolutely against the global gradient scale.
Integer outputs of the packing (row offsets, token ids) are exact; results are run-to-run bit-identical.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import sasrec as S
from test_gpu_parity import _close, _ids, _model, _views

ACT_TOL, LOSS_TOL, GRAD_TOL, GRAD_L2_TOL = 1e-2, 1e-3, 0.15, 3e-2


def _slots(m, M, tcap, block):
    from ader_b200 import ops
    buf = m._enc_ws.buf
    d = m.hp.hidden_units
    T = int(buf[ops.encoder_ws_slot(m.ms, M, tcap, -2, 0):].view(torch.int32)[M].item())
    out = {}
    for s in range(8):
        off = ops.encoder_ws_slot(m.ms, M, tcap, s, block)
        out[s] = buf[off:off + T * d * 4].view(torch.float32).view(T, d).clone()
    off = ops.encoder_ws_slot(m.ms, M, tcap, 9, block)
    L = m.hp.maxlen
    out[9] = buf[off:off + T * L * 4 * m.hp.num_heads].view(torch.float32).clone()
    return T, out


@pytest.mark.parametrize("heads,blocks", [(1, 2), (3, 1), (2, 3)])
def test_fused_forward_matches_exact_slots(heads, blocks):
    m, hp, params = _model(300, num_heads=heads, num_blocks=blocks)
    rng = np.random.RandomState(0)
    lens = [1, 50, 2, 49, 33] + list(rng.randint(1, 51, 40)) + [0, 7]      # n=1, n=50, an empty row, T % 32 != 0
    ids_np = _ids(rng, len(lens), 50, 300, lens)
    ids = torch.tensor(ids_np, device=m.device)
    M = len(lens)
    rep_e, tcap = m.encode(ids, impl="exact")
    rep_e = rep_e.clone()
    exact = [_slots(m, M, tcap, b) for b in range(blocks)]
    rep_t, _ = m.encode(ids, impl="tc")
    fused = [_slots(m, M, tcap, b) for b in range(blocks)]
    names = {0: "x", 1: "q1", 2: "Q", 3: "K", 4: "V", 5: "y", 6: "z", 7: "h", 9: "probs"}
    for b in range(blocks):
        assert exact[b][0] == fused[b][0] == sum(lens)
        for s, nm in names.items():
            if heads > 1 and s == 9:
                continue     # probs of head h live at [h*Tcap + t]: the flat prefix compared here covers head 0 only partially
            _close(fused[b][1][s].cpu(), exact[b][1][s].cpu(), ACT_TOL, 1e-6, "block %d slot %s" % (b, nm))
    _close(rep_t.cpu(), rep_e.cpu(), ACT_TOL, 1e-6, "rep")
    want = S.forward_rep(params, torch.tensor(ids_np[[i for i, n in enumerate(lens) if n]]).long(), hp)
    _close(rep_t.cpu()[[i for i, n in enumerate(lens) if n]], want, ACT_TOL, 1e-6, "rep vs oracle")
    assert float(rep_t[lens.index(0)].abs().max()) == 0.0


@pytest.mark.parametrize("heads,mode", [(1, "kd"), (2, "kd"), (1, "vanilla")])
def test_fused_gradients_match_oracle(heads, mode):
    m, hp, params = _model(400, num_heads=heads, encoder_impl="tc")
    assert m.encoder_impl == "tc" and m.loss_impl == "exact"
    rng = np.random.RandomState(3)
    ids = _ids(rng, 45, 50, 380)
    ids[5] = ids[4]
    ids[:, -1] = np.where(rng.rand(45) < 0.4, 7, ids[:, -1])       # hot id -> segmented scatter
    if mode == "kd":
        pos = rng.randint(1, 381, 30).astype(np.int32)
        teacher = (rng.randn(15, 300) * 2).astype(np.float32)
        m.update_loss(0.73)
        loss = m.loss_and_grad(ids, pos, 380, exemplar_logits=teacher)
        fn = lambda ps: S.loss_ader(ps, torch.tensor(ids).long(), torch.tensor(pos), 380, hp, 0.73,
                                    exemplar_logits=torch.tensor(teacher))
    else:
        pos = rng.randint(1, 381, 45).astype(np.int32)
        loss = m.loss_and_grad(ids, pos, 380)
        fn = lambda ps: S.loss_vanilla(ps, torch.tensor(ids).long(), torch.tensor(pos), 380, hp)
    loss_ref, grads_ref = S.grads_of(fn, params)
    assert float(loss.item()) == pytest.approx(loss_ref, rel=LOSS_TOL)
    got = _views(m, m.grad)
    report = []
    gscale = max(float(w.abs().max()) for w in grads_ref)
    for i, (name, _) in enumerate(S.param_shapes(hp)):
        g, w = got[i].double(), grads_ref[i].double()
        if i == 0:
            g, w = g[1:381], w[1:381]
        floor_ = 1e-5 * gscale                       # absolute floor: tensors with an identically-zero true gradient
        e_max = float((g - w).abs().max()) / (float(w.abs().max()) + floor_)
        e_l2 = float((g - w).norm()) / (float(w.norm()) + floor_ * w.numel() ** 0.5)
        report.append((name, e_max, e_l2))
    print("fused encoder gradient errors (max-abs/max|g|, rel-L2):")
    for name, a, b in report:
        print("   %-28s %.3e %.3e" % (name, a, b))
    for name, a, b in report:
        assert a <= GRAD_TOL and b <= GRAD_L2_TOL, (name, a, b)
    # run-to-run determinism (fixed reduction orders, no float atomics)
    g0 = m.grad.clone()
    if mode == "kd":
        m.loss_and_grad(ids, pos, 380, exemplar_logits=teacher)
    else:
        m.loss_and_grad(ids, pos, 380)
    assert torch.equal(g0, m.grad)


def test_fused_single_row_and_tight_capacity():
    """Fisher-style batch of one (EWC.py:135-150) and a token capacity equal to the exact token count."""
    m, hp, params = _model(300, encoder_impl="tc")
    rng = np.random.RandomState(5)
    ids = _ids(rng, 1, 50, 280, [9])
    pos = np.array([17], np.int32)
    loss = m.loss_and_grad(ids, pos, 280, n_tokens=9)
    fn = lambda ps: S.loss_vanilla(ps, torch.tensor(ids).long(), torch.tensor(pos), 280, hp)
    loss_ref, grads_ref = S.grads_of(fn, params)
    assert float(loss.item()) == pytest.approx(loss_ref, rel=LOSS_TOL)
    got = _views(m, m.grad)
    for i in (1, 4, 14, 31):
        w = grads_ref[i].double()
        assert float((got[i].double() - w).norm()) <= GRAD_L2_TOL * float(w.norm()) + 1e-9, "single-row grad %d" % i


def test_fused_dropout_masks_match_exact_path():
    """Both encoder paths draw the same counter-based dropout masks (site, element) -> with the same seed the
    two losses agree to bf16 tolerance and stored hidden activations are zero at the same places."""
    rng = np.random.RandomState(6)
    ids = _ids(rng, 40, 50, 280)
    pos = rng.randint(1, 281, 40).astype(np.int32)
    losses, hs = [], []
    for impl in ("exact", "tc"):
        m, hp, _ = _model(300, encoder_impl=impl)
        m.global_step = 11
        loss = m.loss_and_grad(ids, pos, 280, dropout_rate=0.3, n_tokens=int((ids != 0).sum()))
        losses.append(float(loss.item()))
        T, sl = _slots(m, 40, int((ids != 0).sum()), 0)
        hs.append(sl[7].cpu())
        g = m.grad.clone()
        m.loss_and_grad(ids, pos, 280, dropout_rate=0.3, n_tokens=int((ids != 0).sum()))
        assert torch.equal(g, m.grad)
    assert losses[1] == pytest.approx(losses[0], rel=5e-3)
    differ = float(((hs[0] == 0) != (hs[1] == 0)).float().mean())
    assert differ < 5e-3, differ        # only ReLU sign flips of near-zero pre-activations may differ


def test_fused_rejects_wide_models():
    from ader_b200 import _lib, ops
    m, hp, _ = _model(100, hidden_units=192, num_heads=1)
    assert m.encoder_impl == "exact"
    ids = torch.tensor(_ids(np.random.RandomState(0), 4, 50, 90), device=m.device)
    with pytest.raises(_lib.AderError):
        m.encode(ids, impl="tc")


def test_graph_step_replays_match_eager_steps():
    """GraphStep (CUDA-graph capture of train_step, device-side dropout counter) == the eager step, bit for bit:
    same kernels, same (seed + step) dropout stream, over several steps and both input modes."""
    rng = np.random.RandomState(7)
    B, Me, V, Vp, E = 48, 16, 280, 250, 40
    pool = _ids(rng, 200, 50, V)
    lab = rng.randint(1, V + 1, 200).astype(np.int32)
    ex = _ids(rng, E, 50, Vp)
    steps = [(rng.randint(0, 200, B), rng.randint(0, E, Me)) for _ in range(4)]
    out = {}
    for mode in ("eager", "graph"):
        m, hp, _ = _model(300, loss_impl="tc", lr=1e-3)
        teacher = torch.randn(E, Vp, device=m.device, generator=torch.Generator(device=m.device).manual_seed(1))
        m.update_loss(0.7)
        losses = []
        if mode == "graph":
            src = (torch.tensor(pool, device=m.device), torch.tensor(lab, device=m.device), torch.tensor(ex, device=m.device),
                   torch.arange(E, dtype=torch.int32, device=m.device))
            gs = m.graph_step(B, Me, V, 1e-3, 0.3, teacher=teacher, sources=src, tcaps=[900])
        for k, (ti, ei) in enumerate(steps):
            ids = np.concatenate([pool[ti], ex[ei]])
            ntok = int((ids != 0).sum())
            if mode == "eager":
                loss = m.train_step(ids, lab[ti], V, 1e-3, 0.3, exemplar_logits=teacher, teacher_rows=ei.astype(np.int32), n_tokens=ntok)
            elif k % 2 == 0:
                loss = gs.run_indices(ti, ei, ntok)
            else:
                loss = gs.run_rows(ids, lab[ti], ei, ntok)
                pending = gs.fetch_loss()                 # async pinned read of the same scalar
                assert pending.result() == float(loss.item())
            losses.append(float(loss.item()))
        assert m.global_step == len(steps) and int(m.adam_state[0].item()) == len(steps)
        out[mode] = (losses, m.theta.clone())
    assert out["eager"][0] == out["graph"][0]
    assert torch.equal(out["eager"][1], out["graph"][1])
    assert len(set(out["eager"][0])) == len(steps)          # dropout masks / batches really changed from step to step


@pytest.mark.parametrize("blocks,mode", [(2, "kd"), (3, "kd"), (2, "er"), (1, "vanilla")])
def test_train_dag_entry_is_bit_identical_to_the_three_groups(blocks, mode):
    """ader_train_fwd_bwd_tc (fork/join DAG over the library's side streams) == ader_encoder_fwd_tc ->
    ader_loss_fwd_bwd_tc -> ader_encoder_bwd_tc, bit for bit (loss, row losses, rep, whole gradient), over many
    different batches (a missing edge shows up as a race), with dropout, and its serial form as well."""
    rng = np.random.RandomState(11)
    B, V, Vp, E = 160, 900, 800, 64
    Me = 0 if mode == "vanilla" else 40
    models = {}
    for impl in ("groups", "dag", "serial"):
        m, hp, _ = _model(1000, loss_impl="tc", num_blocks=blocks, step_impl=impl,
                          disable_distillation=(mode == "er"))
        if mode != "vanilla":
            m.update_loss(0.6)
        models[impl] = m
    dev = models["dag"].device
    teacher = torch.randn(E, Vp, device=dev, generator=torch.Generator(device=dev).manual_seed(3))
    for it in range(12):
        ids = _ids(rng, B + Me, 50, V if Me == 0 else Vp, lens=rng.randint(1, 14, B + Me))
        pos = rng.randint(1, V + 1, B).astype(np.int32)
        kw = {}
        if mode == "kd":
            kw = dict(exemplar_logits=teacher, teacher_rows=rng.randint(0, E, Me).astype(np.int32))
        elif mode == "er":
            kw = dict(exemplar_pos=rng.randint(1, Vp + 1, Me).astype(np.int32))
        ntok = int((ids != 0).sum())
        got = {}
        for impl, m in models.items():
            m.global_step = it                      # same dropout stream in all three
            m.grad.zero_()
            loss = m.loss_and_grad(ids, pos, V, dropout_rate=0.3, n_tokens=ntok, **kw)
            got[impl] = (loss.clone(), m.last_row_loss.clone(), m._keep[5].clone(), m.grad.clone())
        torch.cuda.synchronize()
        for impl in ("dag", "serial"):
            for k, (x, y) in enumerate(zip(got["groups"], got[impl])):
                assert torch.equal(x, y), "%s differs from the three-group sequence (output %d, batch %d)" % (impl, k, it)
    assert float(got["dag"][0].item()) > 0.0


@pytest.mark.parametrize("ewc", [False, True])
def test_fused_train_step_matches_groups_then_adam(ewc):
    """ader_train_step_tc (optimiser inside the DAG: early step size, table rows behind the scatter, dense parameters
    behind their partial reduction, counter bumped last) == three groups + ader_adam_step: parameters, both Adam
    slots and the step counter bit for bit after several steps with dropout (the counter feeds the dropout stream)."""
    from ader_b200.model import Ewc
    from test_gpu_parity import _args
    rng = np.random.RandomState(21)
    B, Me, V, Vp, E = 96, 32, 700, 650, 48
    batches = []
    for _ in range(5):
        ids = _ids(rng, B + Me, 50, Vp, lens=rng.randint(1, 12, B + Me))
        batches.append((ids, rng.randint(1, V + 1, B).astype(np.int32), rng.randint(0, E, Me).astype(np.int32)))
    out = {}
    for impl in ("groups", "dag"):
        if ewc:
            m = Ewc(800, _args(loss_impl="tc", step_impl=impl), init_seed=0)
            g = torch.Generator(device=m.device).manual_seed(5)
            m.fisher = torch.rand(m.layout.total, device=m.device, generator=g)
            m.theta_star = m.theta.clone() + 0.01
            m.update_loss(50.0)
        else:
            m, _, _ = _model(800, loss_impl="tc", step_impl=impl)
            m.update_loss(0.9)
        teacher = torch.randn(E, Vp, device=m.device, generator=torch.Generator(device=m.device).manual_seed(2))
        losses = []
        for ids, pos, rows in batches:
            ntok = int((ids != 0).sum())
            if ewc:
                loss = m.train_step(ids[:B], pos, V, 1e-3, 0.0, n_tokens=int((ids[:B] != 0).sum()))
            else:
                loss = m.train_step(ids, pos, V, 1e-3, 0.3, exemplar_logits=teacher, teacher_rows=rows, n_tokens=ntok)
            losses.append(float(loss.item()))
        out[impl] = (losses, m.theta.clone(), m.adam_m.clone(), m.adam_v.clone(), m.adam_state.clone(), m.global_step)
    assert out["groups"][0] == out["dag"][0]
    for k in range(1, 5):
        assert torch.equal(out["groups"][k], out["dag"][k]), "state tensor %d differs" % k
    assert out["groups"][5] == out["dag"][5] == len(batches)
    assert int(out["dag"][4][0].item()) == len(batches)
