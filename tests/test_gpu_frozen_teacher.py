"""Distillation from a frozen snapshot of the previous model (data.FrozenTeacher) instead of stored [E, V_prev] logits.

Anchor: the exact fp32 entry recomputes the teacher rows with the SGEMM that produced the stored logits, so it must equal
the stored-logit call bit for bit.  The tcgen05 entries build the same bf16 Pc tiles from two tensor-core passes over the
snapshot; they are held to the bars of the stored tcgen05 path against the oracle (which gets the fp32 teacher logits of
the snapshot), and the fused / DAG / serial issue orders must agree bit for bit as they do for stored logits."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import sasrec as S


def _args(**kw):
    base = dict(hidden_units=150, maxlen=50, num_blocks=2, num_heads=1, random_seed=0, lr=5e-4,
                dropout_rate=0.0, disable_distillation=False, loss_impl="exact")
    base.update(kw)
    return type("Args", (), base)()


def _ids(rng, M, L, item_max, lens):
    ids = np.zeros((M, L), np.int32)
    for r in range(M):
        n = int(lens[r])
        if n:
            ids[r, L - n:] = rng.randint(1, item_max + 1, n)
    return ids


def _model(item_num, seed=1, scale=0.05, **kw):
    from ader_b200.model import Ader
    args = _args(**kw)
    m = Ader(item_num, args, init_seed=0)
    hp = S.Hyper(item_num, args.hidden_units, args.maxlen, args.num_blocks, args.num_heads)
    params = S.randomize_params(S.init_params(hp, 0), seed, scale)
    m.theta.copy_(torch.cat([p.reshape(-1) for p in params]))
    return m, hp, params


def _snapshot(item_num, Vp, E, rng, scale=0.05):
    """A 'previous model' (other weights) and its snapshot over E exemplar sessions."""
    from ader_b200.data import FrozenTeacher
    prev, _, _ = _model(item_num, seed=7, scale=scale)
    ex_ids = _ids(rng, E, 50, Vp, np.minimum(50, rng.geometric(0.25, E)))
    return FrozenTeacher(prev, prev.rep(ex_ids), Vp)


# ---- exact form: bit-identical to the stored-logit call ----------------------------------------------------------------
@pytest.mark.parametrize("shape", [(300, 100, 3001, 2477, 260, 4000), (333, 256, 3001, 3001, 90, 3001), (140, 12, 700, 640, 128, 700)],
                         ids=["vp_lt_v_nex200", "vp_eq_v_nex77", "nex128"])
def test_exact_frozen_form_is_bit_identical_to_stored_logits(shape):
    M, Bt, V, Vp, E, item_num = shape
    rng = np.random.RandomState(41)
    ft = _snapshot(item_num, Vp, E, rng)
    stored = ft.logits()
    assert stored.shape == (E, Vp)
    m, _, _ = _model(item_num, loss_impl="exact", encoder_impl="exact")
    m.update_loss(0.8)
    ids = _ids(rng, M, 50, V, np.minimum(50, rng.geometric(0.25, M)))
    pos = rng.randint(1, V + 1, Bt).astype(np.int32)
    trow = rng.randint(0, E, M - Bt).astype(np.int32)          # repeats, non-identity order
    trow[:3] = [E - 1, 0, E - 1]
    out = {}
    for name, teacher in (("stored", stored), ("frozen", ft)):
        loss = m.loss_and_grad(ids, pos, V, exemplar_logits=teacher, teacher_rows=trow).clone()
        out[name] = (loss, m.last_row_loss.clone(), m._keep[6].clone(), m.grad.clone())
    for a, b, what in zip(out["stored"], out["frozen"], ("loss", "row losses", "d_rep", "gradient")):
        assert torch.equal(a, b), what


def test_frozen_logits_are_the_previous_models_logits():
    """FrozenTeacher.logits() (the drop-in list / the stored matrix it stands for) is what the previous model's own logits
    fetch returns for the same reps; the snapshot table is a copy, not a view of the live weights."""
    from ader_b200.data import FrozenTeacher
    rng = np.random.RandomState(5)
    prev, _, _ = _model(900, seed=7)
    ex_ids = _ids(rng, 40, 50, 800, np.full(40, 9))
    rep = prev.rep(ex_ids)
    ft = FrozenTeacher(prev, rep, 800)
    want = prev.logits(rep, 800)
    prev.theta.add_(1.0)                                        # training on must not move the snapshot
    assert torch.equal(ft.logits(), want)
    assert ft.table.data_ptr() != prev.theta.data_ptr() + 150 * 4


# ---- tcgen05 form ---------------------------------------------------------------------------------------------------------
def _oracle(params, hp, ids, pos, V, lam, teacher_rows_logits):
    fn = lambda ps: S.loss_ader(ps, torch.tensor(ids).long(), torch.tensor(pos), V, hp, lam, exemplar_logits=teacher_rows_logits.cpu())
    return S.grads_of(fn, params)


@pytest.mark.parametrize("shape", [(24, 16, 450, 400, 500, 20), (333, 256, 3001, 2500, 4000, 150),
                                   (385, 256, 40135, 38501, 43136, 300), (650, 512, 18661, 17421, 25958, 400)],
                         ids=["small", "mid", "diginetica_p10", "bench_yoochoose_p4"])
def test_tc_frozen_form_matches_oracle_and_stored_form(shape):
    M, Bt, V, Vp, item_num, E = shape
    rng = np.random.RandomState(21)
    ft = _snapshot(item_num, Vp, E, rng, scale=0.02)
    trow = rng.randint(0, E, M - Bt).astype(np.int32)
    teacher_rows = ft.logits(torch.from_numpy(trow))           # fp32 teacher logits of the step's exemplar rows
    lens = np.minimum(50, rng.geometric(0.25, M))
    ids = _ids(rng, M, 50, V, lens)
    pos = rng.randint(1, V + 1, Bt).astype(np.int32)
    pos[0], pos[-1] = 1, V
    m, hp, params = _model(item_num, scale=0.02, loss_impl="tc", encoder_impl="exact")
    m.update_loss(0.9)
    loss = float(m.loss_and_grad(ids, pos, V, exemplar_logits=ft, teacher_rows=trow).item())
    g_frozen = m.grad.clone()
    ref, grads = _oracle(params, hp, ids, pos, V, 0.9, teacher_rows)
    assert loss == pytest.approx(ref, rel=1e-3)
    got = [v.detach().cpu() for v in m.layout.views(g_frozen)]
    for i, (name, _) in enumerate(S.param_shapes(hp)):
        g, w = got[i].double(), grads[i].double()
        if i == 0:
            g, w = g[1:V + 1], w[1:V + 1]
        err, tol = float((g - w).abs().max()), 1e-2 * float(w.abs().max()) + 1e-7
        assert err <= tol, "frozen tc grad of %s: max err %.3e > %.3e" % (name, err, tol)
    # the stored tcgen05 form on the same teacher rows: same bars against each other
    loss_s = float(m.loss_and_grad(ids, pos, V, exemplar_logits=teacher_rows).item())
    assert loss == pytest.approx(loss_s, rel=1e-3)
    gmax = float(m.grad.abs().max())
    assert float((g_frozen - m.grad).abs().max()) <= 1e-2 * gmax
    # run-to-run bit identity
    m.loss_and_grad(ids, pos, V, exemplar_logits=ft, teacher_rows=trow)
    assert torch.equal(g_frozen, m.grad)


def test_default_tc_path_with_frozen_teacher_matches_oracle_at_bench_shape():
    """Fused encoder + tcgen05 loss (the default DAG step) with a snapshot, at the bench.py shape: the bars of
    test_default_tc_path_matches_oracle_at_baseline_shapes (loss 1e-3 rel; per tensor rel-L2 <= 3e-2, max-abs <= 0.15)."""
    M, Bt, V, Vp, item_num, lam, E = 650, 512, 18661, 17421, 25958, 1.0, 400
    rng = np.random.RandomState(31)
    ft = _snapshot(item_num, Vp, E, rng, scale=0.02)
    trow = rng.randint(0, E, M - Bt).astype(np.int32)
    teacher_rows = ft.logits(torch.from_numpy(trow))
    m, hp, params = _model(item_num, scale=0.02, loss_impl="tc")
    assert m.encoder_impl == "tc" and m.step_impl == "dag"
    lens = np.minimum(50, rng.geometric(0.22, M))
    ids = _ids(rng, M, 50, V, lens)
    pos = rng.randint(1, V + 1, Bt).astype(np.int32)
    m.update_loss(lam)
    loss = float(m.loss_and_grad(ids, pos, V, exemplar_logits=ft, teacher_rows=trow, n_tokens=int(lens.sum())).item())
    ref, grads = _oracle(params, hp, ids, pos, V, lam, teacher_rows)
    assert loss == pytest.approx(ref, rel=1e-3)
    got = [v.detach().cpu() for v in m.layout.views(m.grad)]
    gscale = max(float(w.abs().max()) for w in grads)
    floor_ = 1e-5 * gscale
    for i, (name, _) in enumerate(S.param_shapes(hp)):
        g, w = got[i].double(), grads[i].double()
        if i == 0:
            g, w = g[1:V + 1], w[1:V + 1]
        rel = float((g - w).norm() / (w.norm() + floor_ * w.numel() ** 0.5))
        mx = float((g - w).abs().max() / (w.abs().max() + floor_))
        assert rel <= 3e-2 and mx <= 0.15, "%s: rel-L2 %.3e, max-abs/max|g| %.3e" % (name, rel, mx)


@pytest.mark.parametrize("dropout", [0.0, 0.3])
def test_fused_entries_are_bit_identical_to_the_three_groups(dropout):
    """ader_train_step_tc (DAG and serial), ader_train_fwd_bwd_tc + Adam and the three single-group entries + Adam, with a
    snapshot, over several steps: the same bits."""
    M, Bt, V, Vp, item_num, E = 333, 256, 3001, 2500, 4000, 150
    rng = np.random.RandomState(8)
    ft = _snapshot(item_num, Vp, E, rng)
    steps = []
    for _ in range(3):
        lens = np.minimum(50, rng.geometric(0.25, M))
        steps.append((_ids(rng, M, 50, V, lens), rng.randint(1, V + 1, Bt).astype(np.int32),
                      rng.randint(0, E, M - Bt).astype(np.int32)))
    res = {}
    for impl in ("groups", "dag", "serial", "dag_no_fused_adam"):
        m, _, _ = _model(item_num, loss_impl="tc", step_impl=("dag" if impl == "dag_no_fused_adam" else impl), dropout_rate=dropout)
        m.update_loss(0.8)
        losses = []
        for ids, pos, trow in steps:
            if impl == "dag_no_fused_adam":           # ader_train_fwd_bwd_tc, then the optimiser call
                losses.append(m.loss_and_grad(ids, pos, V, exemplar_logits=ft, teacher_rows=trow, dropout_rate=dropout).clone())
                m.apply_gradients(V, 5e-4)
            else:
                losses.append(m.train_step(ids, pos, V, 5e-4, dropout, exemplar_logits=ft, teacher_rows=trow).clone())
        res[impl] = (torch.stack(losses), m.theta.clone(), m.adam_m.clone(), m.adam_v.clone())
    for impl in ("dag", "serial", "dag_no_fused_adam"):
        for a, b, what in zip(res["groups"], res[impl], ("losses", "theta", "adam_m", "adam_v")):
            assert torch.equal(a, b), "%s: %s differs from the three groups" % (impl, what)


def test_peer_memory_dp_with_frozen_teacher_equals_full_batch():
    """Two emulated ranks on one GPU, each with its shard of the exemplar rows (teacher_rows sliced), against one replica
    with the full batch (pattern and bounds of tests/test_gpu_dp.py)."""
    from ader_b200.dist import local_peer_group, shard_rows
    M, Bt, V, Vp, item_num, E, world = 37, 25, 380, 300, 400, 30, 2
    rng = np.random.RandomState(3)
    ft = _snapshot(item_num, Vp, E, rng)
    batches = []
    for _ in range(3):
        ids = np.zeros((M, 50), np.int32)
        for r in range(M):
            k = int(rng.randint(1, 20)); ids[r, 50 - k:] = rng.randint(1, V + 1, k)
        batches.append((ids, rng.randint(1, V + 1, Bt).astype(np.int32), rng.randint(0, E, M - Bt).astype(np.int32)))

    def mk():
        from ader_b200.model import Ader
        m = Ader(item_num, _args(loss_impl="exact"), init_seed=0)
        m.theta.add_(torch.randn(m.theta.shape, generator=torch.Generator().manual_seed(1)).to(m.device) * 0.05)
        m.update_loss(0.7)
        return m
    ref = mk()
    ref_losses = [float(ref.train_step(ids, pos, V, 5e-4, 0.0, exemplar_logits=ft, teacher_rows=tr).item()) for ids, pos, tr in batches]
    models = [mk() for _ in range(world)]
    comms = local_peer_group(models)
    streams = [torch.cuda.Stream() for _ in range(world)]
    torch.cuda.synchronize()

    def shard(r, ids, pos, tr):
        (tl, th), (el, eh) = shard_rows(len(pos), len(ids) - len(pos), r, world)
        rows = list(range(tl, th)) + list(range(len(pos) + el, len(pos) + eh))
        return ids[rows], pos[tl:th], tr[el:eh]
    for r, m in enumerate(models):                        # warm-up step without the back end, rolled back (see test_gpu_dp.py)
        ids, pos, tr = shard(r, *batches[0])
        m.global_counts = (Bt, M - Bt)
        sd = m.state_dict(); comm, m.dp = m.dp, None
        with torch.cuda.stream(streams[r]):
            m.train_step(ids, pos, V, 5e-4, 0.0, exemplar_logits=ft, teacher_rows=tr)
        torch.cuda.synchronize()
        m.load_state_dict(sd); m.dp = comm
        torch.cuda.synchronize()
    losses = []
    for b in batches:
        part = []
        for r, m in enumerate(models):
            ids, pos, tr = shard(r, *b)
            m.global_counts = (Bt, M - Bt)
            with torch.cuda.stream(streams[r]):
                part.append(m.train_step(ids, pos, V, 5e-4, 0.0, exemplar_logits=ft, teacher_rows=tr).clone())
        torch.cuda.synchronize()
        losses.append(sum(float(p.item()) for p in part))
    for c in comms:
        c.check()
    assert losses == pytest.approx(ref_losses, rel=1e-5)
    th = [m.theta.cpu().numpy() for m in models]
    assert np.array_equal(th[0], th[1])
    assert np.abs(th[0] - ref.theta.cpu().numpy()).max() < 3e-5


def test_vocab_parallel_helper_refuses_a_frozen_teacher():
    from ader_b200.data import FrozenTeacher
    from ader_b200.dist import VocabParallelLoss
    rng = np.random.RandomState(2)
    ft = _snapshot(400, 300, 10, rng)
    assert isinstance(ft, FrozenTeacher)
    with pytest.raises(ValueError):
        VocabParallelLoss.fwd_bwd(type("X", (), {"ops": None, "model": None})(), torch.zeros(12, 150, device="cuda"),
                                  torch.ones(2, dtype=torch.int32, device="cuda"), 380, 0.8, 1, teacher=ft)


# ---- the driver end to end on the tiny split ----------------------------------------------------------------------------
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
    a.trace = True
    for k, v in kw.items():
        setattr(a, k, v)
    return a


@pytest.mark.parametrize("selection", ["herding", "random"])
def test_driver_frozen_exact_equals_stored_logits(tmp_path, selection):
    from ader_b200.data import FrozenTeacher
    from ader_b200.main import run
    a = run(_e2e_args(tmp_path / "l", selection=selection, teacher="logits"))
    b = run(_e2e_args(tmp_path / "f", selection=selection, teacher="frozen"))
    for pa, pb in zip(a["trace"]["periods"], b["trace"]["periods"]):
        assert pa["losses"] == pb["losses"]
        assert pa["best_epoch"] == pb["best_epoch"] and pa["test"] == pb["test"] and pa["test_ranks"] == pb["test_ranks"]
        assert pa["exemplars"] == pb["exemplars"]
    assert torch.equal(a["model"].theta, b["model"].theta)
    assert a["per_period"] == b["per_period"]


def test_driver_frozen_tc_path_reaches_same_metrics(tmp_path):
    from ader_b200.main import run
    ra = run(_e2e_args(tmp_path / "exact", selection="random"))
    rb = run(_e2e_args(tmp_path / "tc", loss_impl="tc", selection="random", teacher="frozen"))
    for pa, pb in zip(ra["trace"]["periods"], rb["trace"]["periods"]):
        np.testing.assert_allclose(pb["losses"][:30], pa["losses"][:30], rtol=5e-2)
        assert abs(pa["test"][1] - pb["test"][1]) <= 0.03
    np.testing.assert_allclose(rb["trace"]["periods"][0]["losses"][:10], ra["trace"]["periods"][0]["losses"][:10], rtol=2e-3)


@pytest.mark.parametrize("selection,kw", [("herding", {}), ("random", {"loss_impl": "tc", "dropout_rate": 0.3})])
def test_driver_frozen_resume_reproduces_the_uninterrupted_run(tmp_path, selection, kw):
    from ader_b200.main import run
    full = run(_e2e_args(tmp_path / "full", selection=selection, teacher="frozen", **kw))
    run(_e2e_args(tmp_path / "cut", selection=selection, teacher="frozen", max_periods=2, **kw))
    rest = run(_e2e_args(tmp_path / "cut", selection=selection, teacher="frozen", resume=True, **kw))
    assert len(rest["trace"]["periods"]) == 1
    a, b = full["trace"]["periods"][2], rest["trace"]["periods"][0]
    assert a["losses"] == b["losses"] and a["test_ranks"] == b["test_ranks"] and a["exemplars"] == b["exemplars"]
    assert torch.equal(full["model"].theta, rest["model"].theta)
    with pytest.raises(ValueError):                       # the teacher form is part of the protocol a resume must match
        run(_e2e_args(tmp_path / "cut", selection=selection, teacher="logits", resume=True, **kw))


def test_frozen_selection_builds_no_vocabulary_wide_matrix():
    """In the frozen form selection keeps [E, d] reps and the [V_prev, d] table copy, and never allocates anything with
    V_prev columns, not even transiently: the peak device memory of herding selection grows by far less than the
    E x V_prev fp32 matrix the stored form allocates (and the stored form's peak does hold it)."""
    import random
    from ader_b200.data import ExemplarGenerator, FrozenTeacher
    Vp = 200000
    m, _, _ = _model(Vp, loss_impl="exact")
    rng = np.random.RandomState(0)
    data = [[int(x) for x in rng.randint(1, 500, rng.randint(2, 12))] for _ in range(3000)]
    gens, growth = {}, {}
    for form in ("logits", "frozen"):
        random.seed(0); np.random.seed(0)
        gens[form] = ExemplarGenerator(data, 2000, False, 32, 50, 0.0, Vp, teacher=form)
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        gens[form].herding_selection(None, m)
        torch.cuda.synchronize()
        growth[form] = torch.cuda.max_memory_allocated() - base
        if form == "logits":
            ref = gens[form].exemplars.teacher.clone()
            gens[form].exemplars.teacher = None          # drop the stored matrix before the frozen form is measured
            torch.cuda.empty_cache()
    t = gens["frozen"].exemplars.teacher
    n = len(gens["frozen"].exemplars)
    assert isinstance(t, FrozenTeacher) and n == len(t) > 100
    assert t.rep.shape == (n, 150) and t.table.shape == (Vp, 150)
    matrix = n * Vp * 4
    assert growth["logits"] >= matrix
    assert growth["frozen"] < matrix / 4, (growth, matrix)
    assert gens["frozen"].exemplars.sessions == gens["logits"].exemplars.sessions
    assert torch.equal(ref, t.logits())


def test_graph_replays_with_frozen_teacher_match_eager_steps():
    """GraphStep(teacher=FrozenTeacher) replays == the eager step with the same snapshot, bit for bit (pattern of
    test_gpu_encoder_fused.test_graph_step_replays_match_eager_steps: dropout, both feed forms)."""
    rng = np.random.RandomState(7)
    B, Me, V, Vp, E = 48, 16, 280, 250, 40
    pool = _ids(rng, 200, 50, V, rng.randint(1, 51, 200))
    lab = rng.randint(1, V + 1, 200).astype(np.int32)
    ex = _ids(rng, E, 50, Vp, rng.randint(1, 51, E))
    steps = [(rng.randint(0, 200, B), rng.randint(0, E, Me)) for _ in range(4)]
    ft = _snapshot(300, Vp, E, np.random.RandomState(3))
    out = {}
    for mode in ("eager", "graph"):
        m, _, _ = _model(300, loss_impl="tc", lr=1e-3)
        m.update_loss(0.7)
        losses = []
        if mode == "graph":
            src = (torch.tensor(pool, device=m.device), torch.tensor(lab, device=m.device), torch.tensor(ex, device=m.device),
                   torch.arange(E, dtype=torch.int32, device=m.device))
            gs = m.graph_step(B, Me, V, 1e-3, 0.3, teacher=ft, sources=src, tcaps=[900])
        for k, (ti, ei) in enumerate(steps):
            ids = np.concatenate([pool[ti], ex[ei]])
            ntok = int((ids != 0).sum())
            if mode == "eager":
                loss = m.train_step(ids, lab[ti], V, 1e-3, 0.3, exemplar_logits=ft, teacher_rows=ei.astype(np.int32), n_tokens=ntok)
            elif k % 2 == 0:
                loss = gs.run_indices(ti, ei, ntok)
            else:
                loss = gs.run_rows(ids, lab[ti], ei, ntok)
            losses.append(float(loss.item()))
        out[mode] = (losses, m.theta.clone())
    assert out["eager"][0] == out["graph"][0]
    assert torch.equal(out["eager"][1], out["graph"][1])
    assert len(set(out["eager"][0])) == len(steps)
