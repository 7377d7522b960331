"""Pin oracle/protocol.py to fixtures minted from the reference's own util.py
(tests/golden/make_golden.py), and to the live reference when it is mounted."""
import json
import os
import random

import numpy as np
import pytest

from oracle import protocol as P
from oracle import refstub

MAXLEN = 50


@pytest.fixture(scope="module")
def gold(golden_dir):
    with open(os.path.join(golden_dir, "protocol.json")) as f:
        return json.load(f)


def test_protocol_matches_reference_fixture(gold, golden_dir):
    random.seed(0)
    np.random.seed(0)
    files = P.PeriodFiles(os.path.join(golden_dir, "tiny_data"))
    train_sess, n_act = files.train(0)
    assert "total number of action: %d." % n_act in gold["train_info"]
    assert len(train_sess) == gold["n_train_sessions"]
    s = P.RefSampler(train_sess, MAXLEN, 16)
    assert s.data_size() == gold["n_rows_before_split"]
    valid, train = s.split_data(0.1)
    assert valid == gold["valid_rows"]
    assert train[:20] == gold["train_rows_head"]
    assert len(train) == gold["n_train_rows"]
    assert s.batch_num() == gold["batch_num"]
    for ref in gold["batches"]:
        seq, pos = s.sampler()
        assert np.array(seq).tolist() == ref["seq"]
        assert list(pos) == ref["pos"]
    test_sess, total, removed = files.evaluate(1)
    assert "original total number of action: %d, removed number of action: %d." % (total, removed) in gold["test_info"]
    assert test_sess == gold["test_sessions"]
    assert files.max_item() == gold["max_item"]

    ev = P.RefSampler(test_sess, MAXLEN, 8, is_subseq=False)
    assert ev.data_size() == gold["test_rows_total"]
    for ref in gold["test_batches"]:
        seq, pos = ev.sampler()
        assert np.array(seq).tolist() == ref["seq"] and list(pos) == ref["pos"]

    cand = list(train) + list(valid)
    by_item, count = P.group_by_label(cand, MAXLEN, 16, files.max_item())
    quota = P.exemplar_quota(count, 120, equal=False)
    assert quota.tolist() == gold["quota"]
    assert [int(k) for k in by_item.keys()] == gold["label_order"]
    assert [len(v) for v in by_item.values()] == gold["group_sizes"]
    assert np.array(next(iter(by_item.values()))).tolist() == gold["first_group"]
    by_item2, count2 = P.group_by_label(cand, MAXLEN, 16, files.max_item())
    quota_eq = P.exemplar_quota(count2, 120, equal=True)
    assert quota_eq.tolist() == gold["quota_equal"]
    picks = []
    for item, seqs in by_item2.items():
        m = quota_eq[item - 1]
        picks.append(P.random_picks(len(seqs), m).tolist() if m > 0 else [])
    assert picks == gold["random_picks"]

    exemplars = [[r, [float(len(r)), 0.5]] for r in train[:37]]
    ex = P.RefSampler([], MAXLEN, 5)
    ex.add_exemplar(exemplars)
    for ref in gold["exemplar_batches"]:
        seq, pos, lg = ex.exemplar_sampler()
        assert np.array(seq).tolist() == ref["seq"] and list(pos) == ref["pos"]
        assert [list(x) for x in lg] == ref["logits"]


def test_metrics_match_reference_fixture(gold):
    from oracle.sasrec import metrics_from_ranks
    assert list(metrics_from_ranks(gold["ranks"])) == pytest.approx(gold["metrics"], abs=0)


def test_herding_matches_reference_fixture(golden_dir):
    z = np.load(os.path.join(golden_dir, "herding.npz"))
    for c in range(len(z["m"])):
        rep = z["rep"][z["seg_off"][c]:z["seg_off"][c + 1]]
        want = z["picks"][z["pick_off"][c]:z["pick_off"][c + 1]]
        want = [int(x) for x in want if x >= 0]
        assert P.herding_picks(rep, int(z["m"][c])) == want, "case %d" % c


def test_lambda_and_exemplar_batch():
    assert P.adaptive_lambda(0.8, 18569, 22692, 30000, 26799) == pytest.approx(
        0.8 * ((18569 / 22692) * (30000 / 26799)) ** 0.5)
    assert P.exemplar_rows_per_step(30000, 105) == 285           # SURVEY A.4 period 2
    assert P.loss_picks(5, 3) == [0] and P.loss_picks(5, 0) == []


@pytest.fixture(scope="module")
def sampler_herding(golden_dir):
    import sys
    sys.path.insert(0, golden_dir)
    import make_golden_sampler_herding as G
    with open(os.path.join(golden_dir, "sampler_herding.json")) as f:
        gold = json.load(f)
    return G, {k: v for k, v in gold.items() if k != "source"}


def test_sampler_and_herding_match_stored_outputs(sampler_herding):
    """The live comparison below on every machine: split, 2 * batch_num + 1 batches across two reshuffles and three herding
    cases, against tests/golden/sampler_herding.json."""
    G, gold = sampler_herding
    got = G.oracle_outputs()
    for key in ("valid", "train", "batches", "herding"):
        assert got[key] == gold[key], key


@pytest.mark.skipif(not refstub.available(), reason="reference tree not mounted")
def test_live_reference_sampler_and_herding(sampler_herding):
    G, gold = sampler_herding
    want = G.reference_outputs(refstub.load_reference_util())
    assert G.oracle_outputs() == want
    assert gold == want, "sampler_herding.json is not the reference's output: re-mint it with make_golden_sampler_herding.py"


def test_oracle_herding_matches_reference_on_large_segments(golden_dir):
    """oracle/protocol.py herding_picks against KATs minted from the reference's own ExemplarGenerator.herding on segments of
    400 .. 3 100 candidates (tests/golden/make_golden_herding_big.py)."""
    import sys
    import numpy as np
    from oracle import protocol as P
    sys.path.insert(0, golden_dir)
    from make_golden_herding_big import make_rep
    z = np.load(os.path.join(golden_dir, "herding_big.npz"))
    for c in range(len(z["n"])):
        rep = make_rep(int(z["seed"][c]), int(z["n"][c]))
        want = z["picks"][z["pick_off"][c]:z["pick_off"][c + 1]].tolist()
        assert P.herding_picks(rep, int(z["m"][c])) == want
