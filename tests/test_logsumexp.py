"""CPU checks of the log-sum-exp entries (ader_logsumexp, ader_logsumexp_tc and the tc workspace query): argument refusals
that name the entry and the field, the shape contract of the tensor-core entry over the whole accepted grid (it refuses
exactly where ader_path_check(ADER_PATH_EVAL_TC) does, with the same message, before any CUDA call), and the --probs
option of ``python -m ader_b200.recommend``."""
import ctypes as C

import numpy as np
import pytest

from ader_b200 import _lib, build, ops, recommend
from ader_b200.params import Hyper

P = C.c_void_p(0x10000)      # a non-NULL pointer: every call below is refused before it is dereferenced


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.load()


def _ms(item_num=1000, d=150, L=50, h=1, nb=2):
    return ops.model_struct(Hyper(item_num, d, L, nb, h))


def _call(lib, entry, ms, theta=P, rep=P, gt=P, R=8, V=900, ws=P, lse=P, nll=P):
    fn = lib.ader_logsumexp if entry == "logsumexp" else lib.ader_logsumexp_tc
    return fn(C.byref(ms), theta, rep, gt, R, V, ws, lse, nll, None)


ENTRIES = ["logsumexp", "logsumexp_tc"]


@pytest.mark.parametrize("entry", ENTRIES)
@pytest.mark.parametrize("null", ["theta", "rep", "ws", "lse"])
def test_null_pointers_are_refused(lib, entry, null):
    assert _call(lib, entry, _ms(), **{null: None}) == -1
    assert lib.ader_last_error() == b"%s: %s is NULL" % (entry.encode(), null.encode())


@pytest.mark.parametrize("entry", ENTRIES)
@pytest.mark.parametrize("R", [0, -3])
def test_bad_row_count_is_refused(lib, entry, R):
    assert _call(lib, entry, _ms(), R=R) == -1
    msg = lib.ader_last_error()
    assert msg.startswith(entry.encode() + b":") and b"R must be > 0" in msg


@pytest.mark.parametrize("entry", ENTRIES)
@pytest.mark.parametrize("V", [0, -1, 1001, 5000])
def test_vocabulary_outside_the_table_is_refused(lib, entry, V):
    assert _call(lib, entry, _ms(item_num=1000), V=V) == -1
    msg = lib.ader_last_error()
    assert msg.startswith(entry.encode() + b":") and b"V=%d" % V in msg and b"1..1000" in msg


@pytest.mark.parametrize("entry", ENTRIES)
def test_nll_goes_with_gt(lib, entry):
    assert _call(lib, entry, _ms(), nll=None) == -1
    assert lib.ader_last_error() == b"%s: gt is given but nll is NULL" % entry.encode()
    assert _call(lib, entry, _ms(), gt=None) == -1
    assert lib.ader_last_error() == b"%s: nll is given but gt is NULL" % entry.encode()


@pytest.mark.parametrize("entry", ENTRIES)
def test_bad_model_is_refused(lib, entry):
    assert _call(lib, entry, _lib.AderModel(1001, 151, 50, 2, 1)) == -1
    assert b"hidden_units" in lib.ader_last_error()


def test_workspace_query(lib):
    ms = _ms(item_num=50000)
    for R, V in ((1, 1), (129, 33), (4096, 43105)):
        n = lib.ader_logsumexp_tc_ws_bytes(C.byref(ms), R, V)
        # the evaluation carve plus one (max, sum) pair per (chunk, column half) of every row
        assert n >= lib.ader_eval_rank_tc_ws_bytes(C.byref(ms), R, V) + 8 * R * 2 * lib.ader_eval_topk_chunks(C.byref(ms), R, V)
    assert lib.ader_logsumexp_tc_ws_bytes(C.byref(ms), 0, 100) == 0
    assert lib.ader_logsumexp_tc_ws_bytes(C.byref(ms), 8, 0) == 0


def _heads(d):
    return sorted({1, 2 if d % 2 == 0 else 1, max(h for h in range(1, 17) if d % h == 0)})


def test_tc_entry_refuses_exactly_where_the_path_check_does(lib):
    """Every accepted (hidden_units, maxlen, heads, blocks): served iff ader_path_check serves ADER_PATH_EVAL_TC; on a
    refused shape the entry returns -1 and the query 0, both with the path check's own message (the fake addresses are
    never touched, so no CUDA call was made)."""
    served = refused = 0
    for d in range(2, 257, 2):
        for L in (1, 33, 50, 64):
            for h in _heads(d):
                for nb in (1, 8):
                    ms = _ms(4000, d, L, h, nb)
                    rc = lib.ader_path_check(C.byref(ms), ops.PATH_EVAL_TC)
                    assert rc == (0 if d <= 160 else -1), (d, L)
                    if rc == 0:
                        served += 1
                        assert lib.ader_logsumexp_tc_ws_bytes(C.byref(ms), 4, 3001) > 0
                        continue
                    refused += 1
                    want = lib.ader_last_error()
                    assert b"hidden_units=%d" % d in want and b"maxlen=%d" % L in want
                    assert _call(lib, "logsumexp_tc", ms, R=4, V=3001) == -1
                    assert lib.ader_last_error() == want
                    assert _call(lib, "logsumexp_tc", ms, R=4, V=3001, gt=None, nll=None) == -1
                    assert lib.ader_last_error() == want
                    assert lib.ader_logsumexp_tc_ws_bytes(C.byref(ms), 4, 3001) == 0
                    assert lib.ader_last_error() == want
    assert served and refused


# ---- python -m ader_b200.recommend --probs ------------------------------------------------------------------------------
def test_probs_and_scores_exclude_each_other(capsys):
    p = recommend.build_parser()
    base = ["--checkpoint", "c.pt", "--sessions", "s.txt", "--out", "o.txt"]
    assert p.parse_args(base + ["--probs"]).probs
    assert not p.parse_args(base).probs
    with pytest.raises(SystemExit):
        p.parse_args(base + ["--probs", "--scores"])
    assert "not allowed with argument" in capsys.readouterr().err
    with pytest.raises(SystemExit):           # the command refuses before it reads the checkpoint
        recommend.main(base + ["--scores", "--probs"])


def test_probability_line_format():
    probs = np.array([0.5, 0.25, 1.5e-7, 0.0], np.float32)
    line = recommend.format_line([7, 3, 12, 0], probs)
    toks = line.split()
    assert [int(t.split(":")[0]) for t in toks] == [7, 3, 12, 0]
    assert np.array_equal(np.array([np.float32(t.split(":")[1]) for t in toks]), probs)
    assert toks[-1] == "0:0"
