"""CPU checks of the recommendation entry points and command: argument refusals of the three C entries (they return
before any device work), and the session-file parsing, packing and output format of ``python -m ader_b200.recommend``."""
import ctypes as C

import numpy as np
import pytest

from ader_b200 import _lib, build, ops, recommend
from ader_b200.params import Hyper, ParamLayout

P = C.c_void_p(256)          # a non-NULL pointer: every call below is refused before it is dereferenced


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.load()


def _ms(item_num=1000, d=150):
    return ops.model_struct(Hyper(item_num, d))


def _exact(lib, ms, theta=P, rep=P, ws=P, items=P, scores=P, R=8, V=900, k=20):
    return lib.ader_recommend_topk(C.byref(ms), theta, rep, None, R, V, k, ws, items, scores, None)


def _tc(lib, ms, theta=P, rep=P, ws=P, items=P, scores=P, over=P, R=8, V=900, k=20):
    return lib.ader_recommend_topk_tc(C.byref(ms), theta, rep, None, R, V, k, ws, items, scores, over, None)


@pytest.mark.parametrize("entry", [_exact, _tc], ids=["exact", "tc"])
@pytest.mark.parametrize("null", ["theta", "rep", "ws", "items", "scores"])
def test_null_pointers_are_refused(lib, entry, null):
    assert entry(lib, _ms(), **{null: None}) == -1
    assert b"NULL" in lib.ader_last_error()


def test_tc_null_overflow_is_refused(lib):
    assert _tc(lib, _ms(), over=None) == -1


@pytest.mark.parametrize("entry", [_exact, _tc], ids=["exact", "tc"])
@pytest.mark.parametrize("kw", [dict(k=0), dict(k=101), dict(k=-1), dict(R=0), dict(V=0), dict(V=1001)],
                         ids=["k0", "k101", "kneg", "R0", "V0", "V_outside_table"])
def test_bad_sizes_are_refused(lib, entry, kw):
    assert entry(lib, _ms(), **kw) == -1
    assert b"bad sizes" in lib.ader_last_error()


def test_tc_refuses_wide_hidden(lib):
    assert _tc(lib, _ms(d=200)) == -1
    assert b"hidden_units" in lib.ader_last_error()


def test_bad_model_is_refused(lib):
    ms = _lib.AderModel(1001, 151, 50, 2, 1)
    assert _exact(lib, ms) == -1 and _tc(lib, ms) == -1


def test_ws_queries(lib):
    ms = _ms(43104)
    n = lib.ader_recommend_tc_ws_bytes(C.byref(ms), 4096, 43104)
    assert n >= lib.ader_eval_rank_tc_ws_bytes(C.byref(ms), 4096, 43104) + 4096 * 65 * 4
    assert lib.ader_recommend_tc_ws_bytes(C.byref(ms), 0, 43104) == 0
    assert lib.ader_recommend_tc_ws_bytes(C.byref(ms), 4096, 0) == 0
    assert lib.ader_recommend_tc_ws_bytes(C.byref(_ms(43104, 200)), 4096, 43104) == 0
    with pytest.raises(_lib.AderError):
        ops.recommend_tc_ws_bytes(ms, 0, 10)


# ---- the command ----------------------------------------------------------------------------------------------------
def test_read_sessions(tmp_path):
    f = tmp_path / "s.txt"
    f.write_text("3 1 2\n  7\t8 \n5\n")
    assert recommend.read_sessions(str(f), 10) == [[3, 1, 2], [7, 8], [5]]


@pytest.mark.parametrize("text,line,what", [("1 2\n\n3\n", 2, "empty"), ("1 2\n3 10\n", 2, "outside 1..9"),
                                            ("0 1\n", 1, "outside 1..9"), ("4 x\n", 1, "integers"), ("1\n  \n", 2, "empty")])
def test_read_sessions_names_the_bad_line(tmp_path, text, line, what):
    f = tmp_path / "s.txt"
    f.write_text(text)
    with pytest.raises(ValueError, match=r":%d: .*%s" % (line, what.replace(".", r"\."))):
        recommend.read_sessions(str(f), 10)


def test_bad_line_exits_with_its_number(tmp_path, monkeypatch):
    f = tmp_path / "s.txt"
    f.write_text("1 2\n\n")
    monkeypatch.setattr(recommend, "load_model", lambda path: (type("M", (), {"hp": Hyper(9)})(), 9))
    with pytest.raises(SystemExit, match=":2: empty"):
        recommend.main(["--checkpoint", "c.pt", "--sessions", str(f), "--out", str(tmp_path / "o.txt")])


def test_session_rows_are_right_aligned_and_truncated():
    ids, n_in = recommend.session_rows([[4, 5, 6], list(range(1, 9)), [9]], 5)
    assert ids.dtype == np.int32 and ids.shape == (3, 5)
    assert ids.tolist() == [[0, 0, 4, 5, 6], [4, 5, 6, 7, 8], [0, 0, 0, 0, 9]]
    assert n_in.tolist() == [3, 5, 1]


def test_format_line():
    assert recommend.format_line(np.array([5, 2, 0], np.int32)) == "5 2 0"
    s = np.array([1.5, np.float32(0.1), -np.inf], np.float32)
    line = recommend.format_line([5, 2, 0], s)
    assert line == "5:1.5 2:0.100000001 0:-inf"
    assert [np.float32(x.split(":")[1]) for x in line.split()] == list(s)    # round-trips the fp32 score


def test_model_shape_from_checkpoint():
    import torch
    hp = Hyper(700, 150, 50, 2, 1)
    st = {"args": {"hidden_units": 150, "maxlen": 50, "num_blocks": 2, "num_heads": 1},
          "model": {"theta": torch.zeros(ParamLayout(hp).total)}}
    assert recommend.model_shape(st) == hp
    st["model"]["theta"] = torch.zeros(ParamLayout(hp).total + 7)
    with pytest.raises(ValueError):
        recommend.model_shape(st)
    with pytest.raises(ValueError):
        recommend.model_shape({"args": None, "model": {"theta": torch.zeros(10)}})


@pytest.mark.parametrize("argv", [["--k", "0"], ["--k", "101"], ["--batch", "0"]])
def test_cli_refuses_bad_options(argv):
    with pytest.raises(SystemExit):
        recommend.main(["--checkpoint", "c.pt", "--sessions", "s.txt", "--out", "o.txt", *argv])
