"""CPU checks of the frozen-teacher arguments of the C ABI (AderLossArgs.teacher_rep / teacher_table / teacher_table16):
every rejection below happens in argument validation, before any launch, so fake non-null device addresses suffice."""
import ctypes as C

import pytest

from ader_b200 import _lib, build, ops
from ader_b200.params import Hyper

FAKE = 0x10000          # a non-null "device" address: never dereferenced, validation fails first


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.load()


def _args(teacher=False, frozen=False, table=True, table16=True, n_ex=200, V=3001, V_prev=2477):
    a = ops.make_loss_args(n_ex, 0, n_ex, V, V_prev, 1, 0.8)
    a.teacher_ld = V_prev
    if teacher:
        a.teacher = FAKE
    if frozen:
        a.teacher_rep = FAKE
        a.teacher_table = FAKE if table else None
        a.teacher_table16 = FAKE if table16 else None
    return a


def _call(lib, fn, a, ms):
    p = C.c_void_p(FAKE)
    return fn(C.byref(ms), p, p, C.byref(a), p, p, p, p, p, None)


def test_abi_version_is_2(lib):
    assert lib.ader_abi_version() == 2 == _lib.ABI_VERSION


@pytest.mark.parametrize("entry", ["ader_loss_fwd_bwd", "ader_loss_fwd_bwd_tc"])
@pytest.mark.parametrize("both", [True, False], ids=["both", "neither"])
def test_exactly_one_teacher_source(lib, entry, both):
    ms = ops.model_struct(Hyper(4000))
    a = _args(teacher=both, frozen=both)
    assert _call(lib, getattr(lib, entry), a, ms) == -1
    assert b"exactly one teacher source" in lib.ader_last_error()


def test_exact_entry_needs_the_fp32_table(lib):
    ms = ops.model_struct(Hyper(4000))
    assert _call(lib, lib.ader_loss_fwd_bwd, _args(frozen=True, table=False), ms) == -1
    assert b"teacher_table" in lib.ader_last_error()


def test_tc_entries_need_the_bf16_table(lib):
    ms = ops.model_struct(Hyper(4000))
    a = _args(frozen=True, table16=False)
    assert _call(lib, lib.ader_loss_fwd_bwd_tc, a, ms) == -1
    assert b"teacher_table16" in lib.ader_last_error()
    p = C.c_void_p(FAKE)
    # the fused training pass validates the loss arguments in its first (serial) phase, before the encoder is launched
    rc = lib.ader_train_fwd_bwd_tc(C.byref(ms), p, p, a.M, a.M * 50, C.byref(a), p, p, p, p, p, p, p, p, 0.0, 0, None, 1, None)
    assert rc == -1 and b"teacher_table16" in lib.ader_last_error()


def test_teacher_width_is_checked(lib):
    ms = ops.model_struct(Hyper(4000))
    assert _call(lib, lib.ader_loss_fwd_bwd, _args(frozen=True, V_prev=3002), ms) == -1
    assert b"V_prev" in lib.ader_last_error()


def test_vocab_parallel_refuses_a_frozen_teacher(lib):
    ms = ops.model_struct(Hyper(4000))
    a = _args(frozen=True)
    p = C.c_void_p(FAKE)
    assert lib.ader_loss_tc_vp_fwd(C.byref(ms), p, p, C.byref(a), 0, 1536, p, p, None) == -1
    assert b"frozen teacher" in lib.ader_last_error()
    assert lib.ader_loss_tc_vp_bwd(C.byref(ms), p, p, C.byref(a), 0, 1536, p, p, p, p, None) == -1
    assert lib.ader_loss_tc_vp_ws_bytes(C.byref(ms), C.byref(a), 0, 1536) == 0


def _al(x):
    return (x + 255) // 256 * 256


@pytest.mark.parametrize("n_ex,V_prev", [(200, 2477), (138, 17421), (128, 128)])
def test_workspace_queries_grow_by_the_snapshot_buffers(lib, n_ex, V_prev):
    ms = ops.model_struct(Hyper(25958))
    V = 18661
    stored, frozen = _args(teacher=True, n_ex=n_ex, V=V, V_prev=V_prev), _args(frozen=True, n_ex=n_ex, V=V, V_prev=V_prev)
    # exact: gathered reps [n_ex, d] + teacher logits [n_ex, ld(V_prev)] fp32
    ld = (V_prev + 3) // 4 * 4
    grow = lib.ader_loss_ws_bytes(C.byref(ms), C.byref(frozen)) - lib.ader_loss_ws_bytes(C.byref(ms), C.byref(stored))
    assert grow == _al(4 * n_ex * 150) + _al(4 * n_ex * ld)
    # tcgen05: packed bf16 reps + per-chunk statistics + log-sum-exp of the padded exemplar rows
    n_et = (n_ex - 1) // 128 + 1                 # exemplar row tiles (n_train = 0: the rows start at tile 0)
    tc_s = lib.ader_loss_tc_ws_bytes(C.byref(ms), C.byref(stored))
    tc_f = lib.ader_loss_tc_ws_bytes(C.byref(ms), C.byref(frozen))
    assert tc_f - tc_s >= _al(n_et * 128 * 160 * 2) + _al(4 * 4 * 2 * n_et * 128) + _al(4 * n_et * 128)
    # the queries of the stored form are those of the parent ABI (nothing grows without a snapshot)
    stored.teacher_rep = None
    assert lib.ader_loss_tc_ws_bytes(C.byref(ms), C.byref(stored)) == tc_s


def test_table16_size_query(lib):
    ms = ops.model_struct(Hyper(25958))
    assert lib.ader_table16_ws_bytes(C.byref(ms), 17421) == 137 * 128 * 160 * 2
    assert lib.ader_table16_ws_bytes(C.byref(ms), 128) == 128 * 160 * 2
    assert lib.ader_table16_ws_bytes(C.byref(ms), 0) == 0
    p = C.c_void_p(FAKE)
    assert lib.ader_pack_table16(C.byref(ms), p, 25959, p, None) == -1          # beyond the table
    assert lib.ader_pack_table16(C.byref(ms), None, 100, p, None) == -1
    big = ops.model_struct(Hyper(1000, 192, 50, 2, 1))
    assert lib.ader_pack_table16(C.byref(big), p, 100, p, None) == -1           # hidden_units > 160
    assert lib.ader_table16_ws_bytes(C.byref(big), 100) == 0                    # ... and no size for it either


def test_driver_flag_and_protocol_key():
    from ader_b200.main import PROTOCOL_DEFAULTS, build_parser, protocol_args
    a = build_parser().parse_args([])
    assert a.teacher == "logits"
    assert build_parser().parse_args(["--teacher", "frozen"]).teacher == "frozen"
    with pytest.raises(SystemExit):
        build_parser().parse_args(["--teacher", "bf16"])
    assert protocol_args(a)["teacher"] == "logits"
    assert PROTOCOL_DEFAULTS["teacher"] == "logits"      # checkpoints written before the flag existed resume as "logits"


def test_generator_rejects_an_unknown_teacher_form():
    from ader_b200.data import ExemplarGenerator
    with pytest.raises(ValueError):
        ExemplarGenerator([[1, 2, 3]], 10, False, 4, 5, 0.0, 3, teacher="bf16")
