"""CPU checks of the AderLossArgs validation shared by every logits + CE + distillation entry: the exact and tcgen05 loss,
the two vocab-parallel halves and the fused training pass refuse the same malformed arguments before any CUDA call, so
fake non-null device addresses suffice."""
import ctypes as C

import pytest

from ader_b200 import _lib, build, ops
from ader_b200.params import Hyper

FAKE = 0x10000          # a non-null "device" address: never dereferenced, validation fails first
HP = Hyper(4000)        # item table of 4001 rows
N_TRAIN, N_EX, V, V_PREV = 128, 72, 3001, 2477


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.load()


def _args(mode=1, **over):
    """Valid arguments of the given mode (stored teacher logits in mode 1), then the fields in `over`."""
    a = ops.make_loss_args(N_TRAIN + N_EX, N_TRAIN, N_EX, V, V_PREV, mode, 0.8)
    a.pos = FAKE
    if mode == 1:
        a.teacher, a.teacher_ld = FAKE, V_PREV
    if mode == 2:
        a.ex_pos = FAKE
    for k, v in over.items():
        setattr(a, k, v)
    return a


# (arguments, a field name the refusal must contain)
BAD = {
    "rows": (lambda: _args(M=N_TRAIN + N_EX + 1), b"n_train + n_ex"),
    "V": (lambda: _args(V=HP.item_num + 1), b"max_item"),
    "mode3": (lambda: _args(mode=3), b"mode"),
    "pos": (lambda: _args(pos=None), b"pos"),
    "vanilla_with_exemplars": (lambda: _args(mode=0), b"vanilla mode"),
    "ex_pos": (lambda: _args(mode=2, ex_pos=None), b"exemplar_pos"),
    # the vocab-parallel entries refuse any frozen teacher first; both messages name teacher_rep
    "both_teachers": (lambda: _args(teacher_rep=FAKE, teacher_table=FAKE, teacher_table16=FAKE), b"teacher_rep"),
    "no_teacher": (lambda: _args(teacher=None), b"exactly one teacher source"),
    "teacher_ld": (lambda: _args(teacher_ld=V_PREV - 1), b"teacher_ld"),
    "V_prev": (lambda: _args(V_prev=V + 1, teacher_ld=V + 1), b"V_prev"),
}


def _call(lib, entry, a, ms):
    p = C.c_void_p(FAKE)
    if entry in ("ader_loss_fwd_bwd", "ader_loss_fwd_bwd_tc"):
        return getattr(lib, entry)(C.byref(ms), p, p, C.byref(a), p, p, p, p, p, None)
    if entry == "ader_loss_tc_vp_fwd":
        return lib.ader_loss_tc_vp_fwd(C.byref(ms), p, p, C.byref(a), 0, 1536, p, p, None)
    if entry == "ader_loss_tc_vp_bwd":
        return lib.ader_loss_tc_vp_bwd(C.byref(ms), p, p, C.byref(a), 0, 1536, p, p, p, p, None)
    assert entry == "ader_train_fwd_bwd_tc"      # serial plan: no library streams are created before the loss check
    return lib.ader_train_fwd_bwd_tc(C.byref(ms), p, p, a.M, a.M * 50, C.byref(a), p, p, p, p, p, p, p, p, 0.0, 0, None, 1, None)


@pytest.mark.parametrize("entry", ["ader_loss_fwd_bwd", "ader_loss_fwd_bwd_tc", "ader_loss_tc_vp_fwd",
                                   "ader_loss_tc_vp_bwd", "ader_train_fwd_bwd_tc"])
@pytest.mark.parametrize("case", sorted(BAD))
def test_every_loss_entry_refuses_bad_arguments(lib, entry, case):
    make, field = BAD[case]
    assert _call(lib, entry, make(), ops.model_struct(HP)) == -1
    assert field in lib.ader_last_error()


@pytest.mark.parametrize("mode,n_ex", [(0, 0), (1, 0), (1, 72), (1, 300), (2, 0), (2, 72)])
@pytest.mark.parametrize("V_prev", [128, 1000, V])
def test_one_shard_workspace_is_the_single_gpu_workspace(lib, mode, n_ex, V_prev):
    ms = ops.model_struct(HP)
    a = _args(mode, n_ex=n_ex, M=N_TRAIN + n_ex, V_prev=V_prev, teacher_ld=V_prev)
    assert lib.ader_loss_tc_vp_ws_bytes(C.byref(ms), C.byref(a), 0, V) == lib.ader_loss_tc_ws_bytes(C.byref(ms), C.byref(a)) > 0
