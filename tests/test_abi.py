"""CPU checks of the C-ABI boundary: the library builds, loads, exports every symbol that
include/ader_b200.h declares, and its layout introspection agrees with the Python layout and
the oracle's parameter order.  No compute calls (no GPU here)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from ader_b200 import _lib, build, ops
from ader_b200.params import Hyper, ParamLayout

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.load()


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "ader_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(ader_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_exported_and_bound(lib):
    syms = _declared_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(lib, s), "symbol %s declared in include/ader_b200.h but not exported" % s
        assert s in _lib.SIGNATURES, "symbol %s has no ctypes signature" % s
    assert sorted(_lib.SIGNATURES) == syms


def test_abi_version(lib):
    assert lib.ader_abi_version() == _lib.ABI_VERSION


@pytest.mark.parametrize("hp", [Hyper(43136), Hyper(25958), Hyper(1000000), Hyper(60, 12, 10, 3, 2)])
def test_layout_agrees(lib, hp):
    from oracle import sasrec as S
    lay = ParamLayout(hp)
    ms = ops.model_struct(hp)
    assert lib.ader_param_count(C.byref(ms)) == lay.total
    assert lib.ader_dense_count(C.byref(ms)) == lay.dense_count
    shapes = S.param_shapes(S.Hyper(hp.item_num, hp.hidden_units, hp.maxlen, hp.num_blocks, hp.num_heads))
    assert [n for n, _ in shapes] == lay.names()
    off = 0
    for i, (name, shape) in enumerate(shapes):
        assert lib.ader_param_offset(C.byref(ms), i) == off == lay.offset(i), name
        off += int(np.prod(shape))


def test_init_matches_oracle_init():
    from oracle import sasrec as S
    hp = Hyper(300, 150, 50, 2, 1)
    flat = ParamLayout(hp).init_flat(7)
    want = np.concatenate([p.numpy().ravel() for p in S.init_params(S.Hyper(300), 7)])
    assert np.array_equal(flat, want)


def test_bad_model_is_rejected(lib):
    ms = _lib.AderModel(10, 151, 50, 2, 1)            # odd hidden size
    assert lib.ader_param_count(C.byref(ms)) == -1
    assert b"hidden_units" in lib.ader_last_error()
    ms = _lib.AderModel(100, 150, 50, 2, 4)           # heads do not divide d
    assert lib.ader_encoder_ws_bytes(C.byref(ms), 4, 200) == 0


def test_workspace_queries(lib):
    ms = ops.model_struct(Hyper(43136))
    a = lib.ader_encoder_ws_bytes(C.byref(ms), 608, 608 * 50)
    b = lib.ader_encoder_ws_bytes(C.byref(ms), 608, 3000)
    assert a > b > 0
    assert lib.ader_encoder_ws_slot(C.byref(ms), 608, 3000, 0, 0) >= 0
    assert lib.ader_encoder_ws_slot(C.byref(ms), 608, 3000, 0, 2) == -1
    assert lib.ader_eval_ws_bytes(C.byref(ms), 64, 43105) >= 64 * 43105 * 4
    assert lib.ader_herding_ws_bytes(C.byref(ms), 1000) >= 1000 * 150 * 4


def test_ops_refuse_cpu_tensors():
    import torch
    hp = Hyper(100)
    ms = ops.model_struct(hp)
    t = torch.zeros(4)
    with pytest.raises(_lib.AderError):
        ops.logits(ms, t, t, 10, t)


def test_model_needs_cuda():
    import torch
    from ader_b200.model import Ader
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    args = type("A", (), dict(hidden_units=150, maxlen=50, num_blocks=2, num_heads=1, random_seed=0, lr=5e-4, dropout_rate=0.0))()
    with pytest.raises(RuntimeError):
        Ader(100, args)


def test_every_compute_entry_point_is_a_torch_op(lib):
    """north_star: the C ABI is 'exposed as PyTorch custom ops'.  Every entry point that launches device work is registered
    as torch.ops.ader_b200.<name>; size queries, introspection, IPC plumbing, status reads and debug hooks are host helpers."""
    import torch
    ops.register_torch_ops()
    host_only = ("_ws_bytes", "_ws_slot", "abi_version", "last_error", "param_count", "param_offset", "dense_count", "ipc_",
                 "dp_status", "debug_", "eval_topk_chunks", "path_check")
    want = sorted(s[len("ader_"):] for s in _declared_symbols() if not any(h in s for h in host_only))
    assert want == ops.registered_op_names()
    for name in want:
        assert hasattr(torch.ops.ader_b200, name)
