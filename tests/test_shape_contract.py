"""CPU checks of the shape contract of every kernel path: over the whole grid of model shapes the library accepts,
ader_path_check serves exactly the shapes the path's limit allows, and on every refused shape the path's entries refuse
with the query's own message before any CUDA call (fake non-null device addresses suffice).  The limits are written here
as plain formulas: the shared-memory tiles of the exact attention kernels in bytes, and hidden_units <= 160 for the paths
whose operands are padded to 160 columns."""
import ctypes as C

import pytest

from ader_b200 import _lib, build, ops
from ader_b200.params import Hyper

FAKE = C.c_void_p(0x10000)     # never dereferenced: the path check fails first
ITEMS = 4000
V = 3001


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.load()


def _heads(d):
    return sorted({1, 2 if d % 2 == 0 else 1, max(h for h in range(1, 17) if d % h == 0)})


GRID = [(d, L, h, nb) for d in range(2, 257, 2) for L in range(1, 65) for h in _heads(d) for nb in (1, 8)]


def _ceil4(x):
    return (x + 3) // 4 * 4


def attn_fwd_bytes(d, L):
    """k_attn_fwd: K^T and V^T [d][LP], the row's queries [L*d], one 256-float scratch per warp (8 warps)."""
    return 4 * (2 * d * _ceil4(L) + _ceil4(L * d) + 8 * 256)


def attn_bwd_bytes(d, L):
    """k_attn_bwd: K^T and V^T [d][LP], Q, K and dY [L*d] each, three [L][LP] score tiles."""
    return 4 * (2 * d * _ceil4(L) + 3 * _ceil4(L * d) + 3 * L * _ceil4(L))


FWD_OK = lambda d, L: attn_fwd_bytes(d, L) <= 200 * 1024
BWD_OK = lambda d, L: attn_bwd_bytes(d, L) <= 220 * 1024
TC_OK = lambda d, L: d <= 160

LIMITS = {
    ops.PATH_ENCODER_FWD: FWD_OK,
    ops.PATH_ENCODER_BWD: BWD_OK,
    ops.PATH_ENCODER_TC: TC_OK,
    ops.PATH_LOSS_TC: TC_OK,
    ops.PATH_EVAL_TC: TC_OK,
    ops.PATH_FISHER_BATCHED: lambda d, L: d <= 160 and FWD_OK(d, L) and BWD_OK(d, L),
    ops.PATH_HERDING_ONCHIP: TC_OK,
}


def _ms(d, L, h, nb):
    return ops.model_struct(Hyper(ITEMS, d, L, nb, h))


def _loss_args(M):
    a = ops.make_loss_args(M, M, 0, V)
    a.pos = FAKE
    return a


def _adam_args():
    return _lib.AderAdamArgs(1e-3, 0.9, 0.98, 1e-8, V, 0.0, None, None)


# entries of each path, called with valid arguments for a batch of 4 sessions
M = 4
ENTRIES = {
    ops.PATH_ENCODER_FWD: {
        "ader_encoder_fwd": lambda lib, ms: lib.ader_encoder_fwd(C.byref(ms), FAKE, FAKE, M, M, FAKE, FAKE, 0.0, 0, None),
    },
    ops.PATH_ENCODER_BWD: {
        "ader_encoder_bwd": lambda lib, ms: lib.ader_encoder_bwd(C.byref(ms), FAKE, FAKE, M, M, FAKE, FAKE, FAKE, FAKE, 0.0, 0, None),
    },
    ops.PATH_ENCODER_TC: {
        "ader_encoder_fwd_tc": lambda lib, ms: lib.ader_encoder_fwd_tc(C.byref(ms), FAKE, FAKE, M, M, FAKE, FAKE, 0.0, 0, None, None),
        "ader_encoder_bwd_tc": lambda lib, ms: lib.ader_encoder_bwd_tc(C.byref(ms), FAKE, FAKE, M, M, FAKE, FAKE, FAKE, FAKE, 0.0, 0,
                                                                       None, None),
    },
    ops.PATH_LOSS_TC: {
        "ader_loss_fwd_bwd_tc": lambda lib, ms: lib.ader_loss_fwd_bwd_tc(C.byref(ms), FAKE, FAKE, C.byref(_loss_args(M)), FAKE, FAKE,
                                                                         FAKE, FAKE, FAKE, None),
        "ader_loss_tc_vp_fwd": lambda lib, ms: lib.ader_loss_tc_vp_fwd(C.byref(ms), FAKE, FAKE, C.byref(_loss_args(M)), 0, 1536, FAKE,
                                                                       FAKE, None),
        "ader_loss_tc_vp_bwd": lambda lib, ms: lib.ader_loss_tc_vp_bwd(C.byref(ms), FAKE, FAKE, C.byref(_loss_args(M)), 0, 1536, FAKE,
                                                                       FAKE, FAKE, FAKE, None),
        "ader_pack_table16": lambda lib, ms: lib.ader_pack_table16(C.byref(ms), FAKE, V, FAKE, None),
        # serial plan: no library streams are created before the checks
        "ader_train_fwd_bwd_tc": lambda lib, ms: lib.ader_train_fwd_bwd_tc(C.byref(ms), FAKE, FAKE, M, M, C.byref(_loss_args(M)), FAKE,
                                                                           FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, 0.0, 0, None, 1, None),
        "ader_train_step_tc": lambda lib, ms: lib.ader_train_step_tc(C.byref(ms), FAKE, FAKE, M, M, C.byref(_loss_args(M)), FAKE, FAKE,
                                                                     FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, 0.0, 0, None, FAKE, FAKE, FAKE,
                                                                     C.byref(_adam_args()), 1, None),
    },
    ops.PATH_EVAL_TC: {
        "ader_eval_rank_tc": lambda lib, ms: lib.ader_eval_rank_tc(C.byref(ms), FAKE, FAKE, FAKE, M, V, FAKE, FAKE, FAKE, None),
        "ader_eval_rank_topk_tc": lambda lib, ms: lib.ader_eval_rank_topk_tc(C.byref(ms), FAKE, FAKE, FAKE, M, V, 20, FAKE, FAKE, FAKE,
                                                                             FAKE, FAKE, None),
        "ader_recommend_topk_tc": lambda lib, ms: lib.ader_recommend_topk_tc(C.byref(ms), FAKE, FAKE, FAKE, M, V, 20, FAKE, FAKE, FAKE,
                                                                             FAKE, None),
    },
    ops.PATH_FISHER_BATCHED: {
        "ader_fisher_batched": lambda lib, ms: lib.ader_fisher_batched(C.byref(ms), FAKE, FAKE, FAKE, M, M, V, FAKE, FAKE, FAKE, FAKE,
                                                                       None),
    },
    ops.PATH_HERDING_ONCHIP: {},     # never refused: wider models run the first-generation kernel
}

# workspace queries of a path: 0 (with the query's message) on a refused shape
WS_QUERIES = {
    ops.PATH_LOSS_TC: [lambda lib, ms: lib.ader_table16_ws_bytes(C.byref(ms), V)],
    ops.PATH_EVAL_TC: [lambda lib, ms: lib.ader_eval_rank_tc_ws_bytes(C.byref(ms), M, V),
                       lambda lib, ms: lib.ader_recommend_tc_ws_bytes(C.byref(ms), M, V)],
    ops.PATH_FISHER_BATCHED: [lambda lib, ms: lib.ader_fisher_batched_ws_bytes(C.byref(ms), M, V)],
}


def test_grid_is_the_accepted_grid(lib):
    for d, L, h, nb in GRID:
        assert lib.ader_param_count(C.byref(_ms(d, L, h, nb))) > 0, (d, L, h, nb)
    assert lib.ader_param_count(C.byref(_ms(258, 50, 1, 1))) == -1
    assert lib.ader_param_count(C.byref(_ms(150, 65, 1, 1))) == -1


@pytest.mark.parametrize("path", sorted(LIMITS))
def test_path_check_serves_exactly_the_stated_limit(lib, path):
    limit = LIMITS[path]
    for d, L, h, nb in GRID:
        ms = _ms(d, L, h, nb)
        rc = lib.ader_path_check(C.byref(ms), path)
        assert rc == (0 if limit(d, L) else -1), (path, d, L, h, nb)
        if rc:
            msg = lib.ader_last_error()
            assert b"hidden_units=%d" % d in msg and b"maxlen=%d" % L in msg, msg
            tile_limit = path in (ops.PATH_ENCODER_FWD, ops.PATH_ENCODER_BWD) or (path == ops.PATH_FISHER_BATCHED and d <= 160)
            assert (b"shared memory" in msg) if tile_limit else (b"hidden_units <= 160" in msg), msg


def test_attention_thresholds():
    """The edges the GPU shape tests are built around (tests/test_gpu_shapes.py)."""
    assert BWD_OK(136, 64) and not BWD_OK(138, 64)
    assert BWD_OK(190, 50) and not BWD_OK(192, 50)
    assert BWD_OK(256, 40) and not BWD_OK(256, 41)
    assert attn_fwd_bytes(256, 64) == 200 * 1024          # the widest, longest model fills the forward budget exactly
    assert all(FWD_OK(d, L) for d, L, _, _ in GRID)


@pytest.mark.parametrize("path", sorted(LIMITS))
def test_entries_refuse_before_any_cuda_call(lib, path):
    limit = LIMITS[path]
    refused = 0
    for d, L, h, nb in GRID:
        if limit(d, L):
            continue
        refused += 1
        ms = _ms(d, L, h, nb)
        assert lib.ader_path_check(C.byref(ms), path) == -1
        want = lib.ader_last_error()
        for name, call in ENTRIES[path].items():
            assert call(lib, ms) == -1, (name, d, L, h, nb)
            assert lib.ader_last_error() == want, (name, d, L)
        for q in WS_QUERIES.get(path, []):
            assert q(lib, ms) == 0, (path, d, L)
            assert lib.ader_last_error() == want
    assert (refused == 0) == (path == ops.PATH_ENCODER_FWD)


@pytest.mark.parametrize("N", [1, 1000, 4097])
def test_herding_workspace_holds_the_first_generation_rows(lib, N):
    """k_herding (every segment of hidden_units > 160) writes N rows of max(d, 160) floats before the rest of the carve."""
    al = lambda n: (n + 255) // 256 * 256
    for d in range(2, 257, 2):
        ms = _ms(d, 50, 1, 1)
        want = al(4 * N * max(d, 160)) + al(4 * N) + 4 * al(4 * N) + 256
        assert lib.ader_herding_ws_bytes(C.byref(ms), N) >= want, d


def test_python_query(lib):
    assert ops.path_check(_ms(150, 50, 1, 2), ops.PATH_ENCODER_BWD) is None
    msg = ops.path_check(_ms(150, 64, 1, 2), ops.PATH_ENCODER_BWD)
    assert "hidden_units=150" in msg and "maxlen=64" in msg
    assert str(attn_bwd_bytes(150, 64)) in msg and str(220 * 1024) in msg
    assert "<= 160" in ops.path_check(_ms(162, 50, 1, 2), ops.PATH_LOSS_TC)
