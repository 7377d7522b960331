"""Device ops of the ADER hot path: thin shims from torch tensors to the C ABI.

Each function below passes raw device pointers + the current CUDA stream to one entry point of
``libader_b200.so`` (include/ader_b200.h).  They are also registered as ``torch.ops.ader_b200.*``
custom ops (see ``register_torch_ops``) so the kernels are reachable from the dispatcher; the host
loop calls the shims directly to keep per-step overhead out of the way.  torch is used for device
memory and streams only.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import _lib
from ._lib import AderAdamArgs, AderLossArgs, AderModel, check
from .params import Hyper


def _require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise _lib.AderError("ader_b200 ops need CUDA tensors (no CPU fallback exists)")


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def model_struct(hp: Hyper) -> AderModel:
    return AderModel(hp.v_tab, hp.hidden_units, hp.maxlen, hp.num_blocks, hp.num_heads)


# kernel paths of ader_path_check (include/ader_b200.h ADER_PATH_*)
PATH_ENCODER_FWD, PATH_ENCODER_BWD, PATH_ENCODER_TC, PATH_LOSS_TC, PATH_EVAL_TC, PATH_FISHER_BATCHED, PATH_HERDING_ONCHIP = range(7)


def path_check(ms: AderModel, path: int) -> Optional[str]:
    """None when the kernel path ``path`` (PATH_*) serves the model shape, else the library's refusal, which names the
    limit, hidden_units and maxlen.  Host only: needs no device."""
    lib = _lib.load()
    if lib.ader_path_check(C.byref(ms), path) == 0:
        return None
    return lib.ader_last_error().decode("utf-8", "replace")


class Workspace:
    """Grow-only caller-owned device scratch (the C ABI never allocates)."""

    def __init__(self, device):
        self.device = device
        self.buf: Optional[torch.Tensor] = None

    def get(self, nbytes: int) -> torch.Tensor:
        if self.buf is None or self.buf.numel() < nbytes:
            self.buf = torch.empty(int(nbytes * 1.25) + 256, dtype=torch.uint8, device=self.device)
        return self.buf


def encoder_ws_bytes(ms: AderModel, M: int, Tcap: int) -> int:
    n = _lib.load().ader_encoder_ws_bytes(C.byref(ms), M, Tcap)
    if n == 0:
        raise _lib.AderError("encoder_ws_bytes: bad model / sizes")
    return n


def encoder_bwd_ws_bytes(ms: AderModel, M: int, Tcap: int) -> int:
    n = _lib.load().ader_encoder_bwd_ws_bytes(C.byref(ms), M, Tcap)
    if n == 0:
        raise _lib.AderError("encoder_bwd_ws_bytes: bad model / sizes")
    return n


def encoder_ws_slot(ms: AderModel, M: int, Tcap: int, slot: int, block: int = 0) -> int:
    return _lib.load().ader_encoder_ws_slot(C.byref(ms), M, Tcap, slot, block)


def encoder_fwd(ms: AderModel, theta, ids, Tcap: int, ws, rep, dropout_rate: float = 0.0, seed: int = 0,
                impl: str = "exact", d_step=None):
    """ids [M, maxlen] int32 -> rep [M, d] (ADER.py:25-85).  impl: "exact" (fp32) or "tc" (fused tensor-core path).
    d_step (tc only): device int32 step counter added to the dropout seed on the device (CUDA-graph replays)."""
    _require_cuda(theta, ids, ws, rep)
    lib = _lib.load()
    if impl == "tc":
        check(lib.ader_encoder_fwd_tc(C.byref(ms), _ptr(theta), _ptr(ids), ids.shape[0], Tcap, _ptr(ws), _ptr(rep),
                                      float(dropout_rate), C.c_uint64(seed), _ptr(d_step), _stream()), "encoder_fwd_tc")
        return
    if d_step is not None:
        raise _lib.AderError("d_step is only supported by the tc encoder")
    check(lib.ader_encoder_fwd(C.byref(ms), _ptr(theta), _ptr(ids), ids.shape[0], Tcap, _ptr(ws), _ptr(rep),
                               float(dropout_rate), C.c_uint64(seed), _stream()), "encoder_fwd")


def encoder_bwd(ms: AderModel, theta, ids, Tcap: int, ws, bwd_ws, d_rep, grad, dropout_rate: float = 0.0, seed: int = 0,
                impl: str = "exact", d_step=None):
    _require_cuda(theta, ids, ws, bwd_ws, d_rep, grad)
    lib = _lib.load()
    if impl == "tc":
        check(lib.ader_encoder_bwd_tc(C.byref(ms), _ptr(theta), _ptr(ids), ids.shape[0], Tcap, _ptr(ws), _ptr(bwd_ws),
                                      _ptr(d_rep), _ptr(grad), float(dropout_rate), C.c_uint64(seed), _ptr(d_step), _stream()),
              "encoder_bwd_tc")
        return
    if d_step is not None:
        raise _lib.AderError("d_step is only supported by the tc encoder")
    check(lib.ader_encoder_bwd(C.byref(ms), _ptr(theta), _ptr(ids), ids.shape[0], Tcap, _ptr(ws), _ptr(bwd_ws),
                               _ptr(d_rep), _ptr(grad), float(dropout_rate), C.c_uint64(seed), _stream()), "encoder_bwd")


def make_loss_args(M, n_train, n_ex, V, V_prev=0, mode=0, lambda_=0.0, pos=None, ex_pos=None,
                   teacher=None, teacher_row=None, n_train_global=0, n_ex_global=0,
                   teacher_rep=None, teacher_table=None, teacher_table16=None) -> AderLossArgs:
    """Distillation (mode 1) takes stored logits ``teacher`` [*, V_prev] or a frozen snapshot: ``teacher_rep`` [*, d] fp32,
    ``teacher_table`` fp32 rows of items 1..V_prev (exact entry) and ``teacher_table16`` (``pack_table16``, tcgen05 entries)."""
    a = AderLossArgs()
    a.M, a.n_train, a.n_ex, a.V, a.V_prev, a.mode, a.lambda_ = M, n_train, n_ex, V, V_prev, mode, lambda_
    a.pos = pos.data_ptr() if pos is not None else None
    a.ex_pos = ex_pos.data_ptr() if ex_pos is not None else None
    a.teacher = teacher.data_ptr() if teacher is not None else None
    a.teacher_row = teacher_row.data_ptr() if teacher_row is not None else None
    a.teacher_ld = teacher.stride(0) if teacher is not None else 0
    a.n_train_global, a.n_ex_global = n_train_global, n_ex_global
    a.teacher_rep = teacher_rep.data_ptr() if teacher_rep is not None else None
    a.teacher_table = teacher_table.data_ptr() if teacher_table is not None else None
    a.teacher_table16 = teacher_table16.data_ptr() if teacher_table16 is not None else None
    return a


def loss_ws_bytes(ms: AderModel, a: AderLossArgs) -> int:
    n = _lib.load().ader_loss_ws_bytes(C.byref(ms), C.byref(a))
    if n == 0:
        raise _lib.AderError("loss_ws_bytes: bad model / sizes")
    return n


def loss_fwd_bwd(ms: AderModel, theta, rep, a: AderLossArgs, ws, loss, row_loss, d_rep, grad):
    _require_cuda(theta, rep, ws, loss, row_loss, d_rep, grad)
    check(_lib.load().ader_loss_fwd_bwd(C.byref(ms), _ptr(theta), _ptr(rep), C.byref(a), _ptr(ws), _ptr(loss),
                                        _ptr(row_loss), _ptr(d_rep), _ptr(grad), _stream()), "loss_fwd_bwd")


def loss_tc_ws_bytes(ms: AderModel, a: AderLossArgs) -> int:
    n = _lib.load().ader_loss_tc_ws_bytes(C.byref(ms), C.byref(a))
    if n == 0:
        raise _lib.AderError("loss_tc_ws_bytes: bad model / sizes")
    return n


def loss_fwd_bwd_tc(ms: AderModel, theta, rep, a: AderLossArgs, ws, loss, row_loss, d_rep, grad):
    """tcgen05 fused logits + CE + KD forward/backward (bf16 operands, fp32 accumulation)."""
    _require_cuda(theta, rep, ws, loss, row_loss, d_rep, grad)
    check(_lib.load().ader_loss_fwd_bwd_tc(C.byref(ms), _ptr(theta), _ptr(rep), C.byref(a), _ptr(ws), _ptr(loss),
                                           _ptr(row_loss), _ptr(d_rep), _ptr(grad), _stream()), "loss_fwd_bwd_tc")


def train_fwd_bwd_tc(ms: AderModel, theta, ids, Tcap: int, a: AderLossArgs, enc_ws, bwd_ws, loss_ws, rep, loss, row_loss,
                     d_rep, grad, dropout_rate: float = 0.0, seed: int = 0, d_step=None, serial: bool = False):
    """encoder forward -> logits + CE + KD forward/backward -> encoder backward + scatter as one fork/join DAG of the
    same launches the three single-group entry points issue (bit-identical results; see include/ader_b200.h)."""
    _require_cuda(theta, ids, enc_ws, bwd_ws, loss_ws, rep, loss, row_loss, d_rep, grad)
    check(_lib.load().ader_train_fwd_bwd_tc(C.byref(ms), _ptr(theta), _ptr(ids), ids.shape[0], Tcap, C.byref(a), _ptr(enc_ws),
                                            _ptr(bwd_ws), _ptr(loss_ws), _ptr(rep), _ptr(loss), _ptr(row_loss), _ptr(d_rep),
                                            _ptr(grad), float(dropout_rate), C.c_uint64(seed), _ptr(d_step), int(bool(serial)),
                                            _stream()), "train_fwd_bwd_tc")


def train_step_tc(ms: AderModel, theta, ids, Tcap: int, a: AderLossArgs, enc_ws, bwd_ws, loss_ws, rep, loss, row_loss,
                  d_rep, grad, adam_m, adam_v, state, V: int, lr: float, dropout_rate: float = 0.0, seed: int = 0, d_step=None,
                  ewc_lambda: float = 0.0, fisher=None, theta_star=None, beta1=0.9, beta2=0.999, eps=1e-8, serial: bool = False):
    """train_fwd_bwd_tc + adam_step as one DAG (single GPU; bit-identical to the two calls)."""
    _require_cuda(theta, ids, enc_ws, bwd_ws, loss_ws, rep, loss, row_loss, d_rep, grad, adam_m, adam_v, state, fisher, theta_star)
    opt = AderAdamArgs(lr, beta1, beta2, eps, V, ewc_lambda,
                       fisher.data_ptr() if fisher is not None else None,
                       theta_star.data_ptr() if theta_star is not None else None)
    check(_lib.load().ader_train_step_tc(C.byref(ms), _ptr(theta), _ptr(ids), ids.shape[0], Tcap, C.byref(a), _ptr(enc_ws),
                                         _ptr(bwd_ws), _ptr(loss_ws), _ptr(rep), _ptr(loss), _ptr(row_loss), _ptr(d_rep),
                                         _ptr(grad), float(dropout_rate), C.c_uint64(seed), _ptr(d_step), _ptr(adam_m),
                                         _ptr(adam_v), _ptr(state), C.byref(opt), int(bool(serial)), _stream()), "train_step_tc")


def debug_loss_tc_kernels(ms: AderModel, theta, a: AderLossArgs, ws, grad):
    """Measurement hook: only k_tc_logits<FWD/DREP/DE> on a workspace prepared by loss_fwd_bwd_tc (same arguments)."""
    _require_cuda(theta, ws, grad)
    check(_lib.load().ader_debug_loss_tc_kernels(C.byref(ms), _ptr(theta), C.byref(a), _ptr(ws), _ptr(grad), _stream()),
          "debug_loss_tc_kernels")


def loss_tc_vp_ws_bytes(ms: AderModel, a: AderLossArgs, v_lo: int, v_hi: int) -> int:
    n = _lib.load().ader_loss_tc_vp_ws_bytes(C.byref(ms), C.byref(a), v_lo, v_hi)
    if n == 0:
        raise _lib.AderError("loss_tc_vp_ws_bytes: bad model / sizes")
    return n


def loss_tc_vp_fwd(ms: AderModel, theta, rep, a: AderLossArgs, v_lo: int, v_hi: int, ws, stats):
    _require_cuda(theta, rep, ws, stats)
    check(_lib.load().ader_loss_tc_vp_fwd(C.byref(ms), _ptr(theta), _ptr(rep), C.byref(a), v_lo, v_hi, _ptr(ws), _ptr(stats),
                                          _stream()), "loss_tc_vp_fwd")


def loss_tc_vp_bwd(ms: AderModel, theta, rep, a: AderLossArgs, v_lo: int, v_hi: int, ws, lse, d_rep_partial, grad):
    _require_cuda(theta, rep, ws, lse, d_rep_partial, grad)
    check(_lib.load().ader_loss_tc_vp_bwd(C.byref(ms), _ptr(theta), _ptr(rep), C.byref(a), v_lo, v_hi, _ptr(ws), _ptr(lse),
                                          _ptr(d_rep_partial), _ptr(grad), _stream()), "loss_tc_vp_bwd")


def table16_bytes(ms: AderModel, V: int) -> int:
    n = _lib.load().ader_table16_ws_bytes(C.byref(ms), V)
    if n == 0:
        raise _lib.AderError("table16_ws_bytes: bad model / sizes")
    return n


def pack_table16(ms: AderModel, rows, V: int, out):
    """out (uint8, table16_bytes(ms, V)) = bf16 [ceil(V/128)*128][160] shadow of ``rows`` (fp32 rows of items 1..V, stride d)."""
    _require_cuda(rows, out)
    if out.numel() * out.element_size() < table16_bytes(ms, V):
        raise _lib.AderError("pack_table16: output buffer too small")
    check(_lib.load().ader_pack_table16(C.byref(ms), _ptr(rows), V, _ptr(out), _stream()), "pack_table16")


def logits(ms: AderModel, theta, rep, V: int, out):
    """out [M, >=V] fp32 = rep . E[1..V]^T (ADER.py:90-91)."""
    _require_cuda(theta, rep, out)
    check(_lib.load().ader_logits(C.byref(ms), _ptr(theta), _ptr(rep), rep.shape[0], V, _ptr(out), out.stride(0),
                                  _stream()), "logits")


def adam_step(ms: AderModel, theta, m, v, grad, state, V: int, lr: float, ewc_lambda: float = 0.0,
              fisher=None, theta_star=None, beta1=0.9, beta2=0.999, eps=1e-8):
    _require_cuda(theta, m, v, grad, state, fisher, theta_star)
    a = AderAdamArgs(lr, beta1, beta2, eps, V, ewc_lambda,
                     fisher.data_ptr() if fisher is not None else None,
                     theta_star.data_ptr() if theta_star is not None else None)
    check(_lib.load().ader_adam_step(C.byref(ms), _ptr(theta), _ptr(m), _ptr(v), _ptr(grad), _ptr(state), C.byref(a),
                                     _stream()), "adam_step")


# ---- data parallel over peer memory (csrc/dp.cu) -------------------------------------------------------
def dp_comm(rank: int, world: int, theta_ptrs, grad_ptrs, flag_ptrs, separate_arrive: bool = False,
            mc_theta: int = 0, mc_grad: int = 0) -> "_lib.AderDpComm":
    """mc_theta / mc_grad: optional NVLS multicast addresses of the same buffers (0 = peer loads / stores)."""
    c = _lib.AderDpComm()
    c.rank, c.world, c.separate_arrive, c.reserved = rank, world, int(separate_arrive), 0
    for r in range(world):
        c.theta[r], c.grad[r], c.flags[r] = int(theta_ptrs[r]), int(grad_ptrs[r]), int(flag_ptrs[r])
    c.mc_theta, c.mc_grad = (int(mc_theta) or None), (int(mc_grad) or None)
    return c


def dp_wait(comm):
    check(_lib.load().ader_dp_wait(C.byref(comm), _stream()), "dp_wait")


def dp_adam_step(ms: AderModel, comm, m, v, state, V: int, lr: float, ewc_lambda: float = 0.0, fisher=None, theta_star=None,
                 beta1=0.9, beta2=0.999, eps=1e-8):
    _require_cuda(m, v, state, fisher, theta_star)
    a = AderAdamArgs(lr, beta1, beta2, eps, V, ewc_lambda,
                     fisher.data_ptr() if fisher is not None else None,
                     theta_star.data_ptr() if theta_star is not None else None)
    check(_lib.load().ader_dp_adam_step(C.byref(ms), C.byref(comm), _ptr(m), _ptr(v), _ptr(state), C.byref(a), _stream()),
          "dp_adam_step")


def dp_status(comm):
    err, ep = C.c_int32(0), C.c_uint32(0)
    check(_lib.load().ader_dp_status(C.byref(comm), C.byref(err), C.byref(ep)), "dp_status")
    return int(err.value), int(ep.value)


def ipc_export(t: torch.Tensor):
    """(64-byte handle, byte offset) of the device allocation behind tensor `t` (another process maps it with ipc_open)."""
    _require_cuda(t)
    h = (C.c_ubyte * 64)()
    off = C.c_int64(0)
    check(_lib.load().ader_ipc_export(_ptr(t), h, C.byref(off)), "ipc_export")
    return bytes(h), int(off.value)


def ipc_open(handle: bytes) -> int:
    base = C.c_void_p(0)
    buf = (C.c_ubyte * 64).from_buffer_copy(handle)
    check(_lib.load().ader_ipc_open(buf, C.byref(base)), "ipc_open")
    return int(base.value)


def ipc_close(base: int):
    check(_lib.load().ader_ipc_close(C.c_void_p(base)), "ipc_close")


def eval_ws_bytes(ms: AderModel, M: int, V: int) -> int:
    n = _lib.load().ader_eval_ws_bytes(C.byref(ms), M, V)
    if n == 0:
        raise _lib.AderError("eval_ws_bytes: bad model / sizes")
    return n


def eval_rank_topk(ms: AderModel, theta, rep, gt, V: int, k: int, ws, rank, topk_item, topk_score):
    _require_cuda(theta, rep, gt, ws, rank, topk_item, topk_score)
    check(_lib.load().ader_eval_rank_topk(C.byref(ms), _ptr(theta), _ptr(rep), _ptr(gt), rep.shape[0], V, k, _ptr(ws),
                                          _ptr(rank), _ptr(topk_item), _ptr(topk_score), _stream()), "eval_rank_topk")


def eval_rank_tc_ws_bytes(ms: AderModel, R: int, V: int) -> int:
    n = _lib.load().ader_eval_rank_tc_ws_bytes(C.byref(ms), R, V)
    if n == 0:
        raise _lib.AderError("eval_rank_tc_ws_bytes: bad model / sizes")
    return n


def eval_rank_tc(ms: AderModel, theta, rep, gt, V: int, ws, rank, overflow):
    """Fused tensor-core ranking (scores never materialised); overflow[0] != 0 -> use eval_rank_topk for this batch."""
    _require_cuda(theta, rep, gt, ws, rank, overflow)
    check(_lib.load().ader_eval_rank_tc(C.byref(ms), _ptr(theta), _ptr(rep), _ptr(gt), rep.shape[0], V, _ptr(ws), _ptr(rank),
                                        _ptr(overflow), _stream()), "eval_rank_tc")


def eval_topk_chunks(ms: AderModel, R: int, V: int) -> int:
    return int(_lib.load().ader_eval_topk_chunks(C.byref(ms), R, V))


def eval_rank_topk_tc(ms: AderModel, theta, rep, gt, V: int, k: int, ws, rank, topk_item, topk_score, overflow):
    """Fused tensor-core ranking + exact top-k (see include/ader_b200.h); needs 2 * eval_topk_chunks(R, V) >= k."""
    _require_cuda(theta, rep, gt, ws, rank, topk_item, topk_score, overflow)
    check(_lib.load().ader_eval_rank_topk_tc(C.byref(ms), _ptr(theta), _ptr(rep), _ptr(gt), rep.shape[0], V, k, _ptr(ws), _ptr(rank),
                                             _ptr(topk_item), _ptr(topk_score), _ptr(overflow), _stream()), "eval_rank_topk_tc")


def recommend_topk(ms: AderModel, theta, rep, ids, V: int, k: int, ws, topk_item, topk_score):
    """Top-k items 1..V of every row of rep (exact fp32 scores, ties -> lower id); ids [R, maxlen] (or None): the row's own
    items are left out.  ws: eval_ws_bytes(ms, R, V)."""
    _require_cuda(theta, rep, ids, ws, topk_item, topk_score)
    check(_lib.load().ader_recommend_topk(C.byref(ms), _ptr(theta), _ptr(rep), _ptr(ids), rep.shape[0], V, k, _ptr(ws),
                                          _ptr(topk_item), _ptr(topk_score), _stream()), "recommend_topk")


def recommend_tc_ws_bytes(ms: AderModel, R: int, V: int) -> int:
    n = _lib.load().ader_recommend_tc_ws_bytes(C.byref(ms), R, V)
    if n == 0:
        raise _lib.AderError("recommend_tc_ws_bytes: bad model / sizes")
    return n


def recommend_topk_tc(ms: AderModel, theta, rep, ids, V: int, k: int, ws, topk_item, topk_score, overflow):
    """The same lists on the tensor cores; needs 2 * 8 * eval_topk_chunks(R, V) >= k.  overflow[0] != 0 -> use
    recommend_topk for this batch."""
    _require_cuda(theta, rep, ids, ws, topk_item, topk_score, overflow)
    check(_lib.load().ader_recommend_topk_tc(C.byref(ms), _ptr(theta), _ptr(rep), _ptr(ids), rep.shape[0], V, k, _ptr(ws),
                                             _ptr(topk_item), _ptr(topk_score), _ptr(overflow), _stream()), "recommend_topk_tc")


def logsumexp(ms: AderModel, theta, rep, gt, V: int, ws, lse, nll):
    """lse [R] = log sum_{j=1..V} exp(rep . E_j) from the exact fp32 scores (fp64 sums); gt [R] (or None): nll [R] =
    lse - the ground-truth score (nll None when gt is).  ws: eval_ws_bytes(ms, R, V)."""
    _require_cuda(theta, rep, gt, ws, lse, nll)
    check(_lib.load().ader_logsumexp(C.byref(ms), _ptr(theta), _ptr(rep), _ptr(gt), rep.shape[0], V, _ptr(ws), _ptr(lse),
                                     _ptr(nll), _stream()), "logsumexp")


def logsumexp_tc_ws_bytes(ms: AderModel, R: int, V: int) -> int:
    n = _lib.load().ader_logsumexp_tc_ws_bytes(C.byref(ms), R, V)
    if n == 0:
        raise _lib.AderError("logsumexp_tc_ws_bytes: bad model / sizes")
    return n


def logsumexp_tc(ms: AderModel, theta, rep, gt, V: int, ws, lse, nll):
    """The same on the tensor cores ([R, V] never written): within eps_i = 2^-12 ||rep_i|| max_j ||E_j|| of the exact lse;
    nll uses the exact ground-truth score."""
    _require_cuda(theta, rep, gt, ws, lse, nll)
    check(_lib.load().ader_logsumexp_tc(C.byref(ms), _ptr(theta), _ptr(rep), _ptr(gt), rep.shape[0], V, _ptr(ws), _ptr(lse),
                                        _ptr(nll), _stream()), "logsumexp_tc")


def herding_ws_bytes(ms: AderModel, N: int) -> int:
    n = _lib.load().ader_herding_ws_bytes(C.byref(ms), N)
    if n == 0:
        raise _lib.AderError("herding_ws_bytes: bad model / sizes")
    return n


def herding_segmented(ms: AderModel, rep, cand, seg_off, quota, max_steps, ws, picks, n_picked):
    _require_cuda(rep, cand, seg_off, quota, max_steps, ws, picks, n_picked)
    check(_lib.load().ader_herding_segmented(C.byref(ms), _ptr(rep), rep.shape[0], _ptr(cand), _ptr(seg_off),
                                             seg_off.numel() - 1, _ptr(quota), _ptr(max_steps), _ptr(ws), _ptr(picks),
                                             _ptr(n_picked), _stream()), "herding_segmented")


def fisher_accumulate(ms: AderModel, grad, acc, V: int):
    _require_cuda(grad, acc)
    check(_lib.load().ader_fisher_accumulate(C.byref(ms), _ptr(grad), _ptr(acc), V, _stream()), "fisher_accumulate")


def fisher_finalize(ms: AderModel, acc, fisher, V: int, n_data: int):
    _require_cuda(acc, fisher)
    check(_lib.load().ader_fisher_finalize(C.byref(ms), _ptr(acc), _ptr(fisher), V, n_data, _stream()), "fisher_finalize")


def fisher_batched_ws_bytes(ms: AderModel, S: int, V: int) -> int:
    n = _lib.load().ader_fisher_batched_ws_bytes(C.byref(ms), S, V)
    if n == 0:
        raise _lib.AderError("fisher_batched_ws_bytes: bad model / sizes")
    return n


def fisher_batched(ms: AderModel, theta, ids, pos, Tcap: int, V: int, enc_ws, bwd_ws, ws, acc):
    """acc (fp64, flat) += sum over the rows of `ids` of the squared per-sample gradient (EWC.py:142-161), one batched pass."""
    _require_cuda(theta, ids, pos, enc_ws, bwd_ws, ws, acc)
    check(_lib.load().ader_fisher_batched(C.byref(ms), _ptr(theta), _ptr(ids), _ptr(pos), ids.shape[0], Tcap, V, _ptr(enc_ws),
                                          _ptr(bwd_ws), _ptr(ws), _ptr(acc), _stream()), "fisher_batched")


def gather_rows_i32(src, idx, out):
    _require_cuda(src, idx, out)
    check(_lib.load().ader_gather_rows_i32(_ptr(src), _ptr(idx), idx.numel(), src.shape[1], _ptr(out), _stream()),
          "gather_rows_i32")


def gather_batch(t_ids, t_lab, ti, e_ids, e_aux, ei, ids, pos, aux):
    """ids[:n_train] = t_ids[ti], pos = t_lab[ti], ids[n_train:] = e_ids[ei], aux = e_aux[ei] in one launch."""
    _require_cuda(t_ids, t_lab, ti, e_ids, e_aux, ei, ids, pos, aux)
    n_train = 0 if ti is None else ti.numel()
    n_ex = 0 if ei is None else ei.numel()
    check(_lib.load().ader_gather_batch(_ptr(t_ids), _ptr(t_lab), _ptr(ti), n_train, _ptr(e_ids), _ptr(e_aux), _ptr(ei), n_ex,
                                        ids.shape[1], _ptr(ids), _ptr(pos), _ptr(aux), _stream()), "gather_batch")


def gather_batch_q(t_ids, t_lab, n_train: int, e_ids, e_aux, n_ex: int, q, q_off, counter, ids, pos, aux):
    """Batch assembly of step `counter[0]` from the epoch-resident index queue (q int32, q_off int64)."""
    _require_cuda(t_ids, t_lab, e_ids, e_aux, q, q_off, counter, ids, pos, aux)
    check(_lib.load().ader_gather_batch_q(_ptr(t_ids), _ptr(t_lab), n_train, _ptr(e_ids), _ptr(e_aux), n_ex, _ptr(q), _ptr(q_off),
                                          _ptr(counter), ids.shape[1], _ptr(ids), _ptr(pos), _ptr(aux), _stream()), "gather_batch_q")


def queue_advance(counter):
    _require_cuda(counter)
    check(_lib.load().ader_queue_advance(_ptr(counter), _stream()), "queue_advance")


# ---- torch.ops registration -------------------------------------------------------------------
# Every compute entry point of include/ader_b200.h is also reachable through the dispatcher as torch.ops.ader_b200.<name>
# (CUDA key only: there is no CPU implementation to fall back to).  The POD structs of the C ABI are flattened:
#   model  = int[5]   (v_tab, d, maxlen, num_blocks, num_heads)
#   loss   = int[8]   (M, n_train, n_ex, V, V_prev, mode, n_train_global, n_ex_global) + float lambda_ + Tensor? pos, ex_pos,
#                     teacher, teacher_row (+ trailing Tensor? teacher_rep, teacher_table, teacher_table16 = None: frozen teacher)
#   dp comm = int rank, int world, int[] theta_ptrs, int[] grad_ptrs, int[] flag_ptrs  (peer-mapped device addresses)
# Workspace-size queries, IPC plumbing and status reads are host-only helpers and stay plain Python functions.
_registered = False

_SCHEMAS = {
    "encoder_fwd": "(int[] model, Tensor theta, Tensor ids, int Tcap, Tensor(a!) ws, Tensor(b!) rep, float dropout_rate, int seed) -> ()",
    "encoder_fwd_tc": "(int[] model, Tensor theta, Tensor ids, int Tcap, Tensor(a!) ws, Tensor(b!) rep, float dropout_rate, int seed, Tensor? d_step) -> ()",
    "encoder_bwd": "(int[] model, Tensor theta, Tensor ids, int Tcap, Tensor ws, Tensor(a!) bwd_ws, Tensor d_rep, Tensor(b!) grad, float dropout_rate, int seed) -> ()",
    "encoder_bwd_tc": "(int[] model, Tensor theta, Tensor ids, int Tcap, Tensor ws, Tensor(a!) bwd_ws, Tensor d_rep, Tensor(b!) grad, float dropout_rate, int seed, Tensor? d_step) -> ()",
    "loss_fwd_bwd": "(int[] model, Tensor theta, Tensor rep, int[] loss_dims, float lambda_, Tensor? pos, Tensor? ex_pos, Tensor? teacher, Tensor? teacher_row, Tensor(a!) ws, Tensor(b!) loss, Tensor(c!) row_loss, Tensor(d!) d_rep, Tensor(e!) grad, Tensor? teacher_rep=None, Tensor? teacher_table=None, Tensor? teacher_table16=None) -> ()",
    "loss_fwd_bwd_tc": "(int[] model, Tensor theta, Tensor rep, int[] loss_dims, float lambda_, Tensor? pos, Tensor? ex_pos, Tensor? teacher, Tensor? teacher_row, Tensor(a!) ws, Tensor(b!) loss, Tensor(c!) row_loss, Tensor(d!) d_rep, Tensor(e!) grad, Tensor? teacher_rep=None, Tensor? teacher_table=None, Tensor? teacher_table16=None) -> ()",
    "loss_tc_vp_fwd": "(int[] model, Tensor theta, Tensor rep, int[] loss_dims, float lambda_, Tensor? pos, Tensor? ex_pos, Tensor? teacher, Tensor? teacher_row, int v_lo, int v_hi, Tensor(a!) ws, Tensor(b!) stats) -> ()",
    "loss_tc_vp_bwd": "(int[] model, Tensor theta, Tensor rep, int[] loss_dims, float lambda_, Tensor? pos, Tensor? ex_pos, Tensor? teacher, Tensor? teacher_row, int v_lo, int v_hi, Tensor(a!) ws, Tensor lse, Tensor(b!) d_rep_partial, Tensor(c!) grad) -> ()",
    "train_fwd_bwd_tc": "(int[] model, Tensor theta, Tensor ids, int Tcap, int[] loss_dims, float lambda_, Tensor? pos, Tensor? ex_pos, Tensor? teacher, Tensor? teacher_row, Tensor(a!) enc_ws, Tensor(b!) bwd_ws, Tensor(c!) loss_ws, Tensor(d!) rep, Tensor(e!) loss, Tensor(f!) row_loss, Tensor(g!) d_rep, Tensor(h!) grad, float dropout_rate, int seed, Tensor? d_step, bool serial, Tensor? teacher_rep=None, Tensor? teacher_table=None, Tensor? teacher_table16=None) -> ()",
    "train_step_tc": "(int[] model, Tensor(a!) theta, Tensor ids, int Tcap, int[] loss_dims, float lambda_, Tensor? pos, Tensor? ex_pos, Tensor? teacher, Tensor? teacher_row, Tensor(b!) enc_ws, Tensor(c!) bwd_ws, Tensor(d!) loss_ws, Tensor(e!) rep, Tensor(f!) loss, Tensor(g!) row_loss, Tensor(h!) d_rep, Tensor(i!) grad, Tensor(j!) adam_m, Tensor(k!) adam_v, Tensor(l!) state, int V, float lr, float dropout_rate, int seed, Tensor? d_step, float ewc_lambda, Tensor? fisher, Tensor? theta_star, bool serial, Tensor? teacher_rep=None, Tensor? teacher_table=None, Tensor? teacher_table16=None) -> ()",
    "pack_table16": "(int[] model, Tensor rows, int V, Tensor(a!) out) -> ()",
    "logits": "(int[] model, Tensor theta, Tensor rep, int V, Tensor(a!) out) -> ()",
    "adam_step": "(int[] model, Tensor(a!) theta, Tensor(b!) m, Tensor(c!) v, Tensor grad, Tensor(d!) state, int V, float lr, float ewc_lambda, Tensor? fisher, Tensor? theta_star) -> ()",
    "dp_wait": "(int rank, int world, int[] theta_ptrs, int[] grad_ptrs, int[] flag_ptrs, Tensor(a!) flags) -> ()",
    "dp_adam_step": "(int[] model, int rank, int world, int[] theta_ptrs, int[] grad_ptrs, int[] flag_ptrs, Tensor(a!) theta, Tensor(b!) m, Tensor(c!) v, Tensor(d!) state, int V, float lr, float ewc_lambda, Tensor? fisher, Tensor? theta_star) -> ()",
    "eval_rank_topk": "(int[] model, Tensor theta, Tensor rep, Tensor gt, int V, int k, Tensor(a!) ws, Tensor(b!) rank, Tensor(c!) topk_item, Tensor(d!) topk_score) -> ()",
    "eval_rank_tc": "(int[] model, Tensor theta, Tensor rep, Tensor gt, int V, Tensor(a!) ws, Tensor(b!) rank, Tensor(c!) overflow) -> ()",
    "eval_rank_topk_tc": "(int[] model, Tensor theta, Tensor rep, Tensor gt, int V, int k, Tensor(a!) ws, Tensor(b!) rank, Tensor(c!) topk_item, Tensor(d!) topk_score, Tensor(e!) overflow) -> ()",
    "recommend_topk": "(int[] model, Tensor theta, Tensor rep, Tensor? ids, int V, int k, Tensor(a!) ws, Tensor(b!) topk_item, Tensor(c!) topk_score) -> ()",
    "recommend_topk_tc": "(int[] model, Tensor theta, Tensor rep, Tensor? ids, int V, int k, Tensor(a!) ws, Tensor(b!) topk_item, Tensor(c!) topk_score, Tensor(d!) overflow) -> ()",
    "logsumexp": "(int[] model, Tensor theta, Tensor rep, Tensor? gt, int V, Tensor(a!) ws, Tensor(b!) lse, Tensor(c!)? nll) -> ()",
    "logsumexp_tc": "(int[] model, Tensor theta, Tensor rep, Tensor? gt, int V, Tensor(a!) ws, Tensor(b!) lse, Tensor(c!)? nll) -> ()",
    "herding_segmented": "(int[] model, Tensor rep, Tensor cand, Tensor seg_off, Tensor quota, Tensor max_steps, Tensor(a!) ws, Tensor(b!) picks, Tensor(c!) n_picked) -> ()",
    "fisher_accumulate": "(int[] model, Tensor grad, Tensor(a!) acc, int V) -> ()",
    "fisher_finalize": "(int[] model, Tensor acc, Tensor(a!) fisher, int V, int n_data) -> ()",
    "fisher_batched": "(int[] model, Tensor theta, Tensor ids, Tensor pos, int Tcap, int V, Tensor(a!) enc_ws, Tensor(b!) bwd_ws, Tensor(c!) ws, Tensor(d!) acc) -> ()",
    "gather_rows_i32": "(Tensor src, Tensor idx, Tensor(a!) out) -> ()",
    "gather_batch": "(Tensor t_ids, Tensor t_lab, Tensor ti, Tensor? e_ids, Tensor? e_aux, Tensor? ei, Tensor(a!) ids, Tensor(b!) pos, Tensor(c!)? aux) -> ()",
    "gather_batch_q": "(Tensor t_ids, Tensor t_lab, int n_train, Tensor? e_ids, Tensor? e_aux, int n_ex, Tensor q, Tensor q_off, Tensor counter, Tensor(a!) ids, Tensor(b!) pos, Tensor(c!)? aux) -> ()",
    "queue_advance": "(Tensor(a!) counter) -> ()",
}


def register_torch_ops() -> None:
    """Expose every compute entry point as ``torch.ops.ader_b200.*`` (CUDA implementations only)."""
    global _registered
    if _registered:
        return
    lib = torch.library.Library("ader_b200", "DEF")

    def _ms(model):
        return AderModel(*[int(x) for x in model])

    def _la(dims, lam, pos, ex_pos, teacher, teacher_row, fz=(None, None, None)):
        M, n_train, n_ex, V, V_prev, mode, ntg, neg = [int(x) for x in dims]
        return make_loss_args(M, n_train, n_ex, V, V_prev, mode, lam, pos, ex_pos, teacher, teacher_row, ntg, neg, *fz)

    def _comm(rank, world, tp, gp, fp):
        return dp_comm(int(rank), int(world), list(tp), list(gp), list(fp))

    impls = {
        "encoder_fwd": lambda model, theta, ids, Tcap, ws, rep, p, seed: encoder_fwd(_ms(model), theta, ids, Tcap, ws, rep, p, seed),
        "encoder_fwd_tc": lambda model, theta, ids, Tcap, ws, rep, p, seed, d_step: encoder_fwd(_ms(model), theta, ids, Tcap, ws, rep, p, seed, impl="tc", d_step=d_step),
        "encoder_bwd": lambda model, theta, ids, Tcap, ws, bws, d_rep, grad, p, seed: encoder_bwd(_ms(model), theta, ids, Tcap, ws, bws, d_rep, grad, p, seed),
        "encoder_bwd_tc": lambda model, theta, ids, Tcap, ws, bws, d_rep, grad, p, seed, d_step: encoder_bwd(_ms(model), theta, ids, Tcap, ws, bws, d_rep, grad, p, seed, impl="tc", d_step=d_step),
        "loss_fwd_bwd": lambda model, theta, rep, dims, lam, pos, ex_pos, teacher, trow, ws, loss, row_loss, d_rep, grad, *fz:
            loss_fwd_bwd(_ms(model), theta, rep, _la(dims, lam, pos, ex_pos, teacher, trow, fz), ws, loss, row_loss, d_rep, grad),
        "loss_fwd_bwd_tc": lambda model, theta, rep, dims, lam, pos, ex_pos, teacher, trow, ws, loss, row_loss, d_rep, grad, *fz:
            loss_fwd_bwd_tc(_ms(model), theta, rep, _la(dims, lam, pos, ex_pos, teacher, trow, fz), ws, loss, row_loss, d_rep, grad),
        "loss_tc_vp_fwd": lambda model, theta, rep, dims, lam, pos, ex_pos, teacher, trow, v_lo, v_hi, ws, stats:
            loss_tc_vp_fwd(_ms(model), theta, rep, _la(dims, lam, pos, ex_pos, teacher, trow), v_lo, v_hi, ws, stats),
        "loss_tc_vp_bwd": lambda model, theta, rep, dims, lam, pos, ex_pos, teacher, trow, v_lo, v_hi, ws, lse, d_part, grad:
            loss_tc_vp_bwd(_ms(model), theta, rep, _la(dims, lam, pos, ex_pos, teacher, trow), v_lo, v_hi, ws, lse, d_part, grad),
        "train_fwd_bwd_tc": lambda model, theta, ids, Tcap, dims, lam, pos, ex_pos, teacher, trow, ews, bws, lws, rep, loss, row_loss, d_rep, grad, p, seed, d_step, serial, *fz:
            train_fwd_bwd_tc(_ms(model), theta, ids, Tcap, _la(dims, lam, pos, ex_pos, teacher, trow, fz), ews, bws, lws, rep, loss, row_loss, d_rep, grad, p, seed, d_step, serial),
        "train_step_tc": lambda model, theta, ids, Tcap, dims, lam, pos, ex_pos, teacher, trow, ews, bws, lws, rep, loss, row_loss, d_rep, grad, am, av, state, V, lr, p, seed, d_step, ewc_lambda, fisher, theta_star, serial, *fz:
            train_step_tc(_ms(model), theta, ids, Tcap, _la(dims, lam, pos, ex_pos, teacher, trow, fz), ews, bws, lws, rep, loss, row_loss, d_rep, grad, am, av, state, V, lr, p, seed, d_step, ewc_lambda, fisher, theta_star, serial=serial),
        "pack_table16": lambda model, rows, V, out: pack_table16(_ms(model), rows, V, out),
        "logits": lambda model, theta, rep, V, out: logits(_ms(model), theta, rep, V, out),
        "adam_step": lambda model, theta, m, v, grad, state, V, lr, ewc_lambda, fisher, theta_star: adam_step(_ms(model), theta, m, v, grad, state, V, lr, ewc_lambda, fisher, theta_star),
        "dp_wait": lambda rank, world, tp, gp, fp, flags: dp_wait(_comm(rank, world, tp, gp, fp)),
        "dp_adam_step": lambda model, rank, world, tp, gp, fp, theta, m, v, state, V, lr, ewc_lambda, fisher, theta_star:
            dp_adam_step(_ms(model), _comm(rank, world, tp, gp, fp), m, v, state, V, lr, ewc_lambda, fisher, theta_star),
        "eval_rank_topk": lambda model, theta, rep, gt, V, k, ws, rank, items, scores: eval_rank_topk(_ms(model), theta, rep, gt, V, k, ws, rank, items, scores),
        "eval_rank_tc": lambda model, theta, rep, gt, V, ws, rank, overflow: eval_rank_tc(_ms(model), theta, rep, gt, V, ws, rank, overflow),
        "eval_rank_topk_tc": lambda model, theta, rep, gt, V, k, ws, rank, items, scores, overflow: eval_rank_topk_tc(_ms(model), theta, rep, gt, V, k, ws, rank, items, scores, overflow),
        "recommend_topk": lambda model, theta, rep, ids, V, k, ws, items, scores: recommend_topk(_ms(model), theta, rep, ids, V, k, ws, items, scores),
        "recommend_topk_tc": lambda model, theta, rep, ids, V, k, ws, items, scores, overflow: recommend_topk_tc(_ms(model), theta, rep, ids, V, k, ws, items, scores, overflow),
        "logsumexp": lambda model, theta, rep, gt, V, ws, lse, nll: logsumexp(_ms(model), theta, rep, gt, V, ws, lse, nll),
        "logsumexp_tc": lambda model, theta, rep, gt, V, ws, lse, nll: logsumexp_tc(_ms(model), theta, rep, gt, V, ws, lse, nll),
        "herding_segmented": lambda model, rep, cand, seg_off, quota, max_steps, ws, picks, n_picked: herding_segmented(_ms(model), rep, cand, seg_off, quota, max_steps, ws, picks, n_picked),
        "fisher_accumulate": lambda model, grad, acc, V: fisher_accumulate(_ms(model), grad, acc, V),
        "fisher_finalize": lambda model, acc, fisher, V, n_data: fisher_finalize(_ms(model), acc, fisher, V, n_data),
        "fisher_batched": lambda model, theta, ids, pos, Tcap, V, ews, bws, ws, acc: fisher_batched(_ms(model), theta, ids, pos, Tcap, V, ews, bws, ws, acc),
        "gather_rows_i32": lambda src, idx, out: gather_rows_i32(src, idx, out),
        "gather_batch": lambda t_ids, t_lab, ti, e_ids, e_aux, ei, ids, pos, aux: gather_batch(t_ids, t_lab, ti, e_ids, e_aux, ei, ids, pos, aux),
        "gather_batch_q": lambda t_ids, t_lab, n_train, e_ids, e_aux, n_ex, q, q_off, counter, ids, pos, aux: gather_batch_q(t_ids, t_lab, n_train, e_ids, e_aux, n_ex, q, q_off, counter, ids, pos, aux),
        "queue_advance": lambda counter: queue_advance(counter),
    }
    assert set(impls) == set(_SCHEMAS)
    for name, schema in _SCHEMAS.items():
        lib.define(name + schema)
        lib.impl(name, impls[name], "CUDA")
    register_torch_ops._lib = lib      # keep alive
    _registered = True


def registered_op_names():
    return sorted(_SCHEMAS)
