"""`Ader` / `Ewc` model objects: the reference's TF1 feed/fetch surface re-hosted on the C ABI.

Reference seam (SURVEY 8b): ``Ader(item_num, args)`` (ADER.py:13-103), ``set_vanilla_loss``
(ADER.py:105), ``update_loss(lambda_)`` (ADER.py:108), ``predict(sess, seq, item_idx)``
(ADER.py:140), fetches ``rep`` / ``logits`` / ``loss`` / ``train_op``; ``Ewc`` adds
``compute_fisher`` and ``variables_prev`` (EWC.py:115-164).  ``sess`` arguments are accepted and
ignored.  Exemplar rows are the LAST rows of ``input_seq`` and ``pos`` covers the train rows only
(main.py:229, ADER.py:113-124).

All state is device resident: one flat fp32 parameter vector + Adam slots + gradient buffer
(params.py), so a "checkpoint" (tf.train.Saver, main.py:209-213,280,283) is a clone of four tensors.
"""
from __future__ import annotations

import os
from typing import Optional, Sequence

import numpy as np
import torch

from . import ops
from .params import Hyper, ParamLayout


def _to_ids(seq, maxlen: int, device) -> torch.Tensor:
    """Accept the reference's tuple-of-arrays batches, ndarrays or device tensors -> int32 [M, L] on device."""
    if isinstance(seq, torch.Tensor):
        t = seq.to(device=device, dtype=torch.int32, non_blocking=True)
    else:
        a = np.ascontiguousarray(np.asarray(seq, dtype=np.int32))
        t = torch.from_numpy(a).pin_memory().to(device, non_blocking=True) if a.size else torch.zeros((0, maxlen), dtype=torch.int32, device=device)
    if t.dim() == 1:
        t = t.view(1, -1)
    if t.shape[1] != maxlen:
        raise ValueError("input_seq must have maxlen=%d columns, got %s" % (maxlen, tuple(t.shape)))
    return t.contiguous()


def _to_i32(x, device) -> torch.Tensor:
    if isinstance(x, torch.Tensor):
        return x.to(device=device, dtype=torch.int32, non_blocking=True).contiguous().view(-1)
    a = np.ascontiguousarray(np.asarray(x, dtype=np.int32)).reshape(-1)
    return torch.from_numpy(a).pin_memory().to(device, non_blocking=True)


class Ader:
    """SASRec + CE / distillation model (ADER.py:13-150) on libader_b200."""

    VANILLA, KD, ER = 0, 1, 2

    def __init__(self, item_num: int, args, device: Optional[torch.device] = None, init_seed: Optional[int] = None):
        if not torch.cuda.is_available():
            raise RuntimeError("ader_b200 needs a CUDA device (B200 / sm_100a); there is no CPU path")
        ops._lib.load()
        self.args = args
        self.hp = Hyper(item_num=item_num, hidden_units=args.hidden_units, maxlen=args.maxlen,
                        num_blocks=args.num_blocks, num_heads=args.num_heads)
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self.layout = ParamLayout(self.hp)
        self.ms = ops.model_struct(self.hp)
        seed = getattr(args, "random_seed", 0) if init_seed is None else init_seed
        self.seed = int(getattr(args, "random_seed", 0))
        self.theta = torch.from_numpy(self.layout.init_flat(seed)).to(self.device)
        self.adam_m = torch.zeros_like(self.theta)
        self.adam_v = torch.zeros_like(self.theta)
        self.grad = torch.zeros_like(self.theta)
        self.adam_state = torch.zeros(2, dtype=torch.int32, device=self.device)
        self.disable_distillation = bool(getattr(args, "disable_distillation", False))
        self.mode = self.VANILLA
        self.lambda_ = 0.0
        self.grad_sync = None           # optional callable run between backward and the optimiser (legacy hook)
        self.dp = None                  # data parallel back end (ader_b200.dist.PeerComm / NcclComm): sums gradients over ranks
        self.global_counts = None       # data parallel: (n_train, n_ex) over all ranks -> global means
        self.loss_impl = getattr(args, "loss_impl", "tc")   # "tc": tcgen05 fused logits+CE+KD; "exact": fp32
        # encoder: "tc" = fused bf16 tensor-core kernels, "exact" = fp32.  Training uses encoder_impl; inference
        # passes (rep / eval / herding: bit-exact index parity with the fp32 reference) use infer_encoder_impl.
        self.encoder_impl = getattr(args, "encoder_impl", None) or ("exact" if self.loss_impl == "exact" else "tc")
        self.infer_encoder_impl = getattr(args, "infer_encoder_impl", "exact")
        # evaluation ranks: "tc" = fused tcgen05 scoring + exact refinement (identical ranks), "exact" = fp32 [M, V] scores
        self.eval_impl = getattr(args, "eval_impl", None) or os.environ.get("ADER_B200_EVAL", "tc")
        self.eval_fallbacks = 0
        # how a tc + tc training pass is issued: "dag" = ader_train_fwd_bwd_tc (fork/join over side streams),
        # "serial" = the same entry on one stream, "groups" = the three single-group entry points one after another
        self.step_impl = getattr(args, "step_impl", None) or os.environ.get("ADER_B200_STEP_IMPL", "dag")
        if self.hp.hidden_units > 160:
            self.encoder_impl = self.infer_encoder_impl = "exact"
        self.global_step = 0            # host mirror of adam_state[0] (drives the dropout stream)
        self._enc_ws = ops.Workspace(self.device)
        self._bwd_ws = ops.Workspace(self.device)
        self._loss_ws = ops.Workspace(self.device)
        self._eval_ws = ops.Workspace(self.device)
        self._loss = torch.zeros(1, dtype=torch.float32, device=self.device)
        self.last_row_loss: Optional[torch.Tensor] = None
        self._tight_cap = False
        self._last_enc = None           # (M, Tcap) of the last encoder pass (locates the overflow flag in the workspace)

    # ---- reference surface ----------------------------------------------------------------
    @property
    def variables(self):
        """The 32 trainable tensors in creation order (EWC.py:90) as views of ``theta``."""
        return self.layout.views(self.theta)

    def set_vanilla_loss(self):                       # ADER.py:105-106
        self.mode = self.VANILLA
        self.lambda_ = 0.0

    def update_loss(self, lambda_: float):            # ADER.py:108-138
        self.mode = self.ER if self.disable_distillation else self.KD
        self.lambda_ = float(lambda_)

    # ---- encoder ----------------------------------------------------------------------------
    def _tcap(self, ids: torch.Tensor, n_tokens: Optional[int]) -> int:
        M = ids.shape[0]
        cap = M * self.hp.maxlen if n_tokens is None else max(int(n_tokens), 1)
        self._tight_cap = n_tokens is not None and cap < M * self.hp.maxlen
        return min(max(cap, 1), M * self.hp.maxlen)

    def token_overflow(self) -> bool:
        """True if an encoder pass since the last call was given a token capacity below the real token count (the kernels
        clamp and set flags[0] in the activation workspace: tokens were dropped, reps / gradients are wrong).  One small
        synchronous read; the period loop calls it once per epoch, eval / selection passes after every call."""
        buf = self._enc_ws.buf
        if buf is None or getattr(self, "_last_enc", None) is None:
            return False
        M, tcap = self._last_enc
        off = ops.encoder_ws_slot(self.ms, M, tcap, -4, 0)
        flag = buf[off:off + 4].view(torch.int32)
        hit = bool(int(flag.item()) != 0)
        return hit

    def _check_overflow(self):
        if self._tight_cap and self.token_overflow():
            raise ops._lib.AderError("encoder: n_tokens was smaller than the number of real tokens in the batch (tokens dropped)")

    def encode(self, ids: torch.Tensor, n_tokens: Optional[int] = None, dropout_rate: float = 0.0,
               seed: int = 0, out: Optional[torch.Tensor] = None, impl: Optional[str] = None, d_step=None):
        """ids int32 [M, L] (device) -> rep fp32 [M, d]; returns (rep, Tcap).  The activation
        workspace stays valid until the next encode() (needed by backward)."""
        M = ids.shape[0]
        tcap = self._tcap(ids, n_tokens)
        ws = self._enc_ws.get(ops.encoder_ws_bytes(self.ms, M, tcap))
        rep = out if out is not None else torch.empty((M, self.hp.hidden_units), dtype=torch.float32, device=self.device)
        ops.encoder_fwd(self.ms, self.theta, ids, tcap, ws, rep, dropout_rate, seed,
                        impl=impl or self.infer_encoder_impl, d_step=d_step)
        self._last_enc = (M, tcap)
        return rep, tcap

    def rep(self, seq, n_tokens: Optional[int] = None) -> torch.Tensor:
        """fetch ``model.rep`` in eval mode (util.py:452)."""
        ids = _to_ids(seq, self.hp.maxlen, self.device)
        r = self.encode(ids, n_tokens)[0]
        self._check_overflow()           # inference passes are few and large: verify the caller's token capacity every time
        return r

    def logits(self, rep: torch.Tensor, max_item: int) -> torch.Tensor:
        """fetch ``model.logits`` (ADER.py:91): [M, max_item] fp32."""
        ld = (max_item + 3) // 4 * 4      # 16-byte aligned rows (stored exemplar logits are read with 128-bit loads)
        out = torch.empty((rep.shape[0], ld), dtype=torch.float32, device=self.device)[:, :max_item]
        ops.logits(self.ms, self.theta, rep, max_item, out)
        return out

    def rep_logits(self, seq, max_item: int):
        """fetch [model.rep, model.logits] (util.py:452-455)."""
        r = self.rep(seq)
        return r, self.logits(r, max_item)

    # ---- training step ------------------------------------------------------------------------
    def loss_and_grad(self, seq, pos, max_item: int, exemplar_logits=None, exemplar_pos=None,
                      teacher_rows=None, dropout_rate: float = 0.0, n_tokens: Optional[int] = None,
                      mode: Optional[int] = None, lambda_: Optional[float] = None, _events=None,
                      global_counts=None, _device_step: bool = False, _opt=None) -> torch.Tensor:
        """Forward + backward of the current loss; fills ``self.grad`` (flat).  Returns the device
        scalar loss.  ``exemplar_logits`` is either a host array / list [M_e, V_prev] (reference feed,
        ADER.py:20), a device tensor [E, V_prev] indexed by ``teacher_rows`` [M_e], or a ``data.FrozenTeacher``
        whose reps ``teacher_rows`` indexes the same way."""
        from .data import FrozenTeacher
        mode = self.mode if mode is None else mode
        lam = self.lambda_ if lambda_ is None else lambda_
        ids = _to_ids(seq, self.hp.maxlen, self.device)
        pos_t = _to_i32(pos, self.device)
        M, n_train = ids.shape[0], pos_t.numel()
        n_ex = M - n_train
        teacher = trow = ex_pos_t = None
        frozen = None
        v_prev = 0
        if n_ex > 0:
            if mode == self.KD:
                if exemplar_logits is None:
                    raise ValueError("KD loss needs exemplar_logits")
                if isinstance(exemplar_logits, FrozenTeacher):
                    frozen = exemplar_logits
                    n_rows = len(frozen)
                    v_prev = frozen.width
                    if self.loss_impl == "tc" and frozen.table16 is None:
                        raise ValueError("the tcgen05 loss needs the snapshot's bf16 table (hidden_units <= 160)")
                elif isinstance(exemplar_logits, torch.Tensor):
                    teacher = exemplar_logits
                else:
                    a = np.asarray(exemplar_logits, dtype=np.float32)
                    ld = (a.shape[1] + 3) // 4 * 4
                    buf = np.zeros((a.shape[0], ld), np.float32)
                    buf[:, :a.shape[1]] = a
                    teacher = torch.from_numpy(buf).pin_memory().to(self.device, non_blocking=True)[:, :a.shape[1]]
                if teacher is not None:
                    if teacher.dim() != 2 or teacher.stride(1) != 1 or teacher.dtype != torch.float32:
                        raise ValueError("exemplar_logits must be a 2-D fp32 row-major matrix")
                    v_prev = teacher.shape[1]
                    n_rows = teacher.shape[0]
                if teacher_rows is not None:
                    trow = _to_i32(teacher_rows, self.device)
                    if trow.numel() != n_ex:
                        raise ValueError("teacher_rows must have one entry per exemplar row")
                elif n_rows != n_ex:
                    raise ValueError("exemplar_logits rows (%d) != exemplar rows (%d)" % (n_rows, n_ex))
            elif mode == self.ER:
                if exemplar_pos is None:
                    raise ValueError("one-hot exemplar loss needs exemplar_pos")
                ex_pos_t = _to_i32(exemplar_pos, self.device)
            else:
                raise ValueError("exemplar rows were fed but the loss is vanilla (call update_loss first)")
        # dropout stream: (seed, step).  Under CUDA-graph capture the step is read on the device from the Adam
        # state (incremented by the optimiser kernel), so every replay draws fresh masks.
        d_step = self.adam_state if (_device_step and self.encoder_impl == "tc") else None   # exact encoder: graphs only at p = 0
        seed = (self.seed << 32) + (0 if _device_step else self.global_step)
        gc = global_counts if global_counts is not None else self.global_counts
        a = ops.make_loss_args(M, n_train, n_ex, max_item, v_prev, mode if n_ex > 0 else self.VANILLA, lam,
                               pos_t, ex_pos_t, teacher, trow, *(gc or (0, 0)),
                               *((frozen.rep, frozen.table, frozen.table16) if frozen is not None else ()))
        row_loss = torch.empty(M, dtype=torch.float32, device=self.device)
        if self.step_impl != "groups" and self.encoder_impl == "tc" and self.loss_impl == "tc" and not _events:
            # one C call: the three groups as a fork/join DAG over library-owned side streams (same kernels, same bits)
            tcap = self._tcap(ids, n_tokens)
            self._last_enc = (M, tcap)
            ews = self._enc_ws.get(ops.encoder_ws_bytes(self.ms, M, tcap))
            bws = self._bwd_ws.get(ops.encoder_bwd_ws_bytes(self.ms, M, tcap))
            lws = self._loss_ws.get(ops.loss_tc_ws_bytes(self.ms, a))
            rep = torch.empty((M, self.hp.hidden_units), dtype=torch.float32, device=self.device)
            d_rep = torch.empty_like(rep)
            self._opt_applied = False
            if _opt is not None and self.grad_sync is None and self.dp is None:
                # one GPU: the optimiser joins the DAG (table rows right behind the scatter, dense parameters behind
                # their partial reduction)
                V_, lr_, lam_, fis_, star_ = _opt
                ops.train_step_tc(self.ms, self.theta, ids, tcap, a, ews, bws, lws, rep, self._loss, row_loss, d_rep,
                                  self.grad, self.adam_m, self.adam_v, self.adam_state, V_, lr_, dropout_rate, seed, d_step,
                                  lam_, fis_, star_, serial=(self.step_impl == "serial"))
                self._opt_applied = True
            else:
                ops.train_fwd_bwd_tc(self.ms, self.theta, ids, tcap, a, ews, bws, lws, rep, self._loss, row_loss, d_rep,
                                     self.grad, dropout_rate, seed, d_step, serial=(self.step_impl == "serial"))
            if self.grad_sync is not None:
                self.grad_sync()
            self.last_row_loss = row_loss
            self._keep = (ids, pos_t, teacher, trow, ex_pos_t, rep, d_rep, frozen)
            return self._loss
        rep, tcap = self.encode(ids, n_tokens, dropout_rate, seed, impl=self.encoder_impl, d_step=d_step)
        if _events:
            _events[0].record()
        d_rep = torch.empty_like(rep)
        if self.loss_impl == "tc":       # tcgen05 fused kernels (bf16 operands)
            ws = self._loss_ws.get(ops.loss_tc_ws_bytes(self.ms, a))
            ops.loss_fwd_bwd_tc(self.ms, self.theta, rep, a, ws, self._loss, row_loss, d_rep, self.grad)
        else:                            # exact fp32 path
            ws = self._loss_ws.get(ops.loss_ws_bytes(self.ms, a))
            ops.loss_fwd_bwd(self.ms, self.theta, rep, a, ws, self._loss, row_loss, d_rep, self.grad)
        if _events:
            _events[1].record()
        bws = self._bwd_ws.get(ops.encoder_bwd_ws_bytes(self.ms, M, tcap))
        ops.encoder_bwd(self.ms, self.theta, ids, tcap, self._enc_ws.buf, bws, d_rep, self.grad, dropout_rate, seed,
                        impl=self.encoder_impl, d_step=d_step)
        if _events:
            _events[2].record()
        if self.grad_sync is not None:      # data parallel: NCCL all-reduce of the flat gradient
            self.grad_sync()
        self.last_row_loss = row_loss
        self._keep = (ids, pos_t, teacher, trow, ex_pos_t, rep, d_rep, frozen)   # keep alive until the stream is done
        return self._loss

    def apply_gradients(self, max_item: int, lr: float, ewc_lambda: float = 0.0, fisher=None, theta_star=None):
        """tf.train.AdamOptimizer.apply_gradients (ADER.py:96,106,138)."""
        ops.adam_step(self.ms, self.theta, self.adam_m, self.adam_v, self.grad, self.adam_state, max_item, lr,
                      ewc_lambda, fisher, theta_star)
        self.global_step += 1

    def train_step(self, seq, pos, max_item: int, lr: Optional[float] = None, dropout_rate: Optional[float] = None,
                   exemplar_logits=None, exemplar_pos=None, teacher_rows=None, n_tokens: Optional[int] = None,
                   _device_step: bool = False):
        """sess.run(model.train_op, feed) (main.py:233-256).  Returns the device scalar loss."""
        lr = self.args.lr if lr is None else lr
        p = self.args.dropout_rate if dropout_rate is None else dropout_rate
        self._opt_applied = False
        if self.dp is not None:          # peer back end: every rank has finished the previous update (first launch of the step)
            self.dp.begin_step(self)
        loss = self.loss_and_grad(seq, pos, max_item, exemplar_logits, exemplar_pos, teacher_rows, p, n_tokens,
                                  _device_step=_device_step, _opt=self._opt_args(max_item, lr))
        if self._opt_applied:
            self.global_step += 1
        elif self.dp is not None:        # gradients summed over the ranks + TF1 Adam (one kernel over peer memory, or NCCL + Adam)
            self.dp.apply(self, *self._opt_args(max_item, lr))
            self.global_step += 1
        else:
            self.apply_gradients(max_item, lr)
        return loss

    def _opt_args(self, max_item: int, lr: float):
        """(V, lr, ewc_lambda, fisher, theta_star) of the update ``apply_gradients`` would run."""
        return (max_item, lr, 0.0, None, None)

    def graph_step(self, n_train: int, n_ex: int, max_item: int, lr: Optional[float] = None,
                   dropout_rate: Optional[float] = None, teacher=None, sources=None, tcaps=None, queue=None):
        """The same train step captured as CUDA graphs for a fixed batch geometry (see ader_b200/graph.py)."""
        from .graph import GraphStep
        return GraphStep(self, n_train, n_ex, max_item, self.args.lr if lr is None else lr,
                         self.args.dropout_rate if dropout_rate is None else dropout_rate, teacher, sources, tcaps, queue)

    # ---- evaluation ---------------------------------------------------------------------------
    def rank_topk(self, seq, gt, max_item: int, k: int = 20, n_tokens: Optional[int] = None, guards: Optional[list] = None,
                  force_exact: bool = False):
        """Rank of the ground-truth item among items 1..max_item (== pred_last[row, gt-1],
        ADER.py:103 + util.py:325; ties -> lower index first) and the top-k item ids.
        guards: None = the two guard words of the call (encoder token overflow, candidate-band overflow of the fused path)
        are read here (two small host syncs); a list = they are appended as device tensors ``(tokens, band)`` and the CALLER
        reads them later (``check_guards``) - an evaluation pass then launches all its chunks without a host sync."""
        ids = _to_ids(seq, self.hp.maxlen, self.device)
        gt_t = _to_i32(gt, self.device)
        rep, tcap_used = self.encode(ids, n_tokens)
        M = ids.shape[0]
        tok_flag = None
        if guards is None:
            self._check_overflow()
        else:
            off = ops.encoder_ws_slot(self.ms, M, tcap_used, -4, 0)
            tok_flag = self._enc_ws.buf[off:off + 4].view(torch.int32).clone()
        rank = torch.empty(M, dtype=torch.int32, device=self.device)
        if not force_exact and self.eval_impl == "tc" and self.hp.hidden_units <= 160 and (k <= 0 or 2 * ops.eval_topk_chunks(self.ms, M, max_item) >= k):
            # tcgen05 scores + exact refinement of the columns inside the certainty bands (ader_eval_rank_tc /
            # ader_eval_rank_topk_tc: identical ranks and top-k lists, the [M, V] scores are never written)
            ws = self._eval_ws.get(ops.eval_rank_tc_ws_bytes(self.ms, M, max_item))
            over = torch.zeros(1, dtype=torch.int32, device=self.device)
            if k <= 0:
                ops.eval_rank_tc(self.ms, self.theta, rep, gt_t, max_item, ws, rank, over)
                items = torch.empty((M, 1), dtype=torch.int32, device=self.device)
                scores = items.float()
            else:
                items = torch.empty((M, k), dtype=torch.int32, device=self.device)
                scores = torch.empty((M, k), dtype=torch.float32, device=self.device)
                ops.eval_rank_topk_tc(self.ms, self.theta, rep, gt_t, max_item, k, ws, rank, items, scores, over)
            if guards is not None:
                guards.append((tok_flag, over))
                return rank, items, scores
            if int(over.item()) == 0:
                return rank, items, scores
            self.eval_fallbacks += 1          # a band held more than ADER_EVAL_CAND_CAP columns: exact path for this batch
        if guards is not None:
            guards.append((tok_flag, torch.zeros(1, dtype=torch.int32, device=self.device)))
        ws = self._eval_ws.get(ops.eval_ws_bytes(self.ms, M, max_item))
        items = torch.empty((M, max(k, 1)), dtype=torch.int32, device=self.device)
        scores = torch.empty((M, max(k, 1)), dtype=torch.float32, device=self.device)
        ops.eval_rank_topk(self.ms, self.theta, rep, gt_t, max_item, k, ws, rank, items, scores)
        return rank, items, scores

    def check_guards(self, guards) -> list:
        """One host read of the guard words collected by rank_topk(guards=...): raises on an encoder token overflow, returns
        the indices of the calls whose candidate band overflowed (the caller re-runs those with force_exact=True)."""
        if not guards:
            return []
        words = torch.stack([torch.cat([t.view(-1)[:1], b.view(-1)[:1]]) for t, b in guards]).cpu().numpy()
        if self._tight_cap and bool((words[:, 0] != 0).any()):
            raise ops._lib.AderError("encoder: n_tokens was smaller than the number of real tokens in the batch (tokens dropped)")
        redo = [int(i) for i in np.nonzero(words[:, 1])[0]]
        self.eval_fallbacks += len(redo)
        return redo

    def predict(self, sess, seq, item_idx):
        """Reference signature (ADER.py:140-150): full rank matrix ``argsort(argsort(-logits))`` over
        ``item_idx``.  Kept for drop-in use; the evaluator uses ``rank_topk`` and never builds it."""
        ids = _to_ids(seq, self.hp.maxlen, self.device)
        rep, _ = self.encode(ids)
        items = np.asarray(item_idx, dtype=np.int64)
        vmax = int(items.max())
        lg = self.logits(rep, vmax)
        if not (len(items) == vmax and items[0] == 1 and items[-1] == vmax):
            lg = lg[:, torch.from_numpy(items - 1).to(self.device)]
        order = torch.argsort(lg, dim=1, descending=True, stable=True)
        ranks = torch.empty_like(order)
        ar = torch.arange(order.shape[1], device=self.device).expand_as(order)
        ranks.scatter_(1, order, ar)
        return ranks.cpu().numpy()

    # ---- checkpoint (tf.train.Saver analogue, main.py:209-213,280,283) ---------------------------
    def state_dict(self):
        return {"theta": self.theta.clone(), "adam_m": self.adam_m.clone(), "adam_v": self.adam_v.clone(),
                "adam_state": self.adam_state.clone(), "global_step": self.global_step}

    def _dp_quiesce(self):
        """Peer back end: other ranks store into this replica's theta during their update; wait (stream-ordered) until
        every rank has finished the last one before the host rewrites theta."""
        if self.dp is not None:
            self.dp.begin_step(self)

    def load_state_dict(self, sd):
        self._dp_quiesce()
        self.theta.copy_(sd["theta"]); self.adam_m.copy_(sd["adam_m"]); self.adam_v.copy_(sd["adam_v"])
        self.adam_state.copy_(sd["adam_state"]); self.global_step = int(sd["global_step"])

    def reinitialize(self, seed: Optional[int] = None):
        """sess.run(tf.global_variables_initializer()) (main.py:213)."""
        s = self.seed if seed is None else seed
        self._dp_quiesce()
        self.theta.copy_(torch.from_numpy(self.layout.init_flat(s)))
        self.adam_m.zero_(); self.adam_v.zero_(); self.adam_state.zero_(); self.global_step = 0

    def save(self, path: str):
        torch.save({k: (v.cpu() if isinstance(v, torch.Tensor) else v) for k, v in self.state_dict().items()}, path)

    def restore(self, path: str):
        sd = torch.load(path, map_location=self.device)
        self.load_state_dict(sd)


class Ewc(Ader):
    """EWC baseline (EWC.py:14-177): same network, CE + (lambda/2) sum F (theta - theta*)^2."""

    def __init__(self, item_num: int, args, device=None, init_seed=None):
        super().__init__(item_num, args, device, init_seed)
        self.fisher: Optional[torch.Tensor] = None          # F_accum, flat fp32
        self.theta_star: Optional[torch.Tensor] = None      # variables_prev, flat fp32
        self._fisher_acc: Optional[torch.Tensor] = None
        self.ewc_lambda = 0.0
        self._graph_fisher = None
        self._graph_star = None
        # "batched": ader_fisher_batched (one pass for all samples); "loop": one forward + backward per sample like EWC.py:142-161
        self.fisher_impl = getattr(args, "fisher_impl", None) or os.environ.get("ADER_B200_FISHER", "batched")

    @property
    def variables_prev(self):
        return None if self.theta_star is None else self.layout.views(self.theta_star)

    @variables_prev.setter
    def variables_prev(self, value):
        """main.py:260,321 assign ``sess.run(model.variables)``; accept that list or a flat tensor."""
        if isinstance(value, torch.Tensor):
            self.theta_star = value.detach().clone()
        else:
            self.theta_star = torch.cat([torch.as_tensor(v, device=self.device).reshape(-1) for v in value]).float()

    def snapshot_variables(self):
        """sess.run(model.variables) as one flat device tensor."""
        return self.theta.clone()

    def set_vanilla_loss(self):
        super().set_vanilla_loss()
        self.ewc_lambda = 0.0

    def update_loss(self, lambda_: float):
        """EWC.py:115-124.  TF bakes F_accum / variables_prev into the graph as CONSTANTS at this
        call (SURVEY S13), so later reassignments do not affect the running train_op: freeze copies."""
        self.mode = self.VANILLA
        self.ewc_lambda = float(lambda_)
        self._graph_fisher = self.fisher.clone()
        self._graph_star = self.theta_star.clone()

    def _opt_args(self, max_item: int, lr: float):
        if self.ewc_lambda != 0.0:
            return (max_item, lr, self.ewc_lambda, self._graph_fisher, self._graph_star)
        return (max_item, lr, 0.0, None, None)

    def apply_gradients(self, max_item: int, lr: float, ewc_lambda: float = 0.0, fisher=None, theta_star=None):
        if self.ewc_lambda != 0.0:
            super().apply_gradients(max_item, lr, self.ewc_lambda, self._graph_fisher, self._graph_star)
        else:
            super().apply_gradients(max_item, lr)

    def compute_fisher(self, sess, data: Sequence[Sequence[int]], batch_size: int, max_item: int):
        """EWC.py:126-164: per-sample (batch of one) squared gradients of the vanilla CE in eval mode,
        accumulated in float64, divided by len(data).  Consumes the Python RNG like the reference
        (Sampler shuffle at construction and at wrap)."""
        from .data import Sampler
        sampler = Sampler(data, self.hp.maxlen, batch_size, is_subseq=True)
        if self._fisher_acc is None:
            self._fisher_acc = torch.zeros(self.layout.total, dtype=torch.float64, device=self.device)
        acc = self._fisher_acc
        acc.zero_()
        batched = self.fisher_impl == "batched" and self.hp.hidden_units <= 160
        rows_ids, rows_pos = [], []
        for _ in range(sampler.batch_num()):
            seq, pos = sampler.sampler_arrays()
            if batched:
                rows_ids.append(seq); rows_pos.append(pos)
                continue
            for i in range(seq.shape[0]):                    # the reference's own shape of work: one pass per sample
                self.loss_and_grad(seq[i:i + 1], pos[i:i + 1], max_item, mode=self.VANILLA, lambda_=0.0,
                                   n_tokens=int((seq[i] != 0).sum()))
                ops.fisher_accumulate(self.ms, self.grad, acc, max_item)
        if batched and rows_ids:
            ids_all = np.concatenate(rows_ids).astype(np.int32)
            pos_all = np.concatenate(rows_pos).astype(np.int32)
            CH = 1024                                        # samples per batched pass (bounds the activation workspaces)
            for lo in range(0, ids_all.shape[0], CH):
                ids = _to_ids(ids_all[lo:lo + CH], self.hp.maxlen, self.device)
                pos_t = _to_i32(pos_all[lo:lo + CH], self.device)
                S_ = ids.shape[0]
                tcap = max(int((ids_all[lo:lo + CH] != 0).sum()), 1)
                ews = self._enc_ws.get(ops.encoder_ws_bytes(self.ms, S_, tcap))
                bws = self._bwd_ws.get(ops.encoder_bwd_ws_bytes(self.ms, S_, tcap))
                fws = self._eval_ws.get(ops.fisher_batched_ws_bytes(self.ms, S_, max_item))
                ops.fisher_batched(self.ms, self.theta, ids, pos_t, tcap, max_item, ews, bws, fws, acc)
                self._last_enc = (S_, tcap)
        if self.fisher is None:
            self.fisher = torch.empty(self.layout.total, dtype=torch.float32, device=self.device)
        ops.fisher_finalize(self.ms, acc, self.fisher, max_item, len(data))

    @property
    def F_accum(self):
        return None if self.fisher is None else self.layout.views(self.fisher)
