"""Multi-GPU plumbing for the two ways the path shards (SURVEY 8e); torch.distributed is plumbing only.

* Data parallel (configs 1-4): every rank runs the step on its own rows with the GLOBAL mean
  denominators (AderLossArgs.n_train_global / n_ex_global); the gradients of the ranks are SUMMED.
  Two interchangeable back ends behind ``Ader.dp``:
    - ``PeerComm`` (default): theta / grad / a flag block of every rank are mapped into every process
      (CUDA IPC over NVLink) and the optimiser step is the collective (csrc/dp.cu, ader_dp_adam_step:
      arrive -> reduce-scatter by peer loads + TF1 Adam on the owned slice + all-gather by peer stores ->
      publish; ader_dp_wait at the start of the next step); the optimiser state of a slice is only touched
      by its owner.  No host in the loop, graph-capturable.
    - ``NcclComm``: all-reduce (sum) of the live gradient ranges (table rows 1..max_item and the dense
      parameters: rows above max_item are identically zero), then the ordinary Adam on every rank.
  Row order inside a rank stays [train; exemplar].
* Vocab parallel (config 5, 1 M items): the table rows (and Adam state) are sharded by vocabulary
  range; each rank produces per-row (max, sumexp, label logit, KD dot) partials over its columns --
  exactly what k_tc_logits<FWD> emits per vocabulary chunk -- and the log-sum-exp is merged with an
  all-reduce(max) + all-reduce(sum) (``VocabParallelLoss``: ader_loss_tc_vp_fwd / _bwd on the shard,
  partial d_rep all-reduced).
"""
from __future__ import annotations

import os
from typing import Tuple

import torch
import torch.distributed as dist


def env_rank() -> Tuple[int, int, int]:
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


def shard_range(n: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous balanced shard [lo, hi) of n units: the first n % world ranks get one extra."""
    base, rem = divmod(n, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def shard_rows(n_train: int, n_ex: int, rank: int, world: int):
    """Row shards of one step: train rows and exemplar rows are split SEPARATELY so that every rank
    keeps the [train; exemplar] layout (main.py:229).  Returns ((t_lo, t_hi), (e_lo, e_hi))."""
    return shard_range(n_train, rank, world), shard_range(n_ex, rank, world)


def vocab_shard(V: int, rank: int, world: int, tile: int = 128) -> Tuple[int, int]:
    """Vocabulary columns [lo, hi) of a rank, aligned to the 128-row T128 operand tiles."""
    tiles = (V + tile - 1) // tile
    lo, hi = shard_range(tiles, rank, world)
    return min(lo * tile, V), min(hi * tile, V)


def merge_lse(local_max: torch.Tensor, local_sumexp: torch.Tensor, group=None) -> torch.Tensor:
    """log-sum-exp over vocabulary shards from per-rank (max, sum exp(x - max)) partials."""
    gmax = local_max.clone()
    dist.all_reduce(gmax, op=dist.ReduceOp.MAX, group=group)
    scaled = local_sumexp * torch.exp(local_max - gmax)
    scaled = torch.where(torch.isfinite(local_max), scaled, torch.zeros_like(scaled))
    dist.all_reduce(scaled, op=dist.ReduceOp.SUM, group=group)
    return gmax + torch.log(scaled)


class NcclComm:
    """Gradient all-reduce over NCCL + replicated Adam (fallback back end, and the one gloo tests drive on CPU)."""

    kind = "nccl"

    def __init__(self, model, group=None):
        self.group = group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)

    def begin_step(self, model):
        pass

    def apply(self, model, max_item: int, lr: float, ewc_lambda: float = 0.0, fisher=None, theta_star=None):
        from . import ops
        d = model.hp.hidden_units
        g = model.grad
        # live ranges only: rows > max_item of the table never receive gradient (28 % of the buffer at the bench shape)
        dist.all_reduce(g[d:(max_item + 1) * d], op=dist.ReduceOp.SUM, group=self.group)
        dist.all_reduce(g[model.layout.offset(1):], op=dist.ReduceOp.SUM, group=self.group)
        ops.adam_step(model.ms, model.theta, model.adam_m, model.adam_v, g, model.adam_state, max_item, lr,
                      ewc_lambda, fisher, theta_star)

    def check(self):
        pass


class PeerComm:
    """Peer-memory back end: see csrc/dp.cu.  `peers` = list of (theta_ptr, grad_ptr, flags_ptr) per rank."""

    kind = "p2p"

    def __init__(self, model, rank: int, world: int, peers, flags: torch.Tensor, opened=(), separate_arrive: bool = False,
                 mc_theta: int = 0, mc_grad: int = 0):
        from . import ops
        self.rank, self.world = rank, world
        self.flags = flags                                   # keep the local flag block alive
        self._opened = list(opened)                          # IPC mappings to close
        self.comm = ops.dp_comm(rank, world, [p[0] for p in peers], [p[1] for p in peers], [p[2] for p in peers],
                                separate_arrive=separate_arrive, mc_theta=mc_theta, mc_grad=mc_grad)
        self._ops = ops
        if mc_theta:
            self.kind = "nvls"

    @classmethod
    def from_symmetric_memory(cls, model, group=None):
        """NVLS form: theta, grad and the flag block of every rank live in ONE torch symmetric-memory allocation per rank
        (cuMemCreate + NVSwitch multicast object, set up by torch.distributed._symmetric_memory: plumbing).  The update
        kernel then sums the gradient inside the switch (multimem.ld_reduce) and broadcasts the new parameters with
        multimem.st (csrc/dp.cu k_dp_adam_mc).  The model's ``theta`` / ``grad`` are re-bound to views of that allocation
        (same values).  Returns None when the fabric has no multicast support (the caller falls back to CUDA IPC)."""
        import torch.distributed._symmetric_memory as symm
        from . import ops
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        total = model.theta.numel()
        pad = (total + 3) // 4 * 4                            # grad starts 16-byte aligned, same phase as theta
        words = ops._lib.DP_FLAG_WORDS
        buf = symm.empty(2 * pad + words, dtype=torch.float32, device=model.device)
        hdl = symm.rendezvous(buf, group if group is not None else dist.group.WORLD)
        mc = int(getattr(hdl, "multicast_ptr", 0) or 0)
        have = torch.tensor([1.0 if mc else 0.0], device=model.device)
        dist.all_reduce(have, op=dist.ReduceOp.MIN, group=group)
        if float(have.item()) == 0.0:
            return None
        buf.zero_()
        theta, grad = buf[:total], buf[pad:pad + total]
        flags = buf[2 * pad:2 * pad + words].view(torch.int32)
        theta.copy_(model.theta)
        torch.cuda.synchronize(model.device)
        model.theta, model.grad = theta, grad
        bases = [int(p) for p in hdl.buffer_ptrs]
        peers = [(b, b + 4 * pad, b + 8 * pad) for b in bases]
        dist.barrier(group=group)                             # every replica is initialised before the first step
        comm = cls(model, rank, world, peers, flags, (), mc_theta=mc, mc_grad=mc + 4 * pad)
        comm._symm = (buf, hdl)                               # keep the allocation and the mappings alive
        return comm

    @classmethod
    def from_process_group(cls, model, group=None):
        """Exchange CUDA IPC handles of (theta, grad, flags) through the process group and map the peers."""
        from . import ops
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        if world > ops._lib.DP_MAX_RANKS:
            raise ValueError("PeerComm supports up to %d ranks" % ops._lib.DP_MAX_RANKS)
        flags = torch.zeros(ops._lib.DP_FLAG_WORDS, dtype=torch.int32, device=model.device)
        torch.cuda.synchronize(model.device)
        mine = [ops.ipc_export(t) for t in (model.theta, model.grad, flags)]
        allh = [None] * world
        dist.all_gather_object(allh, mine, group=group)
        opened = {}
        peers = []
        for r in range(world):
            if r == rank:
                peers.append((model.theta.data_ptr(), model.grad.data_ptr(), flags.data_ptr()))
                continue
            ptrs = []
            for handle, off in allh[r]:
                if handle not in opened:                      # two tensors may live in one allocation: map it once
                    opened[handle] = ops.ipc_open(handle)
                ptrs.append(opened[handle] + off)
            peers.append(tuple(ptrs))
        dist.barrier(group=group)                             # every rank has mapped every flag block before the first step
        return cls(model, rank, world, peers, flags, opened.values())

    def begin_step(self, model):
        self._ops.dp_wait(self.comm)

    def apply(self, model, max_item: int, lr: float, ewc_lambda: float = 0.0, fisher=None, theta_star=None):
        self._ops.dp_adam_step(model.ms, self.comm, model.adam_m, model.adam_v, model.adam_state, max_item, lr,
                               ewc_lambda, fisher, theta_star)

    def check(self):
        err, _ = self._ops.dp_status(self.comm)
        if err:
            raise self._ops._lib.AderError("data-parallel peer wait timed out (a rank did not reach the step)")

    def close(self):
        for b in self._opened:
            try:
                self._ops.ipc_close(b)
            except Exception:
                pass
        self._opened = []


def local_peer_group(models):
    """Emulated ranks inside ONE process (tests on a single GPU): every model replica becomes a rank whose peers are
    the other replicas' buffers.  Returns the PeerComm list (also installed as ``model.dp``)."""
    from . import ops
    world = len(models)
    flags = [torch.zeros(ops._lib.DP_FLAG_WORDS, dtype=torch.int32, device=m.device) for m in models]
    peers = [(m.theta.data_ptr(), m.grad.data_ptr(), f.data_ptr()) for m, f in zip(models, flags)]
    comms = []
    for r, m in enumerate(models):
        m.dp = PeerComm(m, r, world, peers, flags[r], separate_arrive=True)
        m.dp._all_flags = flags
        comms.append(m.dp)
    return comms


NVLS_MIN_WORLD = 5      # "auto": in-switch reduction from this world size on (measured: N=4 0.3418 ms nvls vs 0.3375 p2p, N=8 0.3395 vs 0.3554)


def make_comm(model, group=None, backend: str = None):
    """Pick the data-parallel back end: ADER_B200_DP = auto | nvls | p2p | nccl.
    auto (default): NVLS multicast (PeerComm.from_symmetric_memory) for world >= NVLS_MIN_WORLD when the fabric supports
    it, else peer loads / stores over CUDA IPC mappings (p2p), else NCCL.  Every decision is collective."""
    backend = backend or os.environ.get("ADER_B200_DP", "auto")
    world = dist.get_world_size(group)
    if backend in ("auto", "nvls", "p2p") and model.device.type == "cuda":
        want_nvls = backend == "nvls" or (backend == "auto" and world >= NVLS_MIN_WORLD)
        ok = torch.ones(1, device=model.device)
        comm = None
        try:
            if want_nvls:
                try:
                    comm = PeerComm.from_symmetric_memory(model, group)
                except Exception as ex:      # noqa: BLE001 -- no symmetric memory / multicast here: plain peer mappings
                    import sys
                    sys.stderr.write("[ader_b200] NVLS multicast unavailable on rank %d (%r); peer loads / stores\n" % (dist.get_rank(group), ex))
                    comm = None
            if comm is None:
                comm = PeerComm.from_process_group(model, group)
        except Exception as ex:      # noqa: BLE001 -- e.g. IPC not permitted in this container: every rank must agree
            import sys
            sys.stderr.write("[ader_b200] peer-memory data parallel unavailable on rank %d (%r); using NCCL\n" % (dist.get_rank(group), ex))
            ok.zero_()
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
        if float(ok.item()) > 0:
            return comm
        if comm is not None:
            comm.close()
    return NcclComm(model, group)


class DataParallel:
    """Wrap an `Ader` / `Ewc` model: shard each step's rows over the ranks, sum the gradients (``model.dp``)."""

    def __init__(self, model, group=None, backend: str = None):
        self.model, self.group = model, group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        model.dp = make_comm(model, group, backend)

    def train_step(self, seq, pos, max_item, lr=None, dropout_rate=None, exemplar_logits=None, exemplar_pos=None,
                   teacher_rows=None):
        """Same feed as Ader.train_step with the GLOBAL batch on every rank; each rank keeps its shard."""
        n_train = len(pos)
        n_ex = len(seq) - n_train
        (tl, th), (el, eh) = shard_rows(n_train, n_ex, self.rank, self.world)
        rows = list(range(tl, th)) + list(range(n_train + el, n_train + eh))
        if isinstance(seq, torch.Tensor):
            seq_l = seq[torch.as_tensor(rows, device=seq.device)]
        else:
            seq_l = [seq[i] for i in rows]
        kw = {}
        if exemplar_logits is not None:
            if teacher_rows is not None:
                kw["exemplar_logits"], kw["teacher_rows"] = exemplar_logits, teacher_rows[el:eh]
            else:
                kw["exemplar_logits"] = exemplar_logits[el:eh]
        if exemplar_pos is not None:
            kw["exemplar_pos"] = exemplar_pos[el:eh]
        m = self.model
        m.global_counts = (n_train, n_ex)
        loss = m.train_step(seq_l, pos[tl:th], max_item, lr, dropout_rate, **kw)
        loss = loss.clone()
        dist.all_reduce(loss, op=dist.ReduceOp.SUM, group=self.group)
        return loss


class VocabParallelLoss:
    """Vocab-parallel logits + softmax CE + distillation (BASELINE config 5): every rank holds all `rep`
    rows and the table rows of its vocabulary shard [v_lo, v_hi); the tcgen05 kernels run on the shard and
    two tiny collectives stitch the softmax together:
        all-reduce(max) of the per-row maxima, all-reduce(sum) of (rescaled sumexp, label logit, KD dot),
    and one all-reduce(sum) of the partial d_rep [M, d] in backward.  dE needs no communication (each rank
    owns its rows).  With `group=None` and world size 1 it degenerates to the single-GPU kernel."""

    def __init__(self, model, group=None, rank=None, world=None):
        from . import ops
        self.ops, self.model, self.group = ops, model, group
        self.rank = dist.get_rank(group) if rank is None else rank
        self.world = dist.get_world_size(group) if world is None else world
        self.ws = ops.Workspace(model.device)

    def shard(self, V: int):
        return vocab_shard(V, self.rank, self.world)

    def local_forward(self, rep, a, v_lo, v_hi):
        ops, m = self.ops, self.model
        ws = self.ws.get(ops.loss_tc_vp_ws_bytes(m.ms, a, v_lo, v_hi))
        stats = torch.empty((a.M, 4), dtype=torch.float32, device=m.device)
        ops.loss_tc_vp_fwd(m.ms, m.theta, rep, a, v_lo, v_hi, ws, stats)
        return ws, stats

    @staticmethod
    def merge(stats_list_or_tensor, n_train: int, n_ex: int, lambda_: float, kd: bool, reduce_max=None, reduce_sum=None):
        """(max, sumexp, label, dot) partials -> lse, row_loss, loss.  `reduce_*` are the collectives
        (identity when the partials of all shards are passed as a list)."""
        if isinstance(stats_list_or_tensor, (list, tuple)):
            st = torch.stack(list(stats_list_or_tensor))                       # [S, M, 4]
            gmax = st[..., 0].max(dim=0).values
            scale = torch.where(torch.isfinite(st[..., 0]), torch.exp(st[..., 0] - gmax), torch.zeros_like(st[..., 0]))
            rest = torch.stack([(st[..., 1] * scale).sum(0), st[..., 2].sum(0), st[..., 3].sum(0)], dim=1)
        else:
            st = stats_list_or_tensor
            gmax = st[:, 0].clone()
            reduce_max(gmax)
            scale = torch.where(torch.isfinite(st[:, 0]), torch.exp(st[:, 0] - gmax), torch.zeros_like(gmax))
            rest = torch.stack([st[:, 1] * scale, st[:, 2], st[:, 3]], dim=1).contiguous()
            reduce_sum(rest)
        lse = gmax + torch.log(rest[:, 0])
        row_loss = lse - rest[:, 1]
        if kd and n_ex > 0:
            row_loss[n_train:] = lse[n_train:] - rest[n_train:, 2]
        loss = row_loss[:n_train].mean() if n_train > 0 else row_loss.new_zeros(())
        if n_ex > 0:
            loss = loss + lambda_ * row_loss[n_train:].mean()
        return lse.contiguous(), row_loss, loss

    def fwd_bwd(self, rep, pos, max_item, lambda_=0.0, mode=0, teacher=None, teacher_rows=None, ex_pos=None, grad=None):
        """rep [M, d] (replicated) -> (loss, row_loss, d_rep); writes this rank's rows of `grad` (flat)."""
        ops, m = self.ops, self.model
        M, n_train = rep.shape[0], pos.numel()
        n_ex = M - n_train
        if teacher is not None and not isinstance(teacher, torch.Tensor):
            raise ValueError("the vocab-parallel loss takes stored teacher logits only (a frozen teacher would need its "
                             "statistics all-reduced over the vocabulary shards)")
        v_prev = teacher.shape[1] if teacher is not None else 0
        a = ops.make_loss_args(M, n_train, n_ex, max_item, v_prev, mode if n_ex > 0 else 0, lambda_, pos, ex_pos, teacher, teacher_rows)
        v_lo, v_hi = self.shard(max_item)
        ws, stats = self.local_forward(rep, a, v_lo, v_hi)
        lse, row_loss, loss = self.merge(stats, n_train, n_ex, lambda_, mode == 1,
                                         lambda t: dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group),
                                         lambda t: dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group))
        d_rep = torch.empty_like(rep)
        ops.loss_tc_vp_bwd(m.ms, m.theta, rep, a, v_lo, v_hi, ws, lse, d_rep, m.grad if grad is None else grad)
        dist.all_reduce(d_rep, op=dist.ReduceOp.SUM, group=self.group)
        self._keep = (a, pos, teacher, teacher_rows, ex_pos, stats, lse)
        return loss, row_loss, d_rep
