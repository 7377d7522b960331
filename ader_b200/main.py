"""Continual-learning driver with the reference's CLI (main.py:68-336): same flags and defaults
(incl. the ``type=bool`` parsing quirk, SURVEY S8), same period / epoch / early-stop / exemplar
protocol, same Training_logs.txt lines -- re-hosted on the GPU-resident fast paths.

    python -m ader_b200.main --dataset=DIGINETICA            # ADER defaults
    python -m ader_b200.main --dataset=YOOCHOOSE --lambda_=1.0 --batch_size=512 --test_batch=64

Extra flags (not in the reference): --data_root, --max_periods, --results_root.
"""
from __future__ import annotations

import argparse
import gc
import math
import os
import random
import time

import numpy as np
import torch

from . import ops
from .data import DataLoader, Evaluator, ExemplarGenerator, ExemplarSet, FrozenTeacher, Sampler, pack_rows
from .model import Ader, Ewc

ITEM_NUM = {"DIGINETICA": 43136, "YOOCHOOSE": 25958}     # main.py:133-138


def get_periods(data_dir: str):                            # main.py:36-51
    n = len([f for f in os.listdir(data_dir) if f.startswith("period_") and f.endswith(".txt")])
    return list(range(1, n))


def build_parser() -> argparse.ArgumentParser:             # main.py:75-108 (types as in the reference)
    p = argparse.ArgumentParser()
    p.add_argument("--dataset", default="DIGINETICA", type=str)
    p.add_argument("--save_dir", default="ADER", type=str)
    p.add_argument("--exemplar_size", default=30000, type=int)
    p.add_argument("--lambda_", default=0.8, type=float)
    p.add_argument("--finetune", default=False, type=bool)
    p.add_argument("--dropout", default=False, type=bool)
    p.add_argument("--ewc", default=False, type=bool)
    p.add_argument("--joint", default=False, type=bool)
    p.add_argument("--ewc_sample_num", default=1000, type=int)
    p.add_argument("--selection", default="herding", type=str)
    p.add_argument("--disable_distillation", default=False, type=bool)
    p.add_argument("--equal_exemplar", default=False, type=bool)
    p.add_argument("--fix_lambda", default=False, type=bool)
    p.add_argument("--num_epochs", default=100, type=int)
    p.add_argument("--batch_size", default=256, type=int)
    p.add_argument("--test_batch", default=64, type=int)
    p.add_argument("--device_num", default=0, type=int)
    p.add_argument("--lr", default=0.0005, type=float)
    p.add_argument("--num_blocks", default=2, type=int)
    p.add_argument("--num_heads", default=1, type=int)
    p.add_argument("--stop", default=5, type=int)
    p.add_argument("--random_seed", default=0, type=int)
    p.add_argument("--hidden_units", default=150, type=int)
    p.add_argument("--maxlen", default=50, type=int)
    p.add_argument("--dropout_rate", default=0.3, type=float)
    p.add_argument("--l2_emb", default=0.0, type=float)
    # additions
    p.add_argument("--data_root", default=None, type=str)
    p.add_argument("--results_root", default="results", type=str)
    p.add_argument("--max_periods", default=0, type=int)
    p.add_argument("--item_num", default=0, type=int)
    p.add_argument("--loss_impl", default="tc", choices=["tc", "exact"], type=str)      # logits+CE+KD: tcgen05 bf16 / fp32
    # distillation teacher: the exemplars' stored [E, V_prev] logits, or a frozen snapshot (exemplar reps + a copy of the item
    # table) from which the loss recomputes them every step -- O(E*d + V_prev*d) memory instead of O(E*V_prev)
    p.add_argument("--teacher", default="logits", choices=["logits", "frozen"], type=str)
    p.add_argument("--encoder_impl", default=None, choices=["tc", "exact"], type=str)  # training encoder (default follows loss_impl)
    p.add_argument("--infer_encoder_impl", default="exact", choices=["tc", "exact"], type=str)  # eval / herding encoder
    # SURVEY 8(f)1/3: per-period checkpoint + resume (the reference cannot resume a run), binary cache of the period files
    p.add_argument("--checkpoint", default=True, type=lambda v: str(v).lower() not in ("0", "false", "no"))
    p.add_argument("--resume", default=False, type=lambda v: str(v).lower() not in ("0", "false", "no"))
    p.add_argument("--cache_dir", default=None, type=str)
    p.add_argument("--step_impl", default=None, choices=["dag", "serial", "groups"], type=str)   # how a tc train step is issued (model.py)
    p.add_argument("--graph", default=True, type=lambda v: str(v).lower() not in ("0", "false", "no"))  # CUDA-graph train step
    # SURVEY 8e: data parallel under torchrun (one process per GPU).  Every rank runs the same host protocol with the same
    # seeds (identical batches, splits, exemplar sets); a step's train rows and exemplar rows are split over the ranks,
    # losses use the global-mean denominators, gradients are summed (ader_b200/dist.py), evaluation rows are sharded.
    p.add_argument("--epoch_queue", default=True, type=lambda v: str(v).lower() not in ("0", "false", "no"))  # host out of the step loop
    p.add_argument("--dp", default=False, type=lambda v: str(v).lower() not in ("0", "false", "no"))
    return p


class PeriodTrainer:
    """One period's epoch loop on GPU-resident rows (main.py:217-256)."""

    def __init__(self, model: Ader, train_sampler: Sampler, exemplar_sampler, args, max_item: int):
        self.model, self.args, self.max_item = model, args, max_item
        self.ts, self.es = train_sampler, exemplar_sampler
        dev = model.device
        self.t_ids, self.t_lab = train_sampler.device_rows(dev)
        self.t_nin = train_sampler.packed()[2]
        if exemplar_sampler is not None:
            self.e_ids, self.e_lab = exemplar_sampler.device_rows(dev)
            self.e_nin = exemplar_sampler.packed()[2]
        self.rows_seen = 0
        self.trace = None
        self.trace_rows = None
        # the step as CUDA graphs, one GraphStep per batch geometry (n_train, n_ex).  The reference drops rows of length <= 1
        # from a batch (util.py:228-229), so a few rows are missing from about half of the batches of some periods: the
        # full geometry is captured at once, any other after its third appearance (at most MAX_GEOM of them)
        self.gs_map = {}
        self._geom_seen = {}
        self._graph_off = False
        self.n_eager = 0                # steps issued launch by launch (rare batch geometry / no graph)
        # data parallel: this rank's shard of every batch (train rows and exemplar rows split separately, main.py:229 order kept)
        self.rank, self.world = getattr(args, "dp_rank", 0), getattr(args, "dp_world", 1)
        # epoch-resident index queue: the row indices of a whole epoch are uploaded once, every step is then a graph
        # replay that gathers its batch from the queue on the device (run_epoch)
        steps = max(train_sampler.batch_num(), 1)
        width = train_sampler.batch_size + (exemplar_sampler.batch_size if exemplar_sampler is not None else 0)
        self.q = torch.zeros(steps * max(width, 1), dtype=torch.int32, device=dev)
        self.q_off = torch.zeros(steps, dtype=torch.int64, device=dev)
        self.q_counter = torch.zeros(1, dtype=torch.int32, device=dev)
        self.host_s = {"plan": 0.0, "launch": 0.0}         # host seconds spent planning epochs / launching their steps
        self._q_copied = None                               # event: the last epoch's queue copies are done
        self._q_host = torch.zeros(steps * max(width, 1), dtype=torch.int32).pin_memory()
        self._qoff_host = torch.zeros(steps, dtype=torch.int64).pin_memory()

    MAX_GEOM = 8

    @property
    def gs(self):
        """The GraphStep of the full batch geometry (None before its first use)."""
        full = (self.args.batch_size, self.es.batch_size if self.es is not None else 0)
        return self.gs_map.get(full)

    def graph_use(self) -> dict:
        out = {}
        for (nt, ne), g in sorted(self.gs_map.items()):
            out["%d+%d" % (nt, ne)] = dict(sorted(g.use_count.items()))
        return out

    def _shard(self, n_train: int, n_ex: int):
        from .dist import shard_rows
        return shard_rows(n_train, n_ex, self.rank, self.world)

    def _graph(self, n_train: int, n_ex: int):
        """GraphStep for this (global) batch geometry (ader_b200/graph.py), built on demand; None = run the step eagerly.
        Data parallel: the decision depends on global quantities only, so every rank takes the same branch."""
        key = (n_train, n_ex)
        gs = self.gs_map.get(key)
        if gs is not None:
            return gs
        m, args = self.model, self.args
        if self._graph_off or not getattr(args, "graph", True):
            return None
        if self.world > 1 and (n_train < self.world or (self.es is not None and n_ex < self.world)):
            return None                 # a rank would be left without rows: rare tail batch, eager on every rank
        if m.encoder_impl != "tc" and args.dropout_rate > 0:
            self._graph_off = True
            return None
        full = (args.batch_size, self.es.batch_size if self.es is not None else 0)
        seen = self._geom_seen[key] = self._geom_seen.get(key, 0) + 1
        if key != full and (seen < 3 or len(self.gs_map) >= self.MAX_GEOM):
            return None
        dev = m.device
        e_ids = e_aux = teacher = None
        if self.es is not None:
            if m.disable_distillation:
                e_aux = self.e_lab
            elif getattr(self.es, "teacher", None) is not None:
                e_aux = torch.as_tensor(np.asarray(self.es.logits, dtype=np.int32)).to(dev)
                teacher = self.es.teacher
            else:
                self._graph_off = True   # host-resident teacher lists (reference feed): eager path
                return None
            e_ids = self.e_ids
        (tl, th), (el, eh) = self._shard(n_train, n_ex)
        if self.world > 1:
            m.global_counts = (n_train, n_ex)       # baked into the captured loss arguments
        n_train, n_ex = th - tl, eh - el
        mean_tok = n_train * float(np.mean(self.t_nin)) + (n_ex * float(np.mean(self.e_nin)) if self.es is not None else 0.0)
        caps = [int(mean_tok * f) + 64 for f in (1.1, 1.3, 1.7)]
        gs = m.graph_step(n_train, n_ex, self.max_item, args.lr, args.dropout_rate, teacher=teacher,
                          sources=(self.t_ids, self.t_lab, e_ids, e_aux) if self.es is not None
                          else (self.t_ids, self.t_lab, None, None), tcaps=caps, queue=(self.q, self.q_off, self.q_counter))
        self.gs_map[key] = gs
        return gs

    def run_epoch(self, n_steps: int):
        """One epoch (main.py:220-256) with the host out of the loop: the samplers are advanced a chunk of steps ahead of the
        GPU (same calls in the same order as step-by-step, so both host RNG streams move identically), the row indices go to
        the device chunk by chunk, and every step is a graph replay that gathers its batch from that queue.  A step whose
        batch geometry has no graph (rare tail batches) runs eagerly from the same queue."""
        m = self.model
        if self._q_copied is not None:
            self._q_copied.synchronize()                         # last epoch's queue copies have left the pinned buffers
        qh, oh = self._q_host.numpy(), self._qoff_host.numpy()
        self.q_counter.zero_()
        o, s0, loss = 0, 0, None
        # planned and launched in chunks, so the host plans chunk k+1 while the GPU runs chunk k (first chunk short: the
        # GPU starts after a few steps' worth of planning)
        while s0 < n_steps:
            s1 = min(n_steps, s0 + (self.CHUNK0 if s0 == 0 else self.CHUNK))
            t0 = time.time()
            plan, o0 = [], o
            for s_ in range(s0, s1):
                ti = self.ts.next_indices()
                ei = self.es.next_indices() if self.es is not None else np.zeros(0, np.int64)
                key = (len(ti), len(ei))
                self.rows_seen += len(ti) + len(ei)
                if self.world > 1:
                    (tl, th), (el, eh) = self._shard(len(ti), len(ei))
                    ti, ei = ti[tl:th], ei[el:eh]
                n_tok = int(self.t_nin[ti].sum()) + (int(self.e_nin[ei].sum()) if self.es is not None else 0)
                oh[s_] = o
                qh[o:o + len(ti)] = ti
                qh[o + len(ti):o + len(ti) + len(ei)] = ei
                o += len(ti) + len(ei)
                plan.append((key, len(ti), len(ei), n_tok))
            if o > o0:
                self.q[o0:o].copy_(self._q_host[o0:o], non_blocking=True)
            self.q_off[s0:s1].copy_(self._qoff_host[s0:s1], non_blocking=True)
            t1 = time.time()
            self.host_s["plan"] += t1 - t0
            i = 0
            while i < len(plan):
                # runs of GROUP consecutive steps of one batch geometry go out as ONE graph replay (capacity = the largest
                # of their buckets): the replay-to-replay launch gap is paid once per GROUP steps
                key, _, _, n_tok = plan[i]
                n = self.GROUP
                if n > 1 and i + n <= len(plan) and all(plan[i + k][0] == key for k in range(1, n)):
                    gs = self.gs_map.get(key)
                    if gs is not None and self._geom_multi(key):
                        if self.world > 1:
                            m.global_counts = key
                        loss = gs.run_queued(max(plan[i + k][3] for k in range(n)), nsteps=n)
                        i += n
                        continue
                loss = self._launch_queued(*plan[i])
                i += 1
            self.host_s["launch"] += time.time() - t1
            s0 = s1
        if self._q_copied is None:
            self._q_copied = torch.cuda.Event()
        self._q_copied.record()
        return loss

    CHUNK0, CHUNK = 8, 48
    GROUP = int(os.environ.get("ADER_B200_GRAPH_STEPS", "1"))     # steps per graph replay in a queued epoch (measured: 4 buys < 1 %, costs captures)

    def _geom_multi(self, key) -> bool:
        """Multi-step graphs only for the full batch geometry (nearly every step of an epoch; rare geometries are not
        worth another capture)."""
        full = (self.args.batch_size, self.es.batch_size if self.es is not None else 0)
        return key == full

    def _launch_queued(self, key, nt, ne, n_tok):
        """One step of a queued epoch: graph replay, or (rare batch geometry) eager launches from the same queue."""
        m, dev, L = self.model, self.model.device, self.model.hp.maxlen
        gs = self._graph(*key) if (key[0] > 0 and (self.es is None or key[1] > 0)) else None
        if self.world > 1:
            m.global_counts = key
        if gs is not None:
            return gs.run_queued(n_tok)
        self.n_eager += 1
        ids = torch.empty((nt + ne, L), dtype=torch.int32, device=dev)
        pos = torch.empty(nt, dtype=torch.int32, device=dev)
        aux = torch.empty(max(ne, 1), dtype=torch.int32, device=dev)
        e_aux = None
        if self.es is not None:
            e_aux = self.e_lab if m.disable_distillation else self._teacher_rows()
        ops.gather_batch_q(self.t_ids, self.t_lab, nt, self.e_ids if ne else None, e_aux if ne else None, ne, self.q, self.q_off,
                           self.q_counter, ids, pos, aux[:ne] if ne else None)
        ops.queue_advance(self.q_counter)
        if self.es is None or ne == 0:
            return m.train_step(ids, pos, self.max_item, self.args.lr, self.args.dropout_rate, n_tokens=n_tok)
        if m.disable_distillation:
            return m.train_step(ids, pos, self.max_item, self.args.lr, self.args.dropout_rate, exemplar_pos=aux[:ne], n_tokens=n_tok)
        return m.train_step(ids, pos, self.max_item, self.args.lr, self.args.dropout_rate, exemplar_logits=self.es.teacher,
                            teacher_rows=aux[:ne], n_tokens=n_tok)

    def _teacher_rows(self):
        if getattr(self, "_trows", None) is None:
            self._trows = torch.as_tensor(np.asarray(self.es.logits, dtype=np.int32)).to(self.model.device)
        return self._trows

    def can_queue(self) -> bool:
        """The queued epoch needs GPU-resident exemplar logits (ExemplarSet.teacher) or no exemplars at all."""
        if not getattr(self.args, "graph", True):
            return False
        m = self.model
        if m.encoder_impl != "tc" and self.args.dropout_rate > 0:
            return False
        return self.es is None or m.disable_distillation or getattr(self.es, "teacher", None) is not None

    def step(self):
        loss = self._step()
        if self.trace is not None:
            self.trace.append(float(loss.item()))
            if self.trace_rows is not None:
                self.trace_rows.append((self.model.last_row_loss.cpu().numpy(), self.model._keep[0].cpu().numpy()))
        return loss

    def _step(self):
        m, dev, L = self.model, self.model.device, self.model.hp.maxlen
        ti = self.ts.next_indices()
        ei = self.es.next_indices() if self.es is not None else np.zeros(0, np.int64)
        gs = self._graph(len(ti), len(ei)) if (len(ti) > 0 and (self.es is None or len(ei) > 0)) else None
        self.rows_seen += len(ti) + len(ei)                      # rows of the whole step (all ranks)
        if self.world > 1:                                       # keep this rank's rows; the means stay global
            m.global_counts = (len(ti), len(ei))
            (tl, th), (el, eh) = self._shard(len(ti), len(ei))
            ti, ei = ti[tl:th], ei[el:eh]
        n_tok = int(self.t_nin[ti].sum()) + (int(self.e_nin[ei].sum()) if self.es is not None else 0)
        if gs is not None:
            return gs.run_indices(ti, ei if self.es is not None else None, n_tok)
        self.n_eager += 1                                        # rare batch geometry / no graph
        ti_d = torch.from_numpy(ti.astype(np.int32)).pin_memory().to(dev, non_blocking=True)
        ids = torch.empty((len(ti) + len(ei), L), dtype=torch.int32, device=dev)
        ops.gather_rows_i32(self.t_ids, ti_d, ids[:len(ti)])
        pos = self.t_lab[ti_d.long()]
        if self.es is None:
            return m.train_step(ids, pos, self.max_item, self.args.lr, self.args.dropout_rate, n_tokens=n_tok)
        ei_d = torch.from_numpy(ei.astype(np.int32)).pin_memory().to(dev, non_blocking=True)
        if len(ei):
            ops.gather_rows_i32(self.e_ids, ei_d, ids[len(ti):])
        if m.disable_distillation:
            return m.train_step(ids, pos, self.max_item, self.args.lr, self.args.dropout_rate,
                                exemplar_pos=self.e_lab[ei_d.long()], n_tokens=n_tok)
        if getattr(self.es, "teacher", None) is not None:
            rows = torch.as_tensor(np.asarray([self.es.logits[i] for i in ei], dtype=np.int32)).to(dev)
            return m.train_step(ids, pos, self.max_item, self.args.lr, self.args.dropout_rate,
                                exemplar_logits=self.es.teacher, teacher_rows=rows, n_tokens=n_tok)
        lg = np.asarray([self.es.logits[i] for i in ei], dtype=np.float32)
        return m.train_step(ids, pos, self.max_item, self.args.lr, self.args.dropout_rate, exemplar_logits=lg, n_tokens=n_tok)


# ---- per-period checkpoint (SURVEY 8(f)1) -------------------------------------------------------------------
# One file per run, rewritten atomically at the end of every period: everything the next period reads from the
# previous ones -- best weights + Adam slots + step counter, the exemplar SESSIONS (their teacher logits are
# recomputed from those weights on resume: the exact inference path is deterministic, so they come back bit-identical
# without writing up to 5 GB per period), item universe, early-stop counter, metrics, both host RNG states, EWC state.
CKPT_NAME = "checkpoint.pt"


PROTOCOL_KEYS = ("dataset", "exemplar_size", "lambda_", "finetune", "dropout", "ewc", "joint", "ewc_sample_num", "selection",
                 "disable_distillation", "equal_exemplar", "fix_lambda", "batch_size", "lr", "num_blocks", "num_heads",
                 "random_seed", "hidden_units", "maxlen", "dropout_rate", "item_num", "teacher")
PROTOCOL_DEFAULTS = {"teacher": "logits"}         # value of a key a checkpoint written before the key existed stands for


def protocol_args(args) -> dict:
    """The flags that define the run's protocol: a checkpoint only resumes under the same ones."""
    out = {}
    for k in PROTOCOL_KEYS:
        v = getattr(args, k, None)
        out[k] = os.path.basename(str(v).rstrip("/")) if k == "dataset" else v
    return out


def save_period_checkpoint(path: str, period: int, model, dataloader, fast_exemplar, carry: dict, args=None) -> None:
    st = {"format": 1, "period": int(period), "args": None if args is None else protocol_args(args), "model": {k: (v.cpu() if isinstance(v, torch.Tensor) else v)
                                                      for k, v in model.state_dict().items()},
          "item_set": np.array(sorted(dataloader.item_set), dtype=np.int64),
          "exemplar_sessions": None if fast_exemplar is None else [list(map(int, x)) for x in fast_exemplar.sessions],
          "teacher_width": None if fast_exemplar is None or fast_exemplar.teacher is None else _teacher_cols(fast_exemplar.teacher),
          "teacher_form": "frozen" if fast_exemplar is not None and isinstance(fast_exemplar.teacher, FrozenTeacher) else "logits",
          "carry": carry, "py_random": random.getstate(), "np_random": np.random.get_state()}
    if isinstance(model, Ewc):
        st["ewc"] = {"fisher": None if model.fisher is None else model.fisher.cpu(),
                     "theta_star": None if model.theta_star is None else model.theta_star.cpu()}
    tmp = path + ".tmp"
    torch.save(st, tmp)
    os.replace(tmp, path)


def _teacher_cols(teacher) -> int:
    return teacher.width if isinstance(teacher, FrozenTeacher) else int(teacher.shape[1])


def rebuild_exemplars(model, sessions, teacher_width: int, maxlen: int, chunk: int = 4096, form: str = "logits") -> ExemplarSet:
    """Exemplar store of a resumed run: stored logits = logits of the saved sessions under the restored weights
    (what ExemplarGenerator._store computed with the same weights at the end of the period, util.py:433); in the frozen
    form the snapshot of those weights (the sessions' reps and the table), which is what _store kept."""
    rows = [list(x) for x in sessions]
    if teacher_width is None:
        return ExemplarSet(rows, None)
    ids, _, n_in = pack_rows(rows, maxlen)
    if form == "frozen":
        reps = [model.rep(ids[lo:lo + chunk], n_tokens=int(n_in[lo:lo + chunk].sum())).clone() for lo in range(0, len(rows), chunk)]
        rep = torch.cat(reps) if reps else torch.zeros((0, model.hp.hidden_units), device=model.device)
        return ExemplarSet(rows, FrozenTeacher(model, rep, teacher_width))
    # one [E, ld] buffer with 16-byte aligned rows (ld % 4 == 0), as ExemplarGenerator._store builds it: the teacher kernels
    # read stored logits with 128-bit loads only then
    ld = (teacher_width + 3) // 4 * 4
    teacher = torch.zeros((len(rows), ld), dtype=torch.float32, device=model.device)[:, :teacher_width]
    for lo in range(0, len(rows), chunk):
        r = model.rep(ids[lo:lo + chunk], n_tokens=int(n_in[lo:lo + chunk].sum()))
        teacher[lo:lo + chunk] = model.logits(r.contiguous(), teacher_width)
    return ExemplarSet(rows, teacher)


def load_period_checkpoint(path: str, model, dataloader, maxlen: int, args=None):
    st = torch.load(path, map_location="cpu", weights_only=False)
    if st.get("format") != 1:
        raise ValueError("%s: unknown checkpoint format" % path)
    if args is not None and st.get("args") is not None:      # refuse to continue a run under a different protocol
        now = protocol_args(args)
        diff = {k: (st["args"].get(k, PROTOCOL_DEFAULTS.get(k)), now[k]) for k in now
                if st["args"].get(k, PROTOCOL_DEFAULTS.get(k)) != now[k]}
        if diff:
            raise ValueError("%s was written by a run with different flags (saved, now): %s" % (path, diff))
    model.load_state_dict({k: (v.to(model.device) if isinstance(v, torch.Tensor) else v) for k, v in st["model"].items()})
    dataloader.item_set = set(int(x) for x in st["item_set"])
    if isinstance(model, Ewc) and st.get("ewc"):
        e = st["ewc"]
        model.fisher = None if e["fisher"] is None else e["fisher"].to(model.device)
        model.theta_star = None if e["theta_star"] is None else e["theta_star"].to(model.device)
    ex = None
    if st["exemplar_sessions"] is not None:
        ex = rebuild_exemplars(model, st["exemplar_sessions"], st["teacher_width"], maxlen, form=st.get("teacher_form", "logits"))
    random.setstate(st["py_random"])
    np.random.set_state(st["np_random"])
    return st["period"], ex, st["carry"]


def run(args) -> dict:
    res_dir = os.path.join(args.results_root, os.path.basename(args.dataset.rstrip("/")) + "-" + args.save_dir)
    os.makedirs(res_dir, exist_ok=True)
    ckpt_path = os.path.join(res_dir, CKPT_NAME)
    resuming = bool(getattr(args, "resume", False)) and os.path.exists(ckpt_path)
    # data parallel (SURVEY 8e): one process per GPU under torchrun; rank 0 owns the log and the checkpoint
    args.dp_rank, args.dp_world = 0, 1
    if getattr(args, "dp", False) and int(os.environ.get("WORLD_SIZE", "1")) > 1:
        import torch.distributed as dist
        args.device_num = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(args.device_num)
        if not dist.is_initialized():
            dist.init_process_group("nccl", device_id=torch.device("cuda", args.device_num))
        args.dp_rank, args.dp_world = dist.get_rank(), dist.get_world_size()
    lead = args.dp_rank == 0
    logs = open(os.path.join(res_dir, "Training_logs.txt") if lead else os.devnull, mode="a" if resuming else "w")
    if not resuming:
        logs.write("\n".join([str(k) + "," + str(v) for k, v in sorted(vars(args).items(), key=lambda x: x[0])]))

    torch.cuda.set_device(args.device_num)
    np.random.seed(args.random_seed)                           # main.py:123-125
    random.seed(args.random_seed)

    dataloader = DataLoader(args.dataset, args.data_root, cache_dir=getattr(args, "cache_dir", None))
    item_num = args.item_num or ITEM_NUM.get(os.path.basename(args.dataset.rstrip("/")))
    if not item_num:
        raise ValueError("Invalid dataset name")
    args.dropout_rate = 0 if (args.ewc or args.finetune) else args.dropout_rate      # main.py:141
    model = Ader(item_num, args) if not args.ewc else Ewc(item_num, args)
    dp = None
    if args.dp_world > 1:
        from .dist import make_comm
        model.dp = make_comm(model)
        dp = (args.dp_rank, args.dp_world)
        info = "Data parallel: %d ranks, gradient back end %s" % (args.dp_world, model.dp.kind)
        print(info) if lead else None
        logs.write("\n" + info + "\n")

    periods = get_periods(dataloader.path)
    if args.max_periods:
        periods = periods[:args.max_periods]
    print("Continue Learning: number of periods is %d." % len(periods))
    logs.write("Continue Learning: number of periods is %d.\n" % len(periods))
    best_epoch, item_num_prev = 0, 0
    t_start = time.time()
    metrics = {"MRR_20": [], "Recall_20": [], "MRR_10": [], "Recall_10": []}
    stats = []
    fast_exemplar = None
    ckpt = {}                                                  # (period, epoch) -> state (tf.train.Saver max_to_keep=1)
    stop_counter = 0                                           # reference leaves it uninitialised (SURVEY S15)
    trace = {"periods": []} if getattr(args, "trace", False) else None
    no_replay = args.finetune or args.dropout or args.joint

    done_period = 0
    if resuming:                                               # SURVEY 8(f)1: continue after the last finished period
        done_period, fast_exemplar, carry = load_period_checkpoint(ckpt_path, model, dataloader, args.maxlen, args)
        best_epoch, item_num_prev, stop_counter = carry["best_epoch"], carry["item_num_prev"], carry["stop_counter"]
        metrics, stats = carry["metrics"], carry["stats"]
        ckpt = {(done_period, best_epoch): model.state_dict()}
        info = "Resumed after period %d from %s" % (done_period, ckpt_path)
        print(info)
        logs.write(info + "\n")

    for period in periods:
        if period <= done_period:
            continue
        print("Period %d:" % period)
        logs.write("Period %d:\n" % period)
        best_performance, performance = 0, 0
        train_sess, info = dataloader.train_loader(period - 1)
        logs.write(info + "\n")
        if args.joint and period > 1:
            for p in range(1, period):
                pre, info = dataloader.train_loader(p - 1)
                logs.write(info + "\n")
                train_sess.extend(pre)
        train_sampler = Sampler(train_sess, args.maxlen, args.batch_size)
        valid_subseq, train_subseq = train_sampler.split_data(valid_portion=0.1, return_train=True)
        batch_num = train_sampler.batch_num()
        test_sess, info = dataloader.evaluate_loader(period)
        logs.write(info + "\n")
        max_item = dataloader.max_item()

        exemplar_sampler = None
        exemplar_subseq = []
        if period > 1 and not no_replay:                       # main.py:181-191
            exemplar_size = len(fast_exemplar)
            exemplar_subseq = list(fast_exemplar.sessions)
            exemplar_batch = int(exemplar_size / batch_num)
            exemplar_sampler = Sampler([], args.maxlen, exemplar_batch)
            exemplar_sampler.add_exemplar(fast_exemplar)
            if args.ewc or args.fix_lambda:                    # main.py:194-203
                lambda_ = args.lambda_
            else:
                lambda_ = args.lambda_ * math.sqrt((item_num_prev / max_item) * (exemplar_size / train_sampler.data_size()))
            model.update_loss(lambda_=lambda_)
        else:
            model.set_vanilla_loss()

        if period > 1 and not args.joint:                      # main.py:210-213
            model.load_state_dict(ckpt[(period - 1, best_epoch)])
        else:
            model.reinitialize()

        use_ex = exemplar_sampler is not None and not args.ewc
        trainer = PeriodTrainer(model, train_sampler, exemplar_sampler if use_ex else None, args, max_item)
        rec = {"losses": [], "valid": [], "best_epoch": None, "test": None, "exemplars": None}
        if trace is not None:
            trainer.trace = rec["losses"]
            if getattr(args, "trace_rows", False):
                rec["rows"] = []
                trainer.trace_rows = rec["rows"]
            trace["periods"].append(rec)
        best_epoch = 1
        train_time = 0.0
        eval_time, eval_rows = 0.0, 0
        valid_cache = {}                   # packed validation rows + device copies, shared by the per-epoch Evaluators
        epoch_s, epoch_rows = [], []
        for epoch in range(1, args.num_epochs + 1):
            rows0 = trainer.rows_seen
            torch.cuda.synchronize()
            t0 = time.time()
            # the host holds millions of small Python objects (session lists): a generation-2 collection in the middle of
            # the batch loop stalls the launch thread for 0.1-0.5 s while the GPU idles -- collect between epochs instead
            gc_on = gc.isenabled()
            gc.disable()
            try:
                if trainer.trace is None and trainer.can_queue() and getattr(args, "epoch_queue", True):
                    trainer.run_epoch(batch_num)
                else:
                    for _ in range(batch_num):
                        trainer.step()
            finally:
                if gc_on:
                    gc.enable()
            torch.cuda.synchronize()
            train_time += time.time() - t0
            epoch_s.append(time.time() - t0)
            epoch_rows.append(trainer.rows_seen - rows0)
            if model.token_overflow():                          # a step was given a token capacity below its real token count
                raise ops._lib.AderError("period %d epoch %d: encoder token capacity overflow (tokens were dropped)" % (period, epoch))
            if period > 1 and args.ewc:                        # main.py:258-262 (no effect on train_op, S13)
                model.variables_prev = model.snapshot_variables()
                rnd = random.sample(exemplar_subseq, min(len(exemplar_subseq), args.ewc_sample_num))
                model.compute_fisher(None, rnd, 50, max_item)
            valid_evaluator = Evaluator(valid_subseq, True, args.maxlen, args.test_batch, max_item, "valid", model, None, dp=dp,
                                        cache=valid_cache)
            t0 = time.time()
            info = valid_evaluator.evaluate(epoch)
            eval_time += time.time() - t0                         # evaluate() ends with the ranks on the host
            eval_rows += len(valid_evaluator.ranks)
            logs.write(info + "\n")
            performance = valid_evaluator.results()[1]
            rec["valid"].append(valid_evaluator.results())
            if best_performance >= performance:                # main.py:272-280
                stop_counter += 1
                if stop_counter >= args.stop:
                    break
            else:
                stop_counter = 0
                best_epoch = epoch
                best_performance = performance
                ckpt = {(period, epoch): model.state_dict()}
        model.load_state_dict(ckpt[(period, best_epoch)])      # main.py:283
        test_evaluator = Evaluator(test_sess, False, args.maxlen, args.test_batch, max_item, "test", model, None, dp=dp)
        t0 = time.time()
        info = test_evaluator.evaluate(best_epoch)
        eval_time += time.time() - t0
        eval_rows += len(test_evaluator.ranks)
        logs.write(info + "\n")
        r = test_evaluator.results()
        rec["best_epoch"], rec["test"], rec["test_ranks"] = best_epoch, r, list(test_evaluator.ranks)
        metrics["MRR_20"].append(r[0]); metrics["Recall_20"].append(r[1])
        metrics["MRR_10"].append(r[2]); metrics["Recall_10"].append(r[3])
        sps = trainer.rows_seen / max(train_time, 1e-9)
        stats.append({"period": period, "train_rows": trainer.rows_seen, "train_s": train_time, "sessions_per_s": sps,
                      "eval_rows": eval_rows, "eval_s": eval_time, "eval_rows_per_s": eval_rows / max(eval_time, 1e-9),
                      "epochs": epoch, "max_item": int(max_item), "eager_steps": trainer.n_eager,
                      "epoch_s": epoch_s, "epoch_rows": epoch_rows, "host_plan_s": trainer.host_s["plan"], "host_launch_s": trainer.host_s["launch"],
                      # epochs after the first: the CUDA graphs of the period's batch geometries exist by then
                      "steady_sessions_per_s": (sum(epoch_rows[1:]) / max(sum(epoch_s[1:]), 1e-9)) if len(epoch_s) > 1 else None})
        info = "Period %d train throughput: %.0f sessions/s (%d rows in %.2f s; graph replays by batch geometry / token capacity %s, eager steps %d)" % (
            period, sps, trainer.rows_seen, train_time, trainer.graph_use(), trainer.n_eager)
        print(info)
        logs.write(info + "\n")

        if not no_replay:                                      # main.py:294-313
            cand = train_subseq
            cand.extend(valid_subseq)
            cand.extend(exemplar_subseq)
            # the frozen teacher stands in for the distillation logits only: one-hot replay / EWC runs keep the stored form
            form = "frozen" if getattr(args, "teacher", "logits") == "frozen" and not (args.disable_distillation or args.ewc) else "logits"
            gen = ExemplarGenerator(cand, args.exemplar_size, args.equal_exemplar, args.batch_size, args.maxlen,
                                    args.dropout_rate, max_item, teacher=form)
            if args.selection == "herding":
                saved = gen.herding_selection(None, model)
            elif args.selection == "loss":
                saved = gen.loss_selection(None, model)
            elif args.selection == "random":
                saved = gen.randomly_selection(None, model)
            else:
                print("Invalid exemplar selection method")
                saved = 0
            info = "Total saved exemplar: %d" % saved
            print(info)
            logs.write(info + "\n")
            fast_exemplar = gen.exemplars
            rec["exemplars"] = list(fast_exemplar.sessions)
            if trace is not None and args.selection == "herding":
                rec["herding"] = {"reps": gen.last_reps.cpu().numpy(), "cand": gen.cand, "seg_off": gen.seg_off,
                                  "items": gen.items, "quota": gen.last_quota, "picks": gen.last_picks}
            if trace is not None:
                rec["ex_by_item"] = {int(k): [gen.rows[r][-(args.maxlen + 1):] for r in v] for k, v in fast_exemplar.by_item.items()}
            del gen
        item_num_prev = max_item
        if args.ewc:                                           # main.py:319-323
            exemplar_subseq = list(fast_exemplar.sessions)
            model.variables_prev = model.snapshot_variables()
            rnd = random.sample(exemplar_subseq, min(len(exemplar_subseq), args.ewc_sample_num))
            model.compute_fisher(None, rnd, 50, max_item)
        if getattr(args, "checkpoint", True) and lead:
            save_period_checkpoint(ckpt_path, period, model, dataloader, fast_exemplar,
                                   {"best_epoch": best_epoch, "item_num_prev": item_num_prev, "stop_counter": stop_counter,
                                    "metrics": metrics, "stats": stats}, args)
        logs.flush()

    avg = {k: float(np.array(v).mean()) for k, v in metrics.items()}
    info = "Average: (MRR@20: %.4f, RECALL@20: %.4f, MRR@10: %.4f, RECALL@10: %.4f)" % (
        avg["MRR_20"], avg["Recall_20"], avg["MRR_10"], avg["Recall_10"])
    print(info)
    logs.write(info + "\n")
    minutes = (time.time() - t_start) / 60.0
    print("Total time: %.2f minutes." % minutes)
    logs.write("Total time: %.2f minutes\nDone." % minutes)
    logs.close()
    print("Done.")
    if model.dp is not None:
        torch.cuda.synchronize()
        model.dp.check()
    return {"average": avg, "per_period": metrics, "throughput": stats, "minutes": minutes, "trace": trace, "model": model}


def main(argv=None):
    args = build_parser().parse_args(argv)
    out = run(args)
    if args.dp_world > 1:
        # leave without tearing NCCL down: destroy_process_group() with live CUDA graphs that hold NCCL kernels can wedge
        import sys
        sys.stdout.flush(); sys.stderr.flush()
        os._exit(0)
    return out


if __name__ == "__main__":
    main()
