"""Host protocol of the ADER path: DataLoader, Sampler, Evaluator, ExemplarGenerator.

Same class / method names and the same `random` + `numpy.random` consumption order as the
reference's util.py (SURVEY A.5), so with equal seeds the batches, valid split, candidate order,
multinomial quotas and random picks are identical -- but rows are kept as packed int32 matrices
(GPU resident on demand), evaluation and exemplar selection run as a few batched device calls
instead of one ``sess.run`` per 64 rows / per item, and teacher logits stay on the device as one
``[E, V]`` fp32 matrix instead of Python lists (SURVEY S11).
"""
from __future__ import annotations

import math
import os
import random
from collections import defaultdict
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import ops


# ---- util.py:17-107 ----------------------------------------------------------------------------
class DataLoader:
    def __init__(self, dataset: str, data_root: Optional[str] = None, cache_dir: Optional[str] = None):
        """`dataset` is a name under `data_root` (reference: '../../data/<dataset>', util.py:28)
        or a directory that directly holds period_<k>.txt files."""
        if data_root is None:
            data_root = os.environ.get("ADER_DATA_ROOT", os.path.join("..", "..", "data"))
        self.path = os.path.join(data_root, dataset)
        if not os.path.isdir(self.path) and os.path.isdir(dataset):
            self.path = dataset
        self.item_set = set()                                   # util.py:26
        # SURVEY 8(f)3: every period file is parsed once into a binary (session id, item id) pair file and grouped with
        # array operations afterwards.  cache_dir=None (ADER_CACHE_DIR unset) keeps everything in memory.
        self.cache_dir = cache_dir if cache_dir is not None else os.environ.get("ADER_CACHE_DIR")
        self._pairs: Dict[int, Tuple[np.ndarray, np.ndarray]] = {}

    # ---- period file -> (session ids, item ids) arrays, cached -------------------------------------
    def _cache_file(self, period: int) -> Optional[str]:
        if not self.cache_dir:
            return None
        tag = os.path.basename(os.path.normpath(self.path)) or "data"
        return os.path.join(self.cache_dir, "%s.period_%d.pairs.npy" % (tag, period))

    def _read(self, period: int) -> Tuple[np.ndarray, np.ndarray]:
        """The "<session> <item>" lines of period_<k>.txt (util.py:36-40) as two int64 arrays in file order."""
        if period in self._pairs:
            return self._pairs[period]
        src = os.path.join(self.path, "period_%d.txt" % period)
        st = os.stat(src)
        cf = self._cache_file(period)
        pairs = None
        if cf and os.path.exists(cf):
            try:
                arr = np.load(cf)
                # header row = (source size, source mtime in ns): a changed source file invalidates the cache
                if arr.ndim == 2 and arr.shape[1] == 2 and arr[0, 0] == st.st_size and arr[0, 1] == st.st_mtime_ns:
                    pairs = arr[1:]
            except Exception:
                pairs = None
        if pairs is None:
            with open(src, "rb") as f:
                flat = np.array(f.read().split(), dtype=np.int64)
            if flat.size % 2:
                raise ValueError("%s: expected '<session> <item>' pairs" % src)
            pairs = flat.reshape(-1, 2)
            if cf:
                os.makedirs(self.cache_dir, exist_ok=True)
                tmp = cf + ".%d.tmp.npy" % os.getpid()
                np.save(tmp, np.concatenate([np.array([[st.st_size, st.st_mtime_ns]], dtype=np.int64), pairs]))
                os.replace(tmp, cf)
        out = (np.ascontiguousarray(pairs[:, 0]), np.ascontiguousarray(pairs[:, 1]))
        self._pairs[period] = out
        return out

    @staticmethod
    def _group(sess: np.ndarray, item: np.ndarray) -> List[List[int]]:
        """dict-of-lists grouping of the reference (util.py:41-48): sessions in order of first appearance, items of a
        session in file order -- as one stable sort instead of a Python loop over every line."""
        if sess.size == 0:
            return []
        order = np.argsort(sess, kind="stable")
        ss = sess[order]
        starts = np.flatnonzero(np.concatenate([[True], ss[1:] != ss[:-1]]))
        ends = np.concatenate([starts[1:], [ss.size]])
        first = order[starts]                                   # file position of each session's first line
        items_sorted = item[order].tolist()
        return [items_sorted[starts[g]:ends[g]] for g in np.argsort(first, kind="stable")]

    def train_loader(self, period: int) -> Tuple[List[List[int]], str]:        # util.py:32-58
        sess, item = self._read(period)
        self.item_set.update(np.unique(item).tolist())
        info = "Train set information: total number of action: %d." % sess.size
        print(info)
        return self._group(sess, item), info

    def evaluate_loader(self, period: int) -> Tuple[List[List[int]], str]:     # util.py:60-102
        sess, item = self._read(period)
        total = int(sess.size)
        known = np.fromiter(self.item_set, dtype=np.int64, count=len(self.item_set))
        keep = np.isin(item, known)
        removed = total - int(keep.sum())
        groups = self._group(sess[keep], item[keep])
        kept = [g for g in groups if len(g) > 1]
        removed += len(groups) - len(kept)
        info = "Test set information: original total number of action: %d, removed number of action: %d." % (total, removed)
        print(info)
        return kept, info

    def max_item(self) -> int:                                                 # util.py:104-107
        return max(self.item_set)


# ---- util.py:110-273 ---------------------------------------------------------------------------
def pack_rows(rows: Sequence[Sequence[int]], maxlen: int):
    """label_generator (util.py:151-171) for every row at once: ids [N, maxlen] int32 (last
    <= maxlen items before the label, right-aligned), label [N], n_in [N] (0 for rows of length <= 1)."""
    n = len(rows)
    ids = np.zeros((n, maxlen), np.int32)
    label = np.zeros(n, np.int32)
    n_in = np.zeros(n, np.int32)
    for r, s in enumerate(rows):
        k = len(s)
        if k == 0:
            continue
        label[r] = s[-1]
        body = s[:-1][-maxlen:]
        if body:
            ids[r, maxlen - len(body):] = body
            n_in[r] = len(body)
    return ids, label, n_in


class Sampler:
    def __init__(self, data: list, maxlen: int, batch_size: int, is_subseq: bool = False):
        self.maxlen, self.batch_size = maxlen, batch_size
        self.batch_counter = 0
        self.logits: list = []
        self.prepared_data: List[List[int]] = []
        if not is_subseq:                                                       # util.py:136-143
            for session in data:
                self.prepared_data.append(session)
                for t in range(1, len(session) - 1):
                    self.prepared_data.append(session[:-t])
        else:
            self.prepared_data = list(data)
        self._invalidate()
        self.data_indices = list(range(len(self.prepared_data)))
        random.shuffle(self.data_indices)                                       # util.py:148-149

    def _invalidate(self):
        self._packed = None
        self._dev = None

    # -- packed views -----------------------------------------------------------------------------
    def packed(self):
        if self._packed is None:
            self._packed = pack_rows(self.prepared_data, self.maxlen)
        return self._packed

    def device_rows(self, device):
        """GPU-resident (ids [N, L] int32, label [N] int32) of all prepared rows."""
        if self._dev is None or self._dev[0].device != torch.device(device):
            ids, label, _ = self.packed()
            self._dev = (torch.from_numpy(ids).to(device), torch.from_numpy(label).to(device))
        return self._dev

    # -- reference API ----------------------------------------------------------------------------
    def add_exemplar(self, exemplar) -> None:                                   # util.py:173-186
        """`exemplar` is the reference's list of [session, logits] or an ExemplarSet."""
        self.logits = []
        if isinstance(exemplar, ExemplarSet):
            self.prepared_data.extend(exemplar.sessions)
            self.logits = list(range(len(exemplar.sessions)))                   # row ids into exemplar.teacher
            self.teacher = exemplar.teacher
        else:
            for session, logits in exemplar:
                self.prepared_data.append(session)
                self.logits.append(logits)
            self.teacher = None
        self._invalidate()
        self.data_indices = list(range(len(self.prepared_data)))
        random.shuffle(self.data_indices)

    def split_data(self, valid_portion: float, return_train: bool = False):    # util.py:188-216
        n = len(self.prepared_data)
        sidx = np.arange(n, dtype="int32")
        np.random.shuffle(sidx)
        n_train = int(np.round(n * (1.0 - valid_portion)))
        valid = [self.prepared_data[s] for s in sidx[n_train:]]
        train = [self.prepared_data[s] for s in sidx[:n_train]]
        self.prepared_data = train
        self._invalidate()
        self.data_indices = list(range(len(self.prepared_data)))
        random.shuffle(self.data_indices)
        return (valid, train) if return_train else valid

    def data_size(self) -> int:
        return len(self.prepared_data)

    def batch_num(self) -> int:
        return math.ceil(len(self.prepared_data) * 1.0 / self.batch_size)

    def next_indices(self) -> np.ndarray:
        """Row indices of the next batch (rows of length <= 1 skipped, util.py:228-229); advances
        the cursor and reshuffles at wrap exactly like sampler() (util.py:233-237)."""
        _, _, n_in = self.packed()
        lo = self.batch_counter * self.batch_size
        idx = np.asarray(self.data_indices[lo:lo + self.batch_size], dtype=np.int64)
        idx = idx[n_in[idx] > 0] if idx.size else idx
        self.batch_counter += 1
        if self.batch_counter == self.batch_num():
            self.batch_counter = 0
            random.shuffle(self.data_indices)
        return idx

    def sampler_arrays(self):
        """One batch as arrays: (ids [B, L] int32, label [B] int32)."""
        ids, label, _ = self.packed()
        idx = self.next_indices()
        return ids[idx], label[idx]

    def sampler(self):                                                          # util.py:218-239
        seq, pos = self.sampler_arrays()
        return tuple(seq), tuple(pos)

    def exemplar_sampler(self):                                                 # util.py:241-263
        ids, label, _ = self.packed()
        idx = self.next_indices()
        return tuple(ids[idx]), tuple(label[idx]), [self.logits[i] for i in idx]

    def epoch_order(self, defer_shuffle: bool = False) -> np.ndarray:
        """All row indices of one full pass in batch order (rows of length <= 1 dropped); consumes
        the wrap reshuffle like batch_num() calls to sampler() would.  Cursor must be at 0.
        defer_shuffle: the caller runs ``finish_epoch_order()`` itself (same RNG draws, later in wall time: the
        Python-level shuffle of a 50 000-row list takes ~25 ms, which an evaluation pass hides behind its GPU work)."""
        assert self.batch_counter == 0
        _, _, n_in = self.packed()
        idx = np.asarray(self.data_indices, dtype=np.int64)
        idx = idx[n_in[idx] > 0] if idx.size else idx
        if not defer_shuffle:
            self.finish_epoch_order()
        return idx

    def finish_epoch_order(self):
        if self.batch_num() > 0:
            random.shuffle(self.data_indices)


# ---- exemplar store ------------------------------------------------------------------------------
class FrozenTeacher:
    """The distillation teacher as a frozen snapshot of the model that selected the exemplars: every stored logit row is
    rep_prev(session) . E_prev[1..V_prev]^T, so the exemplar reps and a copy of the item table carry the same information
    as the [E, V_prev] logit matrix in O(E*d + V_prev*d) bytes.  The loss kernels recompute the teacher logits per step.

    rep [E, d] fp32 (exact encoder, at selection time); table [V_prev, d] fp32 = rows 1..V_prev of the table (a copy, never a
    view of the live parameters); table16 = its bf16 operand shadow for the tcgen05 kernels (ops.pack_table16); width = V_prev."""

    def __init__(self, model, rep: torch.Tensor, width: int):
        d = model.hp.hidden_units
        self.ms, self.width = model.ms, int(width)
        self.rep = rep.detach().to(torch.float32).contiguous()
        # rows 0..V_prev of the table in one buffer: `table` (rows 1..V_prev) is a view of this copy, and the whole buffer has
        # the layout of a parameter vector's table, so ops.logits can materialise the teacher rows from it (logits()).
        self._rows = model.theta[:(self.width + 1) * d].clone()
        self.table = self._rows[d:].view(self.width, d)
        self.table16 = None
        if d <= 160:
            self.table16 = torch.empty(ops.table16_bytes(model.ms, self.width), dtype=torch.uint8, device=model.device)
            ops.pack_table16(model.ms, self.table, self.width, self.table16)

    def __len__(self):
        return self.rep.shape[0]

    def nbytes(self) -> int:
        return sum(t.numel() * t.element_size() for t in (self.rep, self._rows, self.table16) if t is not None)

    def logits(self, rows: Optional[torch.Tensor] = None) -> torch.Tensor:
        """The stored-logit matrix this snapshot stands for, [len(rows) or E, V_prev] fp32 (bit-identical to what the
        previous model's ``logits`` gave at selection time).  O(E * V_prev) memory: small sizes and tests only."""
        r = self.rep if rows is None else self.rep.index_select(0, rows.to(self.rep.device, torch.int64))
        ld = (self.width + 3) // 4 * 4
        out = torch.empty((r.shape[0], ld), dtype=torch.float32, device=self.rep.device)[:, :self.width]
        if r.shape[0]:
            ops.logits(self.ms, self._rows, r.contiguous(), self.width, out)
        return out


class ExemplarSet:
    """Flattened exemplars of one period: sessions in the order main.py:54-65 (`load_exemplars`)
    would yield them, and their teacher: stored logits as ONE device matrix [E, V] fp32 (SURVEY S11), or a
    ``FrozenTeacher`` snapshot of the selecting model."""

    def __init__(self, sessions: List[List[int]], teacher, by_item: Optional[dict] = None):
        self.sessions = sessions
        self.teacher = teacher
        self.by_item = by_item or {}

    def __len__(self):
        return len(self.sessions)

    def as_reference_list(self):
        """[[session, logits_list], ...] exactly like load_exemplars (small sizes only)."""
        t = (self.teacher.logits() if isinstance(self.teacher, FrozenTeacher) else self.teacher).cpu().numpy()
        return [[s, t[i].tolist()] for i, s in enumerate(self.sessions)]


def load_exemplars(exemplar_pre) -> "ExemplarSet":                               # main.py:54-65
    if isinstance(exemplar_pre, ExemplarSet):
        return exemplar_pre
    out = []
    for item in exemplar_pre.values():
        if isinstance(item, list):
            out.extend([i for i in item if i])
    return out


# ---- util.py:276-350 -----------------------------------------------------------------------------
class Evaluator:
    def __init__(self, data: list, is_subseq: bool, maxlen: int, batch_size: int, max_item: int, mode: str,
                 model, sess=None, chunk_rows: int = 8192, dp=None, cache: Optional[dict] = None):
        """cache: a dict the caller keeps for as long as `data` is unchanged (main.py builds a new Evaluator over the SAME
        validation rows after every epoch, main.py:263): the packed row matrices and their device copies are stored in it
        by the first Evaluator and reused by the next ones (the Sampler itself is rebuilt every time: its constructor
        draws from `random`, util.py:148-149)."""
        self.max_item, self.model, self.mode = max_item, model, mode
        self.cache = cache
        self.dp = dp                      # (rank, world): rows of a pass are sharded over the ranks, ranks all-gathered
        self.ranks: List[int] = []
        self.desc = "Validating epoch " if mode == "valid" else "Testing epoch "
        self.evaluate_sampler = Sampler(data, maxlen, batch_size, is_subseq=is_subseq)
        self.chunk_rows = chunk_rows
        self.topk = None
        self._rows_dev = None
        if cache is not None and cache.get("n") == len(self.evaluate_sampler.prepared_data):
            self.evaluate_sampler._packed = cache["packed"]
            self._rows_dev = cache["dev"]

    def evaluate(self, epoch: int, k: int = 0) -> str:                           # util.py:309-327
        """All rows of one pass are ranked on the device in a few large calls.  The rank list is in
        the reference's batch order; the sampler's RNG is consumed as batch_num() sampler() calls.
        k > 0 additionally keeps the top-k item ids per row in ``self.topk`` (the metrics only need ranks)."""
        s = self.evaluate_sampler
        order = s.epoch_order(defer_shuffle=True)
        ids, label, n_in = s.packed()
        ranks = []
        tops = []
        n_all = len(order)
        if self.dp is not None and self.dp[1] > 1:          # SURVEY 8e: evaluation rows are independent -> shard them
            from .dist import shard_range
            lo_r, hi_r = shard_range(n_all, self.dp[0], self.dp[1])
            order = order[lo_r:hi_r]
        # the rows of the pass live on the device (uploaded once per Evaluator: every epoch ranks the same rows in a new
        # order); a chunk is a device gather by the order indices, the host only launches
        dev = self.model.device
        if self._rows_dev is None:
            self._rows_dev = (torch.from_numpy(np.ascontiguousarray(ids)).to(dev), torch.from_numpy(np.ascontiguousarray(label)).to(dev))
        ids_d, label_d = self._rows_dev
        if self.cache is not None:
            self.cache.update(n=len(s.prepared_data), packed=s.packed(), dev=self._rows_dev)
        order_d = torch.from_numpy(order).to(dev)
        guards, spans = [], []
        for lo in range(0, len(order), self.chunk_rows):
            idx = order[lo:lo + self.chunk_rows]
            idx_d = order_d[lo:lo + self.chunk_rows]
            r, items, _ = self.model.rank_topk(ids_d.index_select(0, idx_d), label_d.index_select(0, idx_d), self.max_item, k,
                                               n_tokens=int(n_in[idx].sum()), guards=guards)
            ranks.append(r)
            tops.append(items)
            spans.append((lo, idx))
        s.finish_epoch_order()                               # the wrap reshuffle (same RNG draws), behind the launches
        for i in self.model.check_guards(guards):            # a candidate band overflowed: that chunk again, exact path
            lo, idx = spans[i]
            idx_d = order_d[lo:lo + self.chunk_rows]
            ranks[i], tops[i], _ = self.model.rank_topk(ids_d.index_select(0, idx_d), label_d.index_select(0, idx_d), self.max_item, k,
                                                       n_tokens=int(n_in[idx].sum()), force_exact=True)
        if self.dp is not None and self.dp[1] > 1:
            import torch.distributed as dist
            from .dist import shard_range
            world = self.dp[1]
            sizes = [shard_range(n_all, r, world)[1] - shard_range(n_all, r, world)[0] for r in range(world)]
            cap = max(max(sizes), 1)
            dev = self.model.device
            mine = torch.full((cap,), -1, dtype=torch.int32, device=dev)
            if ranks:
                r_loc = torch.cat(ranks)
                mine[:r_loc.numel()] = r_loc
            parts = [torch.empty_like(mine) for _ in range(world)]
            dist.all_gather(parts, mine)
            ranks = [p[:n] for p, n in zip(parts, sizes)]
            if k > 0:
                mine_t = torch.zeros((cap, k), dtype=torch.int32, device=dev)
                if tops:
                    t_loc = torch.cat(tops)
                    mine_t[:t_loc.shape[0]] = t_loc
                parts_t = [torch.empty_like(mine_t) for _ in range(world)]
                dist.all_gather(parts_t, mine_t)
                tops = [p[:n] for p, n in zip(parts_t, sizes)]
        if ranks and n_all > 0:
            self.ranks = torch.cat(ranks).cpu().numpy().tolist()
            self.topk = torch.cat(tops) if k > 0 else None
        else:
            self.ranks = []
        return self.display(epoch)

    def results(self):                                                           # util.py:329-339
        n = len(self.ranks)
        r = np.asarray(self.ranks, dtype=np.int64)
        r20, r10 = r[r < 20], r[r < 10]
        mrr20 = float(np.sum(1.0 / (r20 + 1)))
        mrr10 = float(np.sum(1.0 / (r10 + 1)))
        return mrr20 / n, len(r20) / n, mrr10 / n, len(r10) / n

    def display(self, epoch) -> str:                                             # util.py:341-350
        res = self.results()
        info = "epoch:%d, %s (MRR@20: %.4f, RECALL@20: %.4f, MRR@10: %.4f, RECALL@10: %.4f)" % (
            epoch, self.mode, res[0], res[1], res[2], res[3])
        print(info)
        return info


# ---- util.py:353-522 -----------------------------------------------------------------------------
class ExemplarGenerator:
    def __init__(self, data: list, exemplar_size: int, disable_m: bool, batch_size: int, maxlen: int,
                 dropout_rate: float, max_item: int, chunk_rows: int = 16384, teacher: str = "logits"):
        """teacher: "logits" keeps the [E, max_item] teacher logits of the exemplars, "frozen" a FrozenTeacher snapshot."""
        if teacher not in ("logits", "frozen"):
            raise ValueError("teacher must be 'logits' or 'frozen', got %r" % (teacher,))
        self.teacher_form = teacher
        self.m, self.max_item, self.maxlen = exemplar_size, max_item, maxlen
        self.dropout_rate = dropout_rate
        self.chunk_rows = chunk_rows
        sampler = Sampler(data, maxlen, batch_size, is_subseq=True)              # util.py:383
        order = sampler.epoch_order()                                            # encounter order + wrap shuffle
        ids, label, n_in = sampler.packed()
        self.ids, self.label, self.n_in = ids[order], label[order], n_in[order]  # candidate rows, encounter order
        self.rows = [sampler.prepared_data[i] for i in order]
        # group by label, groups in first-appearance order (dict insertion order of sess_by_item)
        lab = self.label.astype(np.int64)
        first = {}
        for pos_, it in enumerate(lab.tolist()):
            if it not in first:
                first[it] = len(first)
        gid = np.fromiter((first[it] for it in lab.tolist()), dtype=np.int64, count=len(lab))
        self.items = np.fromiter(first.keys(), dtype=np.int64, count=len(first))  # label of each group
        srt = np.argsort(gid, kind="stable")
        self.cand = srt.astype(np.int32)                                          # candidate row per slot
        counts = np.bincount(gid, minlength=len(first))
        self.seg_off = np.zeros(len(first) + 1, np.int32)
        np.cumsum(counts, out=self.seg_off[1:])
        item_count = np.zeros(max_item)
        np.add.at(item_count, lab - 1, 1)                                         # util.py:393
        if disable_m:
            item_count = np.ones_like(item_count)                                 # util.py:395-396
        prob = item_count / item_count.sum()
        self.item_count = np.int32(np.random.multinomial(n=self.m, pvals=prob, size=1)[0])   # util.py:398-399
        self.exemplars = None

    # sess_by_item view for drop-in users (small sizes)
    @property
    def sess_by_item(self):
        out = defaultdict(list)
        for g, it in enumerate(self.items.tolist()):
            for c in self.cand[self.seg_off[g]:self.seg_off[g + 1]]:
                out[it].append(np.append(self.ids[c], self.label[c]))
        return out

    def _all_reps(self, model) -> torch.Tensor:
        reps = []
        for lo in range(0, len(self.ids), self.chunk_rows):
            hi = min(len(self.ids), lo + self.chunk_rows)
            reps.append(model.rep(self.ids[lo:hi], n_tokens=int(self.n_in[lo:hi].sum())).clone())
        return torch.cat(reps) if reps else torch.zeros((0, model.hp.hidden_units), device=model.device)

    def _store(self, model, picked_rows: np.ndarray, reps: Optional[torch.Tensor], by_item=None) -> int:
        """Keep sessions (non-zero entries of [input, label], util.py:433) and their logits rows (or, in the frozen form,
        their reps and a snapshot of the table: no [E, max_item] matrix is built)."""
        sessions = [self.rows[r][-(self.maxlen + 1):] for r in picked_rows.tolist()]
        dev = model.device
        if len(picked_rows):
            idx = torch.from_numpy(picked_rows.astype(np.int64)).to(dev)
            r = reps[idx] if reps is not None else model.rep(self.ids[picked_rows], n_tokens=int(self.n_in[picked_rows].sum()))
            teacher = (FrozenTeacher(model, r, self.max_item) if self.teacher_form == "frozen"
                       else model.logits(r.contiguous(), self.max_item))
        elif self.teacher_form == "frozen":
            teacher = FrozenTeacher(model, torch.zeros((0, model.hp.hidden_units), device=dev), self.max_item)
        else:
            teacher = torch.zeros((0, self.max_item), device=dev)
        self.exemplars = ExemplarSet(sessions, teacher, by_item)
        return len(sessions)

    def herding_selection(self, sess, model) -> int:                              # util.py:436-461
        dev = model.device
        reps = self._all_reps(model)
        n_seg = len(self.items)
        seg_n = np.diff(self.seg_off)
        quota = np.minimum(self.item_count[self.items - 1], seg_n).astype(np.int32)   # util.py:458
        max_steps = np.array([int(math.ceil(1.1 * int(m))) for m in quota], dtype=np.int32)   # util.py:425 (float64)
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        picks = torch.zeros(len(self.cand), dtype=torch.int32, device=dev)
        n_picked = torch.zeros(n_seg, dtype=torch.int32, device=dev)
        ws = torch.empty(ops.herding_ws_bytes(model.ms, len(self.cand)), dtype=torch.uint8, device=dev)
        ops.herding_segmented(model.ms, reps, t(self.cand), t(self.seg_off), t(quota), t(max_steps), ws, picks, n_picked)
        picks_h, n_h = picks.cpu().numpy(), n_picked.cpu().numpy()
        rows = []
        by_item = {}
        for g in range(n_seg):
            lo = self.seg_off[g]
            sel = self.cand[lo + picks_h[lo:lo + n_h[g]]]
            by_item[int(self.items[g])] = sel
            rows.append(sel)
        picked = np.concatenate(rows) if rows else np.zeros(0, np.int32)
        self.last_picks = (picks_h, n_h)
        self.last_reps, self.last_quota = reps, quota
        return self._store(model, picked, reps, by_item)

    def loss_selection(self, sess, model) -> int:                                 # util.py:463-492
        """As executed by the reference: ``model.loss`` is a scalar mean, so argsort()[:k] is [0] --
        at most ONE exemplar per item, candidate index 0 (SURVEY S9)."""
        rows = []
        by_item = {}
        for g, it in enumerate(self.items.tolist()):
            m = self.item_count[it - 1]
            if m < 0.5:
                continue
            lo, hi = self.seg_off[g], self.seg_off[g + 1]
            k = int(min(m, hi - lo))
            sel = self.cand[lo:lo + min(k, 1)]
            by_item[it] = sel
            rows.append(sel)
        picked = np.concatenate(rows) if rows else np.zeros(0, np.int32)
        return self._store(model, picked, None, by_item)

    def randomly_selection(self, sess, model) -> int:                             # util.py:494-522
        rows = []
        by_item = {}
        for g, it in enumerate(self.items.tolist()):
            lo, hi = self.seg_off[g], self.seg_off[g + 1]
            n = int(hi - lo)
            m = self.item_count[it - 1]
            if m > 0:
                sel_local = np.random.choice(n, min(m, n), replace=False)        # util.py:512
                sel = self.cand[lo + sel_local]
                by_item[it] = sel
                rows.append(sel)
        picked = np.concatenate(rows) if rows else np.zeros(0, np.int32)
        return self._store(model, picked, None, by_item)
