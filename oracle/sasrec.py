"""Torch-CPU restatement of the reference's TF1 graph (TEST INFRASTRUCTURE ONLY).

Every function cites the reference lines it follows (paths relative to /root/reference).
The computation is *dense over all maxlen slots*, materialises ``[M, V]`` logits and a
one-hot, exactly like the reference -- that is the point: it is the slow, literal version
that the packed / fused CUDA path is compared with.

Parity status: unpinned against TensorFlow (see oracle/__init__.py).
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np
import torch

NEG_PAD = float(-2 ** 32 + 1)  # modules.py:192, modules.py:201

# modules.py:188-193 / 208-211 derive the key and query masks from the ACTIVATIONS
# (sign|sum_d keys|, sign|sum_d queries|), not from the ids.  For real tokens that equals 1 except
# when the fp32 sum is EXACTLY zero.  With a fresh init (LN beta = 0, gamma = 1) the normalised
# queries sum to zero mathematically, so a few percent of real query rows hit an exact fp32 zero
# (which ones depends on the summation order of the BLAS/TF build) and get their attention output
# zeroed.  LITERAL_MASKS = True restates that behaviour; False uses the id-derived masks, i.e. the
# function the reference computes on every input where the sums are not exactly zero.  The CUDA path
# implements the latter (DESIGN.md section 4); parity tests that start from a fresh init switch this off.
LITERAL_MASKS = True


class literal_masks:
    """Context manager: ``with literal_masks(False): ...``"""

    def __init__(self, value: bool):
        self.value = value

    def __enter__(self):
        global LITERAL_MASKS
        self.prev, LITERAL_MASKS = LITERAL_MASKS, self.value

    def __exit__(self, *exc):
        global LITERAL_MASKS
        LITERAL_MASKS = self.prev


@dataclass
class Hyper:
    """Subset of main.py:75-108 flags that shape the network."""
    item_num: int            # main.py:133-138 (43136 / 25958); table has item_num+1 rows
    hidden_units: int = 150  # main.py:103
    maxlen: int = 50         # main.py:104
    num_blocks: int = 2      # main.py:99
    num_heads: int = 1       # main.py:100


# ----------------------------------------------------------------------------------------
# Parameters: creation order == Ewc.variables order (EWC.py:90, SURVEY A.2) -- 32 tensors
# for 2 blocks.  The flat layout [table | pos | block0 ... | final ln] is shared with the
# CUDA path (ader_b200/params.py restates the same table independently).
# ----------------------------------------------------------------------------------------
def param_shapes(hp: Hyper) -> List[tuple]:
    d = hp.hidden_units
    shapes = [("item_table", (hp.item_num + 1, d)),       # modules.py:118-122
              ("pos_table", (hp.maxlen, d))]              # ADER.py:41-51
    for b in range(hp.num_blocks):
        shapes += [(f"b{b}.ln1.beta", (d,)), (f"b{b}.ln1.gamma", (d,)),   # modules.py:45-46
                   (f"b{b}.wq", (d, d)), (f"b{b}.bq", (d,)),               # modules.py:172
                   (f"b{b}.wk", (d, d)), (f"b{b}.bk", (d,)),               # modules.py:173
                   (f"b{b}.wv", (d, d)), (f"b{b}.bv", (d,)),               # modules.py:174
                   (f"b{b}.ln2.beta", (d,)), (f"b{b}.ln2.gamma", (d,)),
                   (f"b{b}.w1", (d, d)), (f"b{b}.b1", (d,)),               # modules.py:254-256
                   (f"b{b}.w2", (d, d)), (f"b{b}.b2", (d,))]               # modules.py:259-261
    shapes += [("lnf.beta", (d,)), ("lnf.gamma", (d,))]                    # ADER.py:82
    return shapes


def init_params(hp: Hyper, seed: int = 0, dtype=torch.float32) -> List[torch.Tensor]:
    """Seeded Glorot-uniform init (TF get_variable / dense / conv1d default), zeros for
    biases and LN beta, ones for LN gamma (SURVEY A.2).  TF's own init stream cannot be
    reproduced outside TF; parity runs share THIS init between oracle and CUDA path."""
    rng = np.random.RandomState(seed)
    out = []
    for name, shape in param_shapes(hp):
        if name.endswith("gamma"):
            a = np.ones(shape, np.float64)
        elif len(shape) == 1:
            a = np.zeros(shape, np.float64)
        else:
            limit = math.sqrt(6.0 / (shape[0] + shape[1]))
            a = rng.uniform(-limit, limit, size=shape)
        out.append(torch.tensor(a.astype(np.float32)).to(dtype))
    return out


def randomize_params(params: Sequence[torch.Tensor], seed: int, scale: float = 0.05):
    """Perturb *every* tensor (incl. biases / LN affine) so parity tests exercise them."""
    rng = np.random.RandomState(seed)
    out = []
    for p in params:
        noise = torch.tensor(rng.standard_normal(tuple(p.shape)).astype(np.float32)).to(p.dtype)
        out.append(p + scale * noise)
    return out


# ----------------------------------------------------------------------------------------
# Layers
# ----------------------------------------------------------------------------------------
def normalize(x, beta, gamma, eps: float = 1e-8):
    """modules.py:44-48 -- population variance, eps inside the sqrt."""
    mean = x.mean(-1, keepdim=True)
    var = ((x - mean) ** 2).mean(-1, keepdim=True)
    return gamma * ((x - mean) / (var + eps) ** 0.5) + beta


def multihead_attention(q, keys, wq, bq, wk, bk, wv, bv, num_heads: int, id_mask=None, drop=None):
    """modules.py:172-223 with causality=True.  drop: None (dropout 0) or the [h*M, T, T] multipliers of the
    attention weights (modules.py:214; oracle/dropout.py draws the library's own)."""
    Q = q @ wq + bq                                                   # :172
    K = keys @ wk + bk                                                # :173
    V = keys @ wv + bv                                                # :174
    Q_ = torch.cat(torch.chunk(Q, num_heads, dim=2), dim=0)           # :177-179
    K_ = torch.cat(torch.chunk(K, num_heads, dim=2), dim=0)
    V_ = torch.cat(torch.chunk(V, num_heads, dim=2), dim=0)
    out = Q_ @ K_.transpose(1, 2)                                     # :182
    out = out / (K_.shape[-1] ** 0.5)                                 # :185
    literal = LITERAL_MASKS or id_mask is None
    key_masks = torch.sign(torch.abs(keys.sum(-1))) if literal else id_mask       # :188
    key_masks = key_masks.repeat(num_heads, 1)[:, None, :].expand_as(out)
    out = torch.where(key_masks == 0, torch.full_like(out, NEG_PAD), out)   # :192-193
    T = out.shape[1]
    tril = torch.tril(torch.ones(T, T, dtype=out.dtype))              # :197-199
    out = torch.where(tril[None] == 0, torch.full_like(out, NEG_PAD), out)  # :201-202
    out = torch.softmax(out, dim=-1)                                  # :205
    query_masks = (torch.sign(torch.abs(q.sum(-1))) if literal else id_mask).repeat(num_heads, 1)[:, :, None]  # :208-210
    out = out * query_masks                                           # :211
    if drop is not None:
        out = out * drop                                              # :214
    out = out @ V_                                                    # :217
    out = torch.cat(torch.chunk(out, num_heads, dim=0), dim=2)        # :220
    return out + q                                                    # :223 residual on queries


def feedforward(z, w1, b1, w2, b2, drop=None):
    """modules.py:254-266 -- conv1d(k=1) == dense; residual on the (normalised) input.  drop: None (dropout 0)
    or the (inner, output) multipliers, each [M, T, d] (modules.py:257, 262)."""
    if drop is None:
        return torch.relu(z @ w1 + b1) @ w2 + b2 + z
    return (torch.relu(z @ w1 + b1) * drop[0] @ w2 + b2) * drop[1] + z


def forward_rep(params: Sequence[torch.Tensor], ids: torch.Tensor, hp: Hyper, drop=None) -> torch.Tensor:
    """ADER.py:25-85: ids [M, maxlen] int -> rep [M, d].  drop: None (eval mode / dropout 0) or a dict site ->
    multipliers in the padded layout (oracle.dropout.dense_multipliers: the library's masks)."""
    d = hp.hidden_units
    table, pos_table = params[0], params[1]
    mask = (ids != 0).to(table.dtype)[..., None]                          # ADER.py:25
    e0 = torch.cat([torch.zeros(1, d, dtype=table.dtype), table[1:]], 0)  # modules.py:124-126
    seq = e0[ids.long()] * (d ** 0.5)                                     # modules.py:127-130
    seq = seq + pos_table[torch.arange(ids.shape[1])][None]               # ADER.py:41-52
    if drop is not None:
        drop = {k: torch.as_tensor(v).to(table.dtype) for k, v in drop.items()}
        seq = seq * drop[0]                                               # ADER.py:55-58
    seq = seq * mask                                                      # ADER.py:60
    for b in range(hp.num_blocks):
        (ln1b, ln1g, wq, bq, wk, bk, wv, bv, ln2b, ln2g, w1, b1, w2, b2) = params[2 + 14 * b: 16 + 14 * b]
        d_att, d_ffn = (None, None) if drop is None else (drop[1 + 3 * b], (drop[2 + 3 * b], drop[3 + 3 * b]))
        seq = multihead_attention(normalize(seq, ln1b, ln1g), seq, wq, bq, wk, bk, wv, bv,
                                  hp.num_heads, id_mask=mask[..., 0], drop=d_att)  # ADER.py:66-74
        seq = feedforward(normalize(seq, ln2b, ln2g), w1, b1, w2, b2, drop=d_ffn)  # ADER.py:77
        seq = seq * mask                                                  # ADER.py:80
    seq = normalize(seq, params[-2], params[-1])                          # ADER.py:82
    return seq[:, -1, :]                                                  # ADER.py:85


def logits_of(rep: torch.Tensor, table: torch.Tensor, max_item: int) -> torch.Tensor:
    """ADER.py:90-91: columns = items 1..max_item of the (row-0-zeroed, unscaled) table."""
    return rep @ table[1:max_item + 1].t()


def ce_rows(logits: torch.Tensor, pos: torch.Tensor) -> torch.Tensor:
    """ADER.py:88-92 softmax_cross_entropy_with_logits against one_hot(pos-1)."""
    lse = torch.logsumexp(logits, dim=1)
    return lse - logits.gather(1, (pos.long() - 1)[:, None])[:, 0]


def loss_vanilla(params, ids, pos, max_item: int, hp: Hyper, drop=None):
    """ADER.py:93 (set_vanilla_loss, ADER.py:105-106).  drop: see forward_rep."""
    rep = forward_rep(params, ids, hp, drop)
    return ce_rows(logits_of(rep, params[0], max_item), pos).mean()


def loss_ader(params, ids, pos, max_item: int, hp: Hyper, lambda_: float,
              exemplar_logits: Optional[torch.Tensor] = None,
              exemplar_pos: Optional[torch.Tensor] = None, drop=None):
    """ADER.py:108-138 (update_loss).  Exemplar rows are the LAST rows of ``ids``; ``pos``
    covers only the leading train rows.  KD branch: student softmax over the first V_prev
    columns only (ADER.py:134); ER branch: one-hot CE on the exemplar rows (ADER.py:126-131).  drop: see
    forward_rep."""
    rep = forward_rep(params, ids, hp, drop)
    logits = logits_of(rep, params[0], max_item)
    n_ex = exemplar_logits.shape[0] if exemplar_logits is not None else exemplar_pos.shape[0]
    n_train = ids.shape[0] - n_ex
    loss = ce_rows(logits[:n_train], pos).mean()                       # ADER.py:118-121
    ex = logits[n_train:]
    if exemplar_logits is None:
        loss = loss + lambda_ * ce_rows(ex, exemplar_pos).mean()       # ADER.py:126-131
    else:
        v_prev = exemplar_logits.shape[1]
        s = ex[:, :v_prev]                                             # ADER.py:134
        t = torch.softmax(exemplar_logits.to(s.dtype), dim=1)          # ADER.py:135 (no grad)
        kd = -(t * torch.log_softmax(s, dim=1)).sum(1)                 # ADER.py:136-137
        loss = loss + lambda_ * kd.mean()
    return loss


def loss_ewc(params, ids, pos, max_item: int, hp: Hyper, lambda_: float,
             fisher: Sequence[torch.Tensor], params_prev: Sequence[torch.Tensor]):
    """EWC.py:115-124: CE + (lambda/2) * sum_v sum(F_v * (theta_v - theta*_v)^2)."""
    loss = loss_vanilla(params, ids, pos, max_item, hp)
    for p, f, q in zip(params, fisher, params_prev):
        loss = loss + (lambda_ / 2.0) * (f.to(p.dtype) * (p - q.to(p.dtype)) ** 2).sum()
    return loss


def grads_of(loss_fn, params: Sequence[torch.Tensor]) -> List[torch.Tensor]:
    ps = [p.detach().clone().requires_grad_(True) for p in params]
    loss = loss_fn(ps)
    gs = torch.autograd.grad(loss, ps, allow_unused=True)
    return float(loss.detach()), [torch.zeros_like(p) if g is None else g for p, g in zip(ps, gs)]


# ----------------------------------------------------------------------------------------
# TF1 Adam (tf.train.AdamOptimizer; ADER.py:96, SURVEY A.3 / S10)
# ----------------------------------------------------------------------------------------
class AdamTF1:
    """theta -= lr * sqrt(1-b2^t)/(1-b1^t) * m / (sqrt(v) + eps); eps NOT bias-corrected.
    Dense update of every row every step (the item-table gradient is dense in the
    reference because it flows through concat/slice, modules.py:124-127)."""

    def __init__(self, params, beta1=0.9, beta2=0.999, eps=1e-8):
        self.m = [torch.zeros_like(p) for p in params]
        self.v = [torch.zeros_like(p) for p in params]
        self.t = 0
        self.beta1, self.beta2, self.eps = beta1, beta2, eps

    def step(self, params, grads, lr: float):
        self.t += 1
        b1, b2 = self.beta1, self.beta2
        lr_t = lr * math.sqrt(1.0 - b2 ** self.t) / (1.0 - b1 ** self.t)
        out = []
        for i, (p, g) in enumerate(zip(params, grads)):
            self.m[i] = b1 * self.m[i] + (1 - b1) * g
            self.v[i] = b2 * self.v[i] + (1 - b2) * g * g
            out.append(p - lr_t * self.m[i] / (self.v[i].sqrt() + self.eps))
        return out


# ----------------------------------------------------------------------------------------
# Evaluation (ADER.py:99-103, util.py:323-339)
# ----------------------------------------------------------------------------------------
def rank_of_gt(logits: np.ndarray, gt: np.ndarray) -> np.ndarray:
    """pred_last = argsort(argsort(-logits)) (ADER.py:103), then pred[gt-1] (util.py:325).
    tf.argsort is top_k based: equal scores keep the lower index first, i.e. a stable sort
    of the negated scores."""
    order = np.argsort(-logits, axis=1, kind="stable")
    ranks = np.argsort(order, axis=1, kind="stable")
    return ranks[np.arange(len(gt)), np.asarray(gt) - 1]


def topk_items(logits: np.ndarray, k: int = 20) -> np.ndarray:
    """Item ids (1-based) of the k best scores per row, ties toward the lower id."""
    order = np.argsort(-logits, axis=1, kind="stable")
    return order[:, :k] + 1


def metrics_from_ranks(ranks: Sequence[int]):
    """util.py:329-339 -> (MRR@20, RECALL@20, MRR@10, RECALL@10)."""
    n = len(ranks)
    r20 = [x for x in ranks if x < 20]
    r10 = [x for x in ranks if x < 10]
    return (sum(1.0 / (x + 1) for x in r20) / n, len(r20) / n,
            sum(1.0 / (x + 1) for x in r10) / n, len(r10) / n)


# ----------------------------------------------------------------------------------------
# EWC Fisher (EWC.py:126-164)
# ----------------------------------------------------------------------------------------
def fisher_diag(params, rows_ids: torch.Tensor, rows_pos: torch.Tensor, max_item: int,
                hp: Hyper, n_data: int) -> List[np.ndarray]:
    """Per-sample (batch of one) gradients of the vanilla CE, squared, summed in float64
    and divided by ``len(data)`` (EWC.py:135-164).  ``n_data`` is len(data) -- rows of
    length <=1 are skipped by the sampler but still counted (SURVEY a14)."""
    acc = [np.zeros(tuple(p.shape), np.float64) for p in params]
    for i in range(rows_ids.shape[0]):
        _, gs = grads_of(lambda ps: loss_vanilla(ps, rows_ids[i:i + 1], rows_pos[i:i + 1],
                                                 max_item, hp), params)
        for a, g in zip(acc, gs):
            a += np.square(g.double().numpy())
    return [a / n_data for a in acc]


# ----------------------------------------------------------------------------------------
# Packed (real-token-only) forward -- used ONLY to self-check that the product's packing
# is exact w.r.t. the dense reference form (SURVEY A.10); not a reference restatement.
# ----------------------------------------------------------------------------------------
def forward_rep_packed(params, ids: torch.Tensor, hp: Hyper) -> torch.Tensor:
    d, L = hp.hidden_units, hp.maxlen
    reps = []
    for r in range(ids.shape[0]):
        row = ids[r]
        n = int((row != 0).sum())
        tok = row[L - n:].long()
        x = params[0][tok] * (d ** 0.5) + params[1][L - n:]
        for b in range(hp.num_blocks):
            (ln1b, ln1g, wq, bq, wk, bk, wv, bv, ln2b, ln2g, w1, b1, w2, b2) = params[2 + 14 * b: 16 + 14 * b]
            q = normalize(x, ln1b, ln1g)
            Q, K, V = q @ wq + bq, x @ wk + bk, x @ wv + bv
            dh = d // hp.num_heads
            outs = []
            for h in range(hp.num_heads):
                sl = slice(h * dh, (h + 1) * dh)
                S = Q[:, sl] @ K[:, sl].t() / (dh ** 0.5)
                S = S.masked_fill(torch.triu(torch.ones(n, n, dtype=torch.bool), 1), float("-inf"))
                outs.append(torch.softmax(S, -1) @ V[:, sl])
            y = torch.cat(outs, 1) + q
            x = feedforward(normalize(y, ln2b, ln2g), w1, b1, w2, b2)
        reps.append(normalize(x, params[-2], params[-1])[-1])
    return torch.stack(reps)
