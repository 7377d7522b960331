"""Top-k next-item lists for a file of sessions, from the checkpoint a training run writes.

    python -m ader_b200.recommend --checkpoint results/DIGINETICA-ADER/checkpoint.pt --sessions sessions.txt --out topk.txt
        [--k 20] [--keep_seen] [--max_item N] [--scores | --probs] [--batch 4096]

Input: one session per line, item ids separated by whitespace, oldest first.  The model reads the last ``maxlen`` items of
each session, right-aligned, as it read the sessions it was trained on.  Output: one line per input line with ``k`` ids,
best first (``id:score`` pairs with ``--scores``, ``id:probability`` pairs with ``--probs``).  A session's own items are
never recommended unless ``--keep_seen``; a session with fewer than ``k`` items left to recommend is padded with item 0
(score -inf, probability 0).

The probability is the model's next-item softmax, p(j | session) = exp(score_j - lse) with lse = log sum exp(score) over
ALL items 1..max_item, the session's own items included (the distribution the model was trained to fit).  A line's listed
probabilities therefore sum to at most 1: the rest belongs to the items not listed, excluded ones among them.
"""
from __future__ import annotations

import argparse
import types
from typing import List, Optional, Sequence

import numpy as np

from .data import pack_rows
from .params import Hyper, ParamLayout

SHAPE_KEYS = ("hidden_units", "maxlen", "num_blocks", "num_heads")


def build_parser() -> argparse.ArgumentParser:
    p = argparse.ArgumentParser(prog="python -m ader_b200.recommend", description=__doc__.split("\n\n")[0])
    p.add_argument("--checkpoint", required=True, help="checkpoint.pt written by ader_b200.main")
    p.add_argument("--sessions", required=True, help="text file: one session per line, item ids oldest first")
    p.add_argument("--out", required=True, help="output file: one line of k items per session")
    p.add_argument("--k", default=20, type=int, help="items per session, 1..100")
    p.add_argument("--keep_seen", action="store_true", help="allow a session's own items in its list")
    p.add_argument("--max_item", default=None, type=int, help="rank items 1..max_item (default: the largest item seen in training)")
    out = p.add_mutually_exclusive_group()
    out.add_argument("--scores", action="store_true", help="write id:score pairs")
    out.add_argument("--probs", action="store_true", help="write id:probability pairs (softmax over all items 1..max_item)")
    p.add_argument("--batch", default=4096, type=int, help="sessions per device pass")
    return p


def model_shape(st: dict) -> Hyper:
    """Network shape of a checkpoint: hidden_units, maxlen, num_blocks and num_heads from the run's recorded flags, the item
    table's row count from the length of theta."""
    args = st.get("args")
    if not args or any(args.get(k) is None for k in SHAPE_KEYS):
        raise ValueError("the checkpoint does not record the model shape (%s)" % ", ".join(SHAPE_KEYS))
    d, L, nb, nh = (int(args[k]) for k in SHAPE_KEYS)
    n = int(st["model"]["theta"].numel())
    rest = n - ParamLayout(Hyper(1, d, L, nb, nh)).dense_count
    if rest <= 0 or rest % d or rest // d < 2:
        raise ValueError("theta of %d elements does not fit hidden_units=%d, maxlen=%d, num_blocks=%d" % (n, d, L, nb))
    hp = Hyper(rest // d - 1, d, L, nb, nh)
    if ParamLayout(hp).total != n:
        raise ValueError("theta of %d elements does not match the layout of %s" % (n, hp))
    return hp


def read_sessions(path: str, v_tab: int) -> List[List[int]]:
    """One session per line; an empty line, a token that is not an integer or an id outside 1..v_tab-1 is an error that
    names the line."""
    out = []
    with open(path) as f:
        for no, line in enumerate(f, 1):
            toks = line.split()
            if not toks:
                raise ValueError("%s:%d: empty session" % (path, no))
            try:
                s = [int(t) for t in toks]
            except ValueError:
                raise ValueError("%s:%d: item ids must be integers" % (path, no)) from None
            bad = [x for x in s if not 1 <= x < v_tab]
            if bad:
                raise ValueError("%s:%d: item id %d outside 1..%d" % (path, no, bad[0], v_tab - 1))
            out.append(s)
    return out


def session_rows(sessions: Sequence[Sequence[int]], maxlen: int):
    """ids [N, maxlen] int32 (the last maxlen items of each session, right-aligned) and the token count of each row."""
    ids, _, n_in = pack_rows([list(s) + [0] for s in sessions], maxlen)
    return ids, n_in


def format_line(items: Sequence[int], scores: Optional[Sequence[float]] = None) -> str:
    if scores is None:
        return " ".join(str(int(i)) for i in items)
    return " ".join("%d:%.9g" % (int(i), float(s)) for i, s in zip(items, scores))


def load_model(path: str, device=None):
    """(Ader with the checkpoint's weights, default max_item)."""
    import torch
    from .model import Ader
    st = torch.load(path, map_location="cpu", weights_only=False)
    if st.get("format") != 1:
        raise ValueError("%s: unknown checkpoint format" % path)
    hp = model_shape(st)
    args = types.SimpleNamespace(hidden_units=hp.hidden_units, maxlen=hp.maxlen, num_blocks=hp.num_blocks,
                                 num_heads=hp.num_heads, random_seed=0, lr=0.0, dropout_rate=0.0)
    model = Ader(hp.item_num, args, device=device, init_seed=0)
    model.theta.copy_(st["model"]["theta"].to(model.device))
    return model, int(np.max(st["item_set"]))


def recommend_sessions(model, sessions, max_item: int, k: int = 20, exclude_seen: bool = True, batch: int = 4096,
                       probs: bool = False):
    """items [N, k] int32 and scores [N, k] fp32 (host arrays) for a list of sessions; probs: probabilities instead of
    scores (``Ader.recommend``)."""
    ids, n_in = session_rows(sessions, model.hp.maxlen)
    items, scores = [], []
    for lo in range(0, len(sessions), batch):
        it, sc = model.recommend(ids[lo:lo + batch], max_item, k, exclude_seen, n_tokens=int(n_in[lo:lo + batch].sum()),
                                 probs=probs)
        items.append(it.cpu().numpy()); scores.append(sc.cpu().numpy())
    if not items:
        return np.zeros((0, k), np.int32), np.zeros((0, k), np.float32)
    return np.concatenate(items), np.concatenate(scores)


def main(argv=None) -> None:
    a = build_parser().parse_args(argv)
    if not 1 <= a.k <= 100:
        raise SystemExit("--k must be in 1..100")
    if a.batch < 1:
        raise SystemExit("--batch must be >= 1")
    model, max_item = load_model(a.checkpoint)
    if a.max_item is not None:
        max_item = a.max_item
    if not 1 <= max_item < model.hp.v_tab:
        raise SystemExit("--max_item must be in 1..%d" % (model.hp.v_tab - 1))
    try:
        sessions = read_sessions(a.sessions, model.hp.v_tab)
    except ValueError as e:
        raise SystemExit(str(e)) from None
    items, scores = recommend_sessions(model, sessions, max_item, a.k, not a.keep_seen, a.batch, probs=a.probs)
    with open(a.out, "w") as f:
        for r in range(items.shape[0]):
            f.write(format_line(items[r], scores[r] if (a.scores or a.probs) else None) + "\n")


if __name__ == "__main__":
    main()
