"""The library's dropout masks, bit for bit, in NumPy (TEST INFRASTRUCTURE ONLY).

The CUDA kernels draw their masks from a stateless hash (ader_b200/csrc/common.cuh: fmix32 / drop_site /
drop_mul): the multiplier of element ``idx`` of dropout site ``site`` at seed ``seed`` is 0 or ``keep = 1/(1-p)``
(float32).  ``seed`` is ``dropout_seed(random_seed, rank) + step`` (ader_b200/model.py); the element index is
that of the packed token layout, so :func:`dense_multipliers` places every multiplier in the oracle's padded
``[M, maxlen]`` layout (oracle/sasrec.py applies them with ``drop=``).

Sites (``b`` = block):
  0       embedding after the position add, before the padding mask (ADER.py:55-58)    idx = tk*d + c
  1 + 3b  attention weights after softmax and query mask (modules.py:214)              idx = (h*Tcap + tk_q)*L + j
  2 + 3b  FFN inner activation after ReLU (modules.py:257)                              idx = tk*d + c
  3 + 3b  FFN output before the residual (modules.py:262)                               idx = tk*d + c
``tk = row_off[r] + i`` is the packed token of the i-th item of row r (slot L - n + i), ``row_off`` the exclusive
cumulative sum of the session lengths in row order, ``j`` the key's index inside the session.  The attention index
depends on the token capacity ``Tcap`` of the pass, so a mask is only reproduced at the Tcap the step was given.
"""
from __future__ import annotations

from typing import Dict

import numpy as np

M32 = np.uint64(0xFFFFFFFF)


def _u32(x):
    return np.asarray(x, dtype=np.uint64) & M32


def fmix32(h):
    """murmur3 finaliser on uint32 values (held in uint64 arrays, reduced mod 2^32 after every product)."""
    h = _u32(h)
    h ^= h >> np.uint64(16)
    h = (h * np.uint64(0x85EBCA6B)) & M32
    h ^= h >> np.uint64(13)
    h = (h * np.uint64(0xC2B2AE35)) & M32
    h ^= h >> np.uint64(16)
    return h


def drop_site(seed: int, site: int, p: float):
    """(key, thr, keep) of one site: key = fmix32(lo(seed)*0x9E3779B1 + hi(seed)*0x7FEB352D + site*0x846CA68B
    + 0x5bd1e995) mod 2^32, thr = ceil(p * 2^24) in float32 (0 at p = 0), keep = 1/(1-p) in float32."""
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    lo, hi = seed & 0xFFFFFFFF, seed >> 32
    k = (lo * 0x9E3779B1 + hi * 0x7FEB352D + (int(site) & 0xFFFFFFFF) * 0x846CA68B + 0x5BD1E995) & 0xFFFFFFFF
    key = int(fmix32(k))
    pf = np.float32(p)
    thr = int(np.ceil(pf * np.float32(16777216.0))) if pf > np.float32(0) else 0
    with np.errstate(divide="ignore"):
        keep = np.float32(1.0) / (np.float32(1.0) - pf)
    return key, thr, keep


def site_bits(key: int, idx) -> np.ndarray:
    """(r >> 8) of every element index: the element is dropped where this is below thr."""
    idx = np.asarray(idx, dtype=np.uint64)
    lo, hi = idx & M32, idx >> np.uint64(32)
    r = fmix32((lo ^ np.uint64(key)) + ((hi * np.uint64(0x27D4EB2F)) & M32))
    return r >> np.uint64(8)


def drop_mul(seed: int, site: int, p: float, idx) -> np.ndarray:
    """float32 multipliers (0 or keep) of the element indices ``idx`` of one site."""
    key, thr, keep = drop_site(seed, site, p)
    return np.where(site_bits(key, idx) < np.uint64(thr), np.float32(0.0), keep).astype(np.float32)


def packed_tokens(ids: np.ndarray):
    """(row_len [M], row_off [M]) of left-padded sessions: the packed token of item i of row r is row_off[r] + i."""
    n = (np.asarray(ids) != 0).sum(axis=1).astype(np.int64)
    return n, np.concatenate([[0], np.cumsum(n)[:-1]]).astype(np.int64)


def dense_multipliers(seed: int, p: float, ids: np.ndarray, Tcap: int, d: int, num_heads: int,
                      num_blocks: int) -> Dict[int, np.ndarray]:
    """site -> float32 multipliers in the oracle's padded layout: [M, L, d] for the embedding and the FFN sites,
    [h*M, L, L] (head-major, as the oracle batches heads) for the attention weights.  Padding slots hold 1: the
    oracle zeroes them (padding mask, key mask) whatever they are multiplied by."""
    ids = np.asarray(ids)
    M, L = ids.shape
    n, off = packed_tokens(ids)
    if int(n.sum()) > Tcap:
        raise ValueError("Tcap %d is below the %d real tokens of the batch" % (Tcap, int(n.sum())))
    slot = np.arange(L)
    real = slot[None, :] >= (L - n)[:, None]                           # [M, L]
    tk = off[:, None] + slot[None, :] - (L - n)[:, None]               # packed token of (r, slot) where real
    tok_idx = (tk[:, :, None] * d + np.arange(d)[None, None, :]).clip(min=0)           # [M, L, d]
    h = np.arange(num_heads)[:, None, None, None]
    att_idx = ((h * Tcap + tk[None, :, :, None]) * L + (slot[None, None, None, :] - (L - n)[None, :, None, None]))
    att_real = real[None, :, :, None] & real[None, :, None, :]                         # [1, M, L, L]
    att_idx = np.where(att_real, att_idx, 0).reshape(num_heads * M, L, L)
    att_real = np.broadcast_to(att_real, (num_heads, M, L, L)).reshape(num_heads * M, L, L)
    out = {}

    def put(site, idx, mask):
        out[site] = np.where(mask, drop_mul(seed, site, p, idx), np.float32(1.0)).astype(np.float32)

    put(0, tok_idx, real[:, :, None])
    for b in range(num_blocks):
        put(1 + 3 * b, att_idx, att_real)
        put(2 + 3 * b, tok_idx, real[:, :, None])
        put(3 + 3 * b, tok_idx, real[:, :, None])
    return out


def block_drop(drop, b: int):
    """(attention, FFN inner, FFN output) multipliers of block b from a ``dense_multipliers`` dict (or None)."""
    if drop is None:
        return None, None, None
    return drop[1 + 3 * b], drop[2 + 3 * b], drop[3 + 3 * b]
