"""CPU checks of the dropout mask stream the kernels draw (csrc/common.cuh: fmix32 / drop_site / drop_mul) and of
its NumPy port in oracle/dropout.py, which the GPU tests (tests/test_gpu_dropout.py) use to replay the library's
masks in the fp64 oracle:

* the port's threshold and keep scale at the edge rates, and the statistics of its stream (drop rate per site,
  independence of two sites of one step and of one site at consecutive steps);
* the packed-token -> padded-layout index map against a per-element loop, and the oracle with all-ones multipliers
  against the oracle without dropout;
* every entry that takes a dropout rate refuses a rate outside [0, 1) before any CUDA call (fake non-null device
  addresses suffice, as in tests/test_loss_args.py);
* the rank salt of the seed: rank 0 keeps the single-GPU stream, ranks 0..7 draw from distinct keys.
"""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from oracle import dropout as D
from oracle import sasrec as S

N_SITES = 25            # 8 blocks: sites 0 .. 3*8
FAKE = 0x10000


# ---- the port ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("p,thr,keep_bits", [
    (2.0 ** -24, 1, 0x3F800001),                   # smallest rate: one value of 2^24 drops; keep = 1 + 2^-23
    (0.3, 5033165, 0x3FB6DB6E),                    # fp32(0.3) * 2^24 is an integer: ceil is exact; keep = fp32(1/fp32(0.7))
    (0.5, 8388608, 0x40000000),                    # keep 2
    (1.0 - 2.0 ** -24, 16777215, 0x4B800000),      # largest rate below 1: one value keeps; keep = 2^24
])
def test_port_threshold_and_keep_at_edge_rates(p, thr, keep_bits):
    _, t, keep = D.drop_site(12345, 7, p)
    assert t == thr
    assert np.float32(keep).view(np.uint32) == keep_bits
    assert D.drop_site(0, 0, 0.0)[1] == 0               # p = 0: nothing drops
    # at the smallest rate only r >> 8 == 0 drops, at the largest only r >> 8 == 2^24 - 1 keeps
    bits = np.array([0, 1, 2 ** 24 - 2, 2 ** 24 - 1], np.uint64)
    assert list(bits < np.uint64(t)) == [bool(b < thr) for b in bits.tolist()]


def test_fmix32_matches_reference_values():
    """murmur3 fmix32 on a few values computed with Python integers (uint32 wrap-around)."""
    def ref(h):
        h ^= h >> 16; h = (h * 0x85EBCA6B) & 0xFFFFFFFF
        h ^= h >> 13; h = (h * 0xC2B2AE35) & 0xFFFFFFFF
        return h ^ (h >> 16)
    xs = [0, 1, 2, 0x7FFFFFFF, 0x80000000, 0xFFFFFFFF, 0xDEADBEEF, 123456789]
    assert [int(v) for v in D.fmix32(np.array(xs, np.uint64))] == [ref(x) for x in xs]
    # indices above 2^32 fold their high half in: two indices 2^32 apart draw different bits
    key = D.drop_site(5, 1, 0.3)[0]
    assert int(D.site_bits(key, [7])[0]) != int(D.site_bits(key, [7 + 2 ** 32])[0])


def _within(k, n, q, sig=5.0):
    """k successes of n Bernoulli(q) trials within sig standard deviations"""
    return abs(k / n - q) <= sig * math.sqrt(q * (1 - q) / n)


@pytest.mark.parametrize("p", [0.1, 0.3, 0.9])
def test_port_stream_statistics(p):
    """Over 10^6 indices: every one of the 25 sites drops at rate p; two sites of one step, and one site at steps t and
    t + 1, agree at the rate p^2 + (1-p)^2 of independent masks (5 sigma).  A regression in how the key mixes the site
    or the step (two sites or two steps sharing a key, or keys differing in a way the hash does not spread) fails here."""
    n = 10 ** 6
    idx = np.arange(n, dtype=np.uint64) * np.uint64(3) + np.uint64(11)
    seed = (17 << 32) + 5
    q = p * p + (1 - p) * (1 - p)
    drops = []
    for site in range(N_SITES):
        key, thr, _ = D.drop_site(seed, site, p)
        dr = D.site_bits(key, idx) < np.uint64(thr)
        assert _within(int(dr.sum()), n, p), "site %d drops %.5f" % (site, dr.mean())
        drops.append(dr)
    for a, b in [(0, 1), (1, 2), (2, 3), (0, 24), (3, 4), (22, 23)]:
        assert _within(int((drops[a] == drops[b]).sum()), n, q), "sites %d / %d" % (a, b)
    for site in (0, 1, 5, 24):
        key, thr, _ = D.drop_site(seed + 1, site, p)
        nxt = D.site_bits(key, idx) < np.uint64(thr)
        assert _within(int((drops[site] == nxt).sum()), n, q), "site %d, steps t / t+1" % site


# ---- the padded-layout multipliers --------------------------------------------------------------------------------
def _ids(rng, M, L, lens):
    ids = np.zeros((M, L), np.int32)
    for r, k in enumerate(lens):
        ids[r, L - k:] = rng.randint(1, 50, k)
    return ids


@pytest.mark.parametrize("L,d,h,nb,tight", [(7, 6, 2, 2, True), (7, 6, 2, 2, False), (1, 3, 1, 1, True), (9, 4, 4, 3, False)])
def test_dense_multipliers_match_a_per_element_loop(L, d, h, nb, tight):
    rng = np.random.RandomState(L * 10 + d)
    lens = [L, 1, 0, max(L - 2, 1)] + list(rng.randint(1, L + 1, 3))
    ids = _ids(rng, len(lens), L, lens)
    T = sum(lens)
    Tcap = T if tight else len(lens) * L
    seed, p = (3 << 32) + 9, 0.4
    got = D.dense_multipliers(seed, p, ids, Tcap, d, h, nb)
    assert sorted(got) == list(range(1 + 3 * nb))
    one = lambda site, idx: float(D.drop_mul(seed, site, p, [idx])[0])
    tk = 0
    M = len(lens)
    for r, n in enumerate(lens):
        for i in range(n):
            s = L - n + i
            for c in range(d):
                assert got[0][r, s, c] == one(0, tk * d + c)
                for b in range(nb):
                    for site in (2 + 3 * b, 3 + 3 * b):
                        assert got[site][r, s, c] == one(site, tk * d + c)
            for b in range(nb):
                for hh in range(h):
                    for j in range(n):
                        assert got[1 + 3 * b][hh * M + r, s, L - n + j] == one(1 + 3 * b, (hh * Tcap + tk) * L + j)
            tk += 1
        # padding slots are neutral
        for site, a in got.items():
            if site % 3 == 1:
                for hh in range(h):
                    assert np.all(a[hh * M + r, :L - n, :] == 1) and np.all(a[hh * M + r, :, :L - n] == 1)
            else:
                assert np.all(a[r, :L - n] == 1)
    with pytest.raises(ValueError):
        D.dense_multipliers(seed, p, ids, T - 1, d, h, nb)


def test_oracle_with_all_ones_multipliers_is_the_unmasked_oracle():
    hp = S.Hyper(60, 8, 6, 2, 2)
    params = [p.double() for p in S.randomize_params(S.init_params(hp, 0), 1, 0.05)]
    rng = np.random.RandomState(2)
    ids = torch.tensor(_ids(rng, 5, 6, [6, 1, 3, 5, 2])).long()
    pos = torch.tensor(rng.randint(1, 40, 3))
    ones = {k: np.ones_like(v) for k, v in D.dense_multipliers(0, 0.3, ids.numpy(), 17, 8, 2, 2).items()}
    ex_pos = torch.tensor([3, 9])
    for lit in (True, False):
        with S.literal_masks(lit):
            assert torch.equal(S.forward_rep(params, ids, hp, ones), S.forward_rep(params, ids, hp))
            assert torch.equal(S.loss_vanilla(params, ids, ids[:, -1], 50, hp, drop=ones),
                               S.loss_vanilla(params, ids, ids[:, -1], 50, hp))
            assert torch.equal(S.loss_ader(params, ids, pos, 50, hp, 0.5, exemplar_pos=ex_pos, drop=ones),
                               S.loss_ader(params, ids, pos, 50, hp, 0.5, exemplar_pos=ex_pos))
    # and a real mask changes the result
    drop = D.dense_multipliers(0, 0.3, ids.numpy(), 17, 8, 2, 2)
    with S.literal_masks(False):
        assert not torch.equal(S.forward_rep(params, ids, hp, drop), S.forward_rep(params, ids, hp))


# ---- rate refusals ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    from ader_b200 import _lib, build
    build.build()
    return _lib.load()


def _call(lib, entry, p):
    from ader_b200 import _lib, ops
    from ader_b200.params import Hyper
    ms = ops.model_struct(Hyper(4000))
    f = C.c_void_p(FAKE)
    M, Tcap = 64, 64 * 50
    if entry == "ader_encoder_fwd":
        return lib.ader_encoder_fwd(C.byref(ms), f, f, M, Tcap, f, f, p, 0, None)
    if entry == "ader_encoder_fwd_tc":
        return lib.ader_encoder_fwd_tc(C.byref(ms), f, f, M, Tcap, f, f, p, 0, None, None)
    if entry == "ader_encoder_bwd":
        return lib.ader_encoder_bwd(C.byref(ms), f, f, M, Tcap, f, f, f, f, p, 0, None)
    if entry == "ader_encoder_bwd_tc":
        return lib.ader_encoder_bwd_tc(C.byref(ms), f, f, M, Tcap, f, f, f, f, p, 0, None, None)
    a = ops.make_loss_args(M, M, 0, 3000, 0, 0, 0.0)
    a.pos = FAKE
    if entry == "ader_train_fwd_bwd_tc":     # serial plan: no library streams exist before the checks
        return lib.ader_train_fwd_bwd_tc(C.byref(ms), f, f, M, Tcap, C.byref(a), f, f, f, f, f, f, f, f, p, 0, None, 1, None)
    assert entry == "ader_train_step_tc"
    opt = _lib.AderAdamArgs(5e-4, 0.9, 0.999, 1e-8, 3000, 0.0, None, None)
    return lib.ader_train_step_tc(C.byref(ms), f, f, M, Tcap, C.byref(a), f, f, f, f, f, f, f, f, p, 0, None, f, f, f,
                                  C.byref(opt), 1, None)


ENTRIES = ["ader_encoder_fwd", "ader_encoder_fwd_tc", "ader_encoder_bwd", "ader_encoder_bwd_tc", "ader_train_fwd_bwd_tc",
           "ader_train_step_tc"]


@pytest.mark.parametrize("entry", ENTRIES)
@pytest.mark.parametrize("p", [-0.1, 1.0, 1.5, float("nan"), float("inf")], ids=["neg", "one", "above_one", "nan", "inf"])
def test_every_entry_refuses_a_bad_dropout_rate_before_any_launch(lib, entry, p):
    """Rate 1 would scale by 1/(1-1) = inf (NaN gradients), a rate above 1 by a negative factor, and a NaN rate turns
    the masks off (p > 0 is false) in one pass but not the other.  The refusal comes before any CUDA call: the fake
    addresses are never touched."""
    assert _call(lib, entry, p) == -1
    msg = lib.ader_last_error().decode()
    assert "dropout_rate" in msg and entry[len("ader_"):] in msg, msg


# ---- the rank salt ------------------------------------------------------------------------------------------------
def test_rank_salt_keeps_rank_zero_and_separates_ranks():
    from ader_b200.model import DROPOUT_RANK_SALT, dropout_seed
    assert DROPOUT_RANK_SALT % 2 == 1
    for rs in (0, 1, 7, 12345, 2 ** 31 - 1):
        assert dropout_seed(rs) == dropout_seed(rs, 0) == (rs << 32)     # single GPU / rank 0: the unsalted stream
        for step in (0, 1, 1000, 2 ** 31 + 3):
            keys = {}
            for rank in range(8):
                seed = dropout_seed(rs, rank) + step
                assert seed < 2 ** 64
                for site in range(N_SITES):
                    keys.setdefault(D.drop_site(seed, site, 0.3)[0], []).append((rank, site))
            # 200 pairwise distinct keys: no two ranks share the masks of any site, nor does one rank's site repeat
            # another rank's other site
            assert len(keys) == 8 * N_SITES, [v for v in keys.values() if len(v) > 1]
