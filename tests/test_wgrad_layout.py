"""The shared-memory addressing of the weight-gradient kernel (ader_b200/csrc/encoder_fused.cuh: k_wgrad2),
restated on the CPU: the k slots of a TF32 m16n8k8 step are mapped to rows of the 32-token tile so that
  (a) every tile row is consumed by exactly one (k-step, k slot) -- the product sums over all 32 tokens once, and
  (b) with the tile stored at its natural row stride d = 150 floats (one bulk copy, no padding) the 32 lanes of every
      fragment load touch 32 different shared-memory banks.
The kernel itself is checked against the oracle on the GPU; this pins the index arithmetic the comments claim."""
import numpy as np

WG_TK = 32


def rows_of_kstep(ks):
    """lane -> (row of k slot t4, row of k slot t4 + 4) for k-step ks (encoder_fused.cuh: `row = (ks >> 1) * 16 + (ks & 1) * 2 + 4 * t4`)."""
    t4 = np.arange(32) & 3
    row = (ks >> 1) * 16 + (ks & 1) * 2 + 4 * t4
    return row, row + 1


def test_every_tile_row_is_used_exactly_once():
    used = []
    for ks in range(WG_TK // 8):
        lo, hi = rows_of_kstep(ks)
        used += sorted(set(lo.tolist())) + sorted(set(hi.tolist()))
    assert sorted(used) == list(range(WG_TK))


def test_fragment_loads_are_bank_conflict_free_at_d_150():
    d = 150
    g = np.arange(32) >> 2
    for ks in range(WG_TK // 8):
        lo, hi = rows_of_kstep(ks)
        for rows in (lo, hi):
            for col0 in (0, 8, 16, 24, 40, 80, 88, 120, 152):       # wm * 80 + i * 16 (+ 8), half * 80 + wn * 40 + j * 8
                banks = (rows * d + col0 + g) % 32
                assert len(set(banks.tolist())) == 32, (ks, col0)
