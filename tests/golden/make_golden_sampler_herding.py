"""Mint sampler_herding.json: the outputs on the inputs of test_live_reference_sampler_and_herding, so that its comparison
runs on every machine, not only where the reference is mounted.

    python tests/golden/make_golden_sampler_herding.py                  # from the reference's own util.py (needs it mounted)
    python tests/golden/make_golden_sampler_herding.py --from-oracle    # from oracle/protocol.py

Inputs: 200 random sessions (seed 3) through Sampler(maxlen 50, batch 32) after random.seed(5) / np.random.seed(5):
split_data(0.1), then 2 * batch_num + 1 batches (two reshuffles); and herding picks for (n, m) = (4, 2), (17, 9), (60, 31)
on float32 reps drawn from the same seed-3 stream.  `source` in the file records which code produced it;
test_live_reference_sampler_and_herding checks the file against the reference whenever the reference is mounted.
"""
import json
import os
import random
import sys
from collections import defaultdict

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import protocol as P  # noqa: E402
from oracle import refstub  # noqa: E402

MAXLEN = 50
HERDING_CASES = [(4, 2), (17, 9), (60, 31)]


def outputs(sampler_cls, split, herding):
    """split(sampler) -> (valid, train); herding(rep, m) -> list of picked candidate indices."""
    rng = np.random.RandomState(3)
    data = [rng.randint(1, 40, rng.randint(1, 9)).tolist() for _ in range(200)]
    random.seed(5)
    np.random.seed(5)
    s = sampler_cls(data, MAXLEN, 32)
    valid, train = split(s)
    batches = []
    for _ in range(s.batch_num() * 2 + 1):
        q, p = s.sampler()
        batches.append([np.array(q).tolist(), list(map(int, p))])
    picks = [herding(rng.randn(n, 150).astype(np.float32), m) for n, m in HERDING_CASES]
    # JSON form: plain ints and lists, as the stored file reads back
    return json.loads(json.dumps({"valid": valid, "train": train, "batches": batches, "herding": picks},
                                 default=lambda o: o.tolist()))


def oracle_outputs():
    return outputs(P.RefSampler, lambda s: s.split_data(0.1), P.herding_picks)


def reference_outputs(util):
    gen = util.ExemplarGenerator.__new__(util.ExemplarGenerator)
    gen.exemplars = defaultdict(list)

    def herding(rep, m):
        n = len(rep)
        seq = np.zeros((n, MAXLEN + 1), np.int64)
        seq[:, -1] = 1
        seq[:, -2] = np.arange(1, n + 1)
        gen.herding(rep, np.zeros((n, 1), np.float32), seq, 0, m)
        return [e[0][0] - 1 for e in gen.exemplars[0]]

    return outputs(util.Sampler, lambda s: s.split_data(valid_portion=0.1, return_train=True), herding)


def main():
    if "--from-oracle" in sys.argv:
        out, source = oracle_outputs(), "oracle/protocol.py (RefSampler, herding_picks)"
    else:
        out, source = reference_outputs(refstub.load_reference_util()), "reference util.py (Sampler, ExemplarGenerator.herding)"
    out["source"] = source
    with open(os.path.join(HERE, "sampler_herding.json"), "w") as f:
        json.dump(out, f, separators=(",", ":"))
    print("wrote sampler_herding.json from", source)


if __name__ == "__main__":
    main()
