"""SURVEY T4: the reference driven by its own libc rand() and the same reference driven by the Philox draw
tape are two samples of one distribution.  Where the reference is built (oracle/_ref): 10 seeds each of
RandomAccessWithNOMA.c at 10 500 UEs (loaded but not saturated, so every statistic has visible spread).
Everywhere: 10 tape seeds of the restatement (bit-identical to the tape-mode reference, tests/test_oracle_golden.py)
against the rand() build's published 100-seed means (tests/golden/rand_build_published.json).  Means must agree
within 4 standard errors."""
import json
import os

import numpy as np

NAMES = ("success %", "preamble tx", "delay ms", "collided preambles / 1e5")


def _stats(results, n):
    return np.asarray([(100.0 * r.nSuccess / n, r.preambleTxSum / r.nSuccess, r.delaySum / r.nSuccess,
                        r.collisionPreambles / 1e5) for r in results])


def test_rand_and_tape_builds_agree_statistically(oracle):
    runs = 10
    with open(os.path.join(os.path.dirname(__file__), "golden", "rand_build_published.json")) as f:
        pub = json.load(f)
    for n, row in pub["points"].items():
        n = int(n)
        b = _stats([oracle.run_port(oracle.make_config(nUE=n, seed=1000 + s, rep=s), per_ue=False)[0]
                    for s in range(runs)], n)
        for k, name in enumerate(NAMES[:3]):
            # one distribution, so one spread: the tape sample's, for both means
            se = np.sqrt(b[:, k].var(ddof=1) * (1.0 / runs + 1.0 / pub["runs"])) + 1e-9
            assert abs(b[:, k].mean() - row[name]) <= 4.0 * se + 1e-6 * abs(row[name]), \
                (n, name, b[:, k].mean(), row[name], se)
    if not oracle.ref_available("w"):
        return
    n = 10500
    out = {0: [], 1: []}
    for tape in (0, 1):
        for seed in range(runs):
            cfg = oracle.make_config(nUE=n, seed=1000 + seed, rep=seed, useTape=tape)
            out[tape].append(oracle.run_ref("w", cfg, per_ue=False)[0])
    a, b = _stats(out[0], n), _stats(out[1], n)
    for k, name in enumerate(NAMES):
        se = np.sqrt(a[:, k].var(ddof=1) / runs + b[:, k].var(ddof=1) / runs) + 1e-9
        assert abs(a[:, k].mean() - b[:, k].mean()) <= 4.0 * se + 1e-6 * abs(a[:, k].mean()), \
            (name, a[:, k].mean(), b[:, k].mean(), se)
