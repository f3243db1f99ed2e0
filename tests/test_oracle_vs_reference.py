"""The C restatement against the reference sources THEMSELVES (tape-mode build under
oracle/_ref, built by oracle/build_ref.sh from the reference's source directory).  Every case is also
checked against a stored digest of the restatement's output on the same case
(tests/golden/recorded_outputs.json; how it was recorded: tests/conftest.py, Recorded), so the
comparison runs where the reference sources are not built too."""
import os
import random

import numpy as np

KEYS_W = ["simTimeMs", "nSuccess", "preambleTxSum", "delaySum", "failCountSum", "continueFailed",
          "collisionPreambles", "totalPreambleTxop", "draws", "maxDrawsPerUeMs"]
KEYS_B = ["simTimeMs", "nSuccess", "preambleTxSum", "delaySum", "collisionScans", "totalScans",
          "draws", "maxDrawsPerUeMs"]


def _compare(O, recorded, key, variant, kw):
    cfg = O.make_config(**kw)
    p, ue2, g2 = O.run_port(cfg, geom=(variant == "w"))
    pd = p.as_dict()
    cols = list(range(14)) + ([14, 15] if variant == "w" else [])
    keys = KEYS_W if variant == "w" else KEYS_B
    geom = {"geom": g2.view(np.uint32)} if variant == "w" else {}
    recorded.check(key, recorded.digest(config=kw, ue=ue2[:, cols], **geom, **{k: pd[k] for k in keys}))
    if O.ref_available(variant):
        r, ue, g = O.run_ref(variant, cfg, geom=(variant == "w"))
        rd = r.as_dict()
        for k in keys:
            assert rd[k] == pd[k], (k, kw)
        np.testing.assert_array_equal(ue[:, cols], ue2[:, cols], err_msg=str(kw))
        if variant == "w":
            np.testing.assert_array_equal(g.view(np.uint32), g2.view(np.uint32))
    assert pd["aborted"] == 0
    return pd


def test_defaults_w_and_b(oracle, recorded):
    _compare(oracle, recorded, "defaults_w", "w", dict(nUE=6000, seed=42, rep=1))
    _compare(oracle, recorded, "defaults_b", "b", dict(nUE=6000, nGrantUL=54, geometry=0, seed=42))


def test_fuzz_parameters(oracle, recorded):
    """Exotic corners: 1-2 UEs, 1-3 preambles, BI=1 (always immediate), limit branch always
    (mrc 1), RAR window 1, subframes 6/7/10 (grant reset stays on %5, W:268; Msg3 restart
    aligns on 5, W:687), Uniform traffic."""
    rnd = random.Random(2024)
    late = 0
    for i in range(40):
        variant = rnd.choice(["w", "w", "b"])
        kw = dict(nUE=rnd.choice([1, 2, 7, 50, 300, 1500, 3000]),
                  distribution=rnd.choice([1, 2, 2]),
                  nPreamble=rnd.choice([1, 2, 3, 8, 54, 64]),
                  backoffIndicator=rnd.choice([1, 2, 5, 20, 40]),
                  nGrantUL=rnd.choice([1, 2, 4, 12, 54]),
                  maxRarWindow=rnd.choice([2, 3, 6, 6, 9]),
                  maxMsg2TxCount=rnd.choice([0, 1, 3, 9, 19]),
                  accessTime=rnd.choice([5, 5, 5, 6, 7, 10]),
                  seed=rnd.getrandbits(64), rep=rnd.randrange(5000),
                  geometry=1 if variant == "w" else 0,
                  cellRadius=rnd.choice([400.0, 777.5]))
        late += _compare(oracle, recorded, "fuzz_%d" % i, variant, kw)["lateRestarts"]
    assert late > 0     # the Msg3-restart-lands-on-this-ms corner (SURVEY H5) was exercised


def test_noma_variant_against_noma_c(oracle, recorded):
    """rach_oracle_n.c against NOMA.c itself in tape mode: 16 ints and the fp64 channelGain of every UE."""
    live = os.path.exists(os.path.join(os.path.dirname(oracle.__file__), "_ref", "libref_n.so"))
    rnd = random.Random(99)
    cases = [dict(nUE=2000), dict(nUE=12000, seed=3, rep=2)]
    for _ in range(25):
        cases.append(dict(nUE=rnd.choice([1, 5, 300, 3000, 8000]), nPreamble=rnd.choice([1, 3, 54, 64]),
                          backoffIndicator=rnd.choice([1, 2, 20, 40]), nGrantUL=rnd.choice([1, 2, 4, 12]),
                          maxMsg2TxCount=rnd.choice([1, 3, 10]), accessTime=rnd.choice([5, 5, 6, 10]),
                          maxRarWindow=rnd.choice([3, 5]), cellRadius=rnd.choice([100.0, 500.0]),
                          seed=rnd.getrandbits(60), rep=rnd.randrange(1000), geometry=rnd.choice([0, 1])))
    cases += [dict(nUE=9000, geometry=0, seed=5), dict(nUE=15000, geometry=0, nGrantUL=12, seed=6)]   # N:325-447 variant
    keys = ("nSuccess", "preambleTxSum", "delaySum", "draws", "maxDrawsPerUeMs")
    for i, kw in enumerate(cases):
        cfg = oracle.make_config_n(**kw)
        p, ue2, g2 = oracle.run_port_n(cfg)
        recorded.check("noma_%d" % i, recorded.digest(config=kw, ue=ue2, gain=g2.view(np.uint64),
                                                      **{k: getattr(p, k) for k in keys}))
        if not live:
            continue
        r, ue, g = oracle.run_ref_n(cfg)
        for k in keys:
            assert getattr(r, k) == getattr(p, k), (k, kw)
        np.testing.assert_array_equal(ue, ue2, err_msg=str(kw))
        np.testing.assert_array_equal(g.view(np.uint64), g2.view(np.uint64))


def test_legacy_variant_against_randomaccesssimulator_c(oracle, recorded):
    """rach_oracle_u0.c against RandomAccessSimulator.c itself in tape mode (with the two-line fix):
    light load as shipped, and overload with few preambles where dropped UEs keep colliding (U0:207)."""
    live = os.path.exists(os.path.join(os.path.dirname(oracle.__file__), "_ref", "libref_u0.so"))
    rnd = random.Random(5)
    cases = [dict(nUE=2000), dict(nUE=15000, seed=2), dict(nUE=40000, nPreamble=1, seed=3), dict(nUE=36000, nPreamble=2, backoffIndicator=5, seed=4)]
    for _ in range(10):
        cases.append(dict(nUE=rnd.choice([1, 2, 50, 400, 3000, 8000]), nPreamble=rnd.choice([1, 2, 3, 8, 64]),
                          backoffIndicator=rnd.choice([1, 2, 5, 20, 40]), seed=rnd.getrandbits(60), rep=rnd.randrange(1000)))
    keys = ("simTimeMs", "nSuccess", "preambleTxSum", "delaySum", "collisionPreambles", "totalPreambleTxop", "draws")
    dropped = 0
    for i, kw in enumerate(cases):
        cfg = oracle.make_config_u0(**kw)
        p, ue2 = oracle.run_port_u0(cfg)
        recorded.check("legacy_u0_%d" % i, recorded.digest(config=kw, ue=ue2, **{k: getattr(p, k) for k in keys}))
        dropped += int((ue2[:, 11] == -1).sum())
        if not live:
            continue
        r, ue = oracle.run_ref_u0(cfg)
        for k in keys:
            assert getattr(r, k) == getattr(p, k), (k, kw)
        np.testing.assert_array_equal(ue, ue2, err_msg=str(kw))
    assert dropped > 0
