"""Histograms of the successful UEs built on the GPU (ra_options.histograms, ra_sim_histogram, rach_sim --hist): every
histogram equals np.bincount over per-UE rows -- the reference's own rows, the oracle's, or the engine's dumps -- and
sums over replications and devices; the counters of a run do not change when histograms are on."""
import importlib
import os
import random
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TOP = 256
KEYS = ["simTimeMs", "nSuccess", "preambleTxSum", "delaySum", "failCountSum", "continueFailed",
        "collisionPreambles", "totalPreambleTxop", "collisionScans", "totalScans", "recordMoves"]
# per-UE row columns: (success flag, timer, tx, fail or None) of each variant's dump layout
COLS = {"w": (13, 0, 10, 14), "b": (13, 0, 10, None), "n": (13, 0, 10, None), "u0": (10, 0, 7, None)}


@pytest.fixture(scope="module")
def pkg():
    p = importlib.import_module("5g-nr-randomaccess_b200")
    p.load_lib()
    return p


def _bincount(values, n):
    return np.bincount(np.minimum(values, n - 1), minlength=n).astype(np.uint64)


def _expected(pkg, p, rows, variant):
    """{kind: bincount} of the successful rows"""
    done, timer, tx, fail = COLS[variant]
    ok = rows[:, done] == 1
    out = {pkg.HIST_DELAY: _bincount(rows[ok, timer], pkg.hist_bins(p, pkg.HIST_DELAY)),
           pkg.HIST_TX: _bincount(rows[ok, tx], TOP)}
    if fail is not None:
        out[pkg.HIST_FAIL] = _bincount(rows[ok, fail], TOP)
    return out


def _kinds(pkg, p):
    return (pkg.HIST_DELAY, pkg.HIST_TX) + ((pkg.HIST_FAIL,) if p.variant == 0 else ())


def _hists(pkg, sim, point):
    p = sim.points[point]
    return {k: sim.histogram(point, k) for k in _kinds(pkg, p)}


def _assert_equal(a, b, msg=""):
    assert sorted(a) == sorted(b), msg
    for k in a:
        np.testing.assert_array_equal(a[k], b[k], err_msg="kind %d %s" % (k, msg))


def _identities(pkg, h, stats):
    """the histograms of a point against the counters of its replications"""
    n = int(stats["nSuccess"].sum())
    for v in h.values():
        assert int(v.sum()) == n
    d = h[pkg.HIST_DELAY]
    assert int((np.arange(len(d), dtype=np.uint64) * d).sum()) == int(stats["delaySum"].sum())
    for kind, key in ((pkg.HIST_TX, "preambleTxSum"), (pkg.HIST_FAIL, "failCountSum")):
        if kind in h and h[kind][-1] == 0:
            assert int((np.arange(TOP, dtype=np.uint64) * h[kind]).sum()) == int(stats[key].sum())


def _params(pkg, cfg, variant):
    kw = {k: v for k, v in cfg.items() if k not in ("useTape", "echo", "rep", "stopMs")}
    if variant == "n":
        for k in ("distribution", "hBS", "hUT"):
            kw.pop(k)
        return pkg.default_params(variant=2, **kw)
    if variant == "u0":
        return pkg.default_params(variant=1, **{k: kw[k] for k in ("nUE", "nPreamble", "backoffIndicator", "seed")})
    p = pkg.default_params(**kw)
    if cfg.get("stopMs"):
        p.maxTimeMs = cfg["stopMs"]
    return p


def test_reference_fixtures(pkg, golden):
    """every fixture with the reference's own per-UE rows (W, B, N and U0)"""
    stats, ues = golden
    for name, rows in ues.items():
        g = stats[name]
        p = _params(pkg, g["config"], g["variant"])
        with pkg.RachSim([p], reps=1, devices=[0], rep_offset=g["config"]["rep"], histograms=True) as sim:
            sim.run()
            h = _hists(pkg, sim, 0)
            _identities(pkg, h, sim.stats_all()[0])
        if g["variant"] == "b":
            h.pop(pkg.HIST_FAIL)                             # RandomAccessSimulatorBeta.c has no failCount column
        _assert_equal(h, _expected(pkg, p, rows.astype(np.int64), g["variant"]), name)


def test_every_kernel_instantiation(pkg, oracle, monkeypatch):
    """the cases of test_gpu_parity.test_every_kernel_instantiation, under every block shape and point view, with and
    without the per-UE dump: the histogram is the oracle's, and the counters are those of the run without histograms"""
    cases = [dict(nUE=6000, seed=11, rep=3), dict(nUE=2500, nPreamble=64, backoffIndicator=40, nGrantUL=4, seed=12),
             dict(nUE=3000, distribution=1, nPreamble=3, maxRarWindow=9, accessTime=7, seed=13, geometry=1),
             dict(nUE=9000, maxMsg2TxCount=49, nGrantUL=3, seed=15), dict(nUE=4000, distribution=1, seed=16, geometry=0)]
    for kw in cases:
        _, rows, _ = oracle.run_port(oracle.make_config(**kw))
        p = _params(pkg, kw, "w")
        exp = _expected(pkg, p, rows.astype(np.int64), "w")
        for shape in ("huge", "big", "small"):
            for fixed in ("1", "0"):
                monkeypatch.setenv("RACH_BLOCK", shape)
                monkeypatch.setenv("RACH_FIXED", fixed)
                for dump in (True, False):
                    out = []
                    for hist in (True, False):
                        with pkg.RachSim([p], reps=1, devices=[0], rep_offset=kw.get("rep", 0), dump_ues=dump,
                                         histograms=hist) as sim:
                            sim.run()
                            out.append(sim.stats(0, 0).as_dict())
                            if hist:
                                _assert_equal(_hists(pkg, sim, 0), exp, "%s %s %s %s" % (shape, fixed, dump, kw))
                    assert out[0] == out[1], (shape, fixed, dump, kw)
    monkeypatch.delenv("RACH_BLOCK")
    monkeypatch.delenv("RACH_FIXED")


def test_sums_over_replications_and_devices(pkg):
    pts = [pkg.default_params(nUE=5000, seed=5), pkg.default_params(nUE=3000, seed=6, nGrantUL=3, distribution=1)]
    reps = 24
    with pkg.RachSim(pts, reps=reps, devices=[0], rep_offset=2, dump_ues=True, histograms=True) as sim:
        sim.run()
        ref = [_hists(pkg, sim, k) for k in range(2)]
        stats = sim.stats_all()
        for k, p in enumerate(pts):
            exp = None
            for r in range(reps):
                e = _expected(pkg, p, sim.dump_ues(k, r).astype(np.int64), "w")
                exp = e if exp is None else {kind: exp[kind] + e[kind] for kind in e}
            _assert_equal(ref[k], exp, "point %d" % k)
            _identities(pkg, ref[k], stats[k])
        sim.run()                                            # a second run starts from zero
        for k in range(2):
            _assert_equal(_hists(pkg, sim, k), ref[k], "second run")
    for kw in (dict(devices=[0]), dict(devices=[0, 0, 0, 0]), dict(devices=[0], ctas_per_sm=1)):
        with pkg.RachSim(pts, reps=reps, rep_offset=2, histograms=True, **kw) as sim:
            sim.run()
            for k in range(2):
                _assert_equal(_hists(pkg, sim, k), ref[k], str(kw))


def test_streaming_run(pkg):
    pts = [pkg.default_params(nUE=4000, seed=8), pkg.default_params(nUE=2000, seed=9, nPreamble=8)]
    with pkg.RachSim(pts, reps=6, devices=[0, 0], dump_ues=True, histograms=True) as sim:
        sim.run()
        a = [_hists(pkg, sim, k) for k in range(2)]
        sim.run_stream(lambda point, rep, st, rows: None)
        for k in range(2):
            _assert_equal(_hists(pkg, sim, k), a[k], "point %d" % k)


def test_noma_cell_radii(pkg, oracle):
    radii = (100.0, 500.0, 1500.0)
    pts = [pkg.default_params(variant=2, nUE=6000, seed=77, cellRadius=r) for r in radii]
    with pkg.RachSim(pts, reps=3, devices=[0], rep_offset=4, dump_ues=True, histograms=True) as sim:
        sim.run()
        stats = sim.stats_all()
        for k, (r, p) in enumerate(zip(radii, pts)):
            h = _hists(pkg, sim, k)
            exp = None
            for rep in range(3):
                _, rows, _ = oracle.run_port_n(oracle.make_config_n(nUE=6000, seed=77, cellRadius=r, rep=4 + rep))
                e = _expected(pkg, p, rows.astype(np.int64), "n")
                exp = e if exp is None else {kind: exp[kind] + e[kind] for kind in e}
            _assert_equal(h, exp, str(r))
            _identities(pkg, h, stats[k])


def test_legacy_u0_warp_and_serial(pkg, oracle, monkeypatch):
    cases = [dict(nUE=9000, seed=21), dict(nUE=250000, nPreamble=64, backoffIndicator=2, seed=22),
             dict(nUE=30000, nPreamble=1, seed=23)]
    pts, exps = [], []
    for kw in cases:
        p = pkg.default_params(variant=1, **kw)
        p.maxTimeMs = 5000
        _, rows = oracle.run_port_u0(oracle.make_config_u0(stopMs=5000, **kw))
        pts.append(p)
        exps.append(_expected(pkg, p, rows.astype(np.int64), "u0"))
    for mode in ("warp", "serial"):
        monkeypatch.setenv("RACH_U0", mode)
        for dump in (False, True):
            with pkg.RachSim(pts, reps=1, devices=[0], dump_ues=dump, histograms=True) as sim:
                sim.run()
                for k in range(len(cases)):
                    _assert_equal(_hists(pkg, sim, k), exps[k], "%s %s" % (mode, cases[k]))
    monkeypatch.delenv("RACH_U0")


@pytest.mark.parametrize("dist,reps", [(2, 64), (1, 16)])
def test_headline_size(pkg, dist, reps):
    p = pkg.default_params(nUE=100000, distribution=dist, seed=0)
    with pkg.RachSim([p], reps=reps, histograms=True) as sim:
        sim.run()
        h = _hists(pkg, sim, 0)
        _identities(pkg, h, sim.stats_all()[0])
    assert h[pkg.HIST_DELAY][-1] == 0                       # the delay bound holds: the clamp never engaged


def test_error_paths(pkg):
    p = pkg.default_params(nUE=500, seed=1)
    with pkg.RachSim([p], reps=2, histograms=True) as sim:
        with pytest.raises(pkg.RachError, match="error -5"):          # RA_E_STATE: before a run
            sim.histogram(0, pkg.HIST_DELAY)
        sim.run()
        for point, kind in ((0, 3), (0, -1), (1, pkg.HIST_TX), (-1, pkg.HIST_TX)):
            with pytest.raises(pkg.RachError, match="error -1"):      # RA_E_INVAL
                sim.histogram(point, kind)
    with pkg.RachSim([p], reps=2) as sim:
        sim.run()
        with pytest.raises(pkg.RachError, match="error -5"):          # without the option
            sim.histogram(0, pkg.HIST_DELAY)
    for variant in (1, 2):
        q = pkg.default_params(variant=variant, nUE=500, seed=1)
        with pkg.RachSim([q], reps=1, histograms=True) as sim:
            sim.run()
            sim.histogram(0, pkg.HIST_TX)
            with pytest.raises(pkg.RachError, match="error -1"):      # no failCount in N or U0
                sim.histogram(0, pkg.HIST_FAIL)


def _read_csv(path):
    rows = open(path).read().splitlines()
    assert rows[0] == "metric,value,count"
    out = {}
    for r in rows[1:]:
        m, v, c = r.split(",")
        assert int(c) > 0
        out.setdefault(m, {})[int(v)] = int(c)
    return out


def _nonzero(h):
    return {int(v): int(c) for v, c in enumerate(h) if c}


def test_cli_distributions(pkg, tmp_path):
    exe = pkg.build_host()
    nues = (3000, 20000)
    out = tmp_path / "w"
    subprocess.run([exe, "--hist", "-t", "3", "--nue", ",".join(map(str, nues)), "--no-logs", "--outdir", str(out)],
                   check=True, capture_output=True)
    pts = [pkg.default_params(nUE=n) for n in nues]
    with pkg.RachSim(pts, reps=3, histograms=True) as sim:
        sim.run()
        for k, n in enumerate(nues):
            got = _read_csv(out / "NomaBetaResults" / ("54_%d_Distributions.csv" % n))
            assert got == {"delay_ms": _nonzero(sim.histogram(k, pkg.HIST_DELAY)),
                           "preamble_tx": _nonzero(sim.histogram(k, pkg.HIST_TX)),
                           "fail_count": _nonzero(sim.histogram(k, pkg.HIST_FAIL))}
    for fmt, sub, metrics in (("b", "BasicBetaSimulationResults", {"delay_ms", "preamble_tx"}),
                              ("n", "TestResults", {"delay_ms", "preamble_tx"}),
                              ("u", "2_SimulationResults", {"delay_ms", "preamble_tx"})):
        d = tmp_path / fmt
        subprocess.run([exe, "--hist", "--format", fmt, "--nue", "3000", "--no-logs", "--outdir", str(d)],
                       check=True, capture_output=True)
        p = 64 if fmt == "u" else 54
        got = _read_csv(d / sub / ("%d_3000_Distributions.csv" % p))
        assert set(got) == metrics, fmt
        assert sum(got["delay_ms"].values()) == sum(got["preamble_tx"].values()) > 0
    d = tmp_path / "plain"
    subprocess.run([exe, "--nue", "3000", "--no-logs", "--outdir", str(d)], check=True, capture_output=True)
    assert not [f for _, _, fs in os.walk(d) for f in fs if f.endswith("_Distributions.csv")]


def test_fuzz_against_oracle(pkg, oracle):
    """mixed points of one launch, against the oracle's rows"""
    rnd = random.Random(4243)
    cases = []
    for _ in range(12):
        cases.append(dict(nUE=rnd.choice([1, 7, 300, 1500, 4000]), nPreamble=rnd.choice([2, 8, 54, 64]),
                          backoffIndicator=rnd.choice([1, 5, 20, 40]), nGrantUL=rnd.choice([1, 4, 12]),
                          maxRarWindow=rnd.choice([2, 6, 9]), maxMsg2TxCount=rnd.choice([0, 3, 9, 19]),
                          accessTime=rnd.choice([1, 5, 7]), seed=rnd.getrandbits(60), geometry=rnd.choice([0, 1]),
                          stopMs=rnd.choice([0, 777, 3001])))
    pts = [_params(pkg, kw, "w") for kw in cases]
    with pkg.RachSim(pts, reps=1, devices=[0], rep_offset=9, histograms=True) as sim:
        sim.run()
        for k, kw in enumerate(cases):
            _, rows, _ = oracle.run_port(oracle.make_config(rep=9, **kw))
            _assert_equal(_hists(pkg, sim, k), _expected(pkg, pts[k], rows.astype(np.int64), "w"), str(kw))
