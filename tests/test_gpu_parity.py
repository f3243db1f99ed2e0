"""GPU parity: librach_gpu (CUDA, through the C ABI) against the oracle restatement, the reference
sources in tape mode (oracle/_ref, prebuilt) and the committed reference fixtures."""
import hashlib
import importlib
import random

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

KEYS = ["simTimeMs", "nSuccess", "preambleTxSum", "delaySum", "failCountSum", "continueFailed",
        "collisionPreambles", "totalPreambleTxop", "collisionScans", "totalScans"]


@pytest.fixture(scope="module")
def pkg():
    p = importlib.import_module("5g-nr-randomaccess_b200")
    p.load_lib()
    return p


def _params(pkg, cfg_kw):
    kw = dict(cfg_kw)
    rep = kw.pop("rep", 0)
    stop = kw.pop("stopMs", 0)
    for k in ("useTape", "echo"):
        kw.pop(k, None)
    p = pkg.default_params(**kw)
    if stop:
        p.maxTimeMs = stop
    return p, rep


def _run_gpu(pkg, cfg_kw, dump=True):
    p, rep = _params(pkg, cfg_kw)
    with pkg.RachSim([p], reps=1, devices=[0], rep_offset=rep, dump_ues=dump) as sim:
        sim.run()
        st = sim.stats(0, 0)
        ue = sim.dump_ues(0, 0) if dump else None
        geom = sim.geometry(0, 0) if (dump and p.geometry) else None
    return st, ue, geom


def test_fixtures_from_the_reference(pkg, golden):
    stats, ues = golden
    for name, g in stats.items():
        if g["variant"] in ("n", "u0"):
            continue
        st, ue, geom = _run_gpu(pkg, g["config"])
        keys = KEYS[:8] if g["variant"] == "w" else ["simTimeMs", "nSuccess", "preambleTxSum", "delaySum", "collisionScans", "totalScans"]
        for k in keys:
            assert getattr(st, k) == g["stats"][k], (name, k)
        if g["variant"] == "b":
            ue[:, 14] = 0
            ue[:, 15] = -1
        assert hashlib.sha256(np.ascontiguousarray(ue).tobytes()).hexdigest() == g["ue_sha256"], name
        if name in ues:
            np.testing.assert_array_equal(ue, ues[name].astype(np.int32))


def test_geometry_side_outputs(pkg, oracle):
    """W:392-415: fp64 libm results rounded to float; tolerance 1e-6 relative on the float
    outputs (CUDA's double cos/sin/log10 are within 1-2 ulp of glibc's before rounding), and
    ZERO sector flips."""
    cfg = oracle.make_config(nUE=20000, seed=9, rep=4, cellRadius=400.0)
    _, _, g_ref = oracle.run_port(cfg, geom=True)
    _, _, g = _run_gpu(pkg, dict(nUE=20000, seed=9, rep=4, cellRadius=400.0))
    assert np.array_equal(g[:, 5], g_ref[:, 5])
    assert np.array_equal(g[:, 0], g_ref[:, 0]) and np.array_equal(g[:, 3], g_ref[:, 3])
    np.testing.assert_allclose(g[:, [1, 2, 4]], g_ref[:, [1, 2, 4]], rtol=1e-6, atol=1e-4)
    exact = (g.view(np.uint32) == g_ref.view(np.uint32)).mean()
    assert exact > 0.999


def test_fuzz_against_oracle(pkg, oracle):
    rnd = random.Random(4242)
    for _ in range(40):
        kw = dict(nUE=rnd.choice([1, 2, 7, 50, 300, 1500, 4000, 9000]),
                  distribution=rnd.choice([1, 2, 2, 2]),
                  nPreamble=rnd.choice([1, 2, 3, 8, 54, 64]),
                  backoffIndicator=rnd.choice([1, 2, 5, 20, 40]),
                  nGrantUL=rnd.choice([1, 2, 4, 12, 54]),
                  maxRarWindow=rnd.choice([2, 3, 6, 6, 9]),
                  maxMsg2TxCount=rnd.choice([0, 1, 3, 9, 19]),
                  accessTime=rnd.choice([1, 2, 3, 5, 5, 5, 6, 7, 10]),
                  seed=rnd.getrandbits(64), rep=rnd.randrange(5000),
                  geometry=rnd.choice([0, 1]), stopMs=rnd.choice([0, 0, 0, 777, 3001]))
        if kw["distribution"] == 1 and kw["nUE"] > 4000:
            kw["nUE"] = 4000
        cfg = oracle.make_config(**kw)
        res, ue_ref, _ = oracle.run_port(cfg)
        st, ue, _ = _run_gpu(pkg, kw)
        for k in KEYS:
            assert getattr(st, k) == getattr(res, k), (k, kw)
        np.testing.assert_array_equal(ue, ue_ref, err_msg=str(kw))


def test_every_kernel_instantiation(pkg, oracle, monkeypatch):
    """The W step kernel has three block shapes (128 x 8, 256 x 5, 512 x 2 threads x blocks/SM, picked by table size and
    by how many replications there are per SM; RACH_BLOCK forces one) and two views of the parameter point (the
    reference's default family P 54 / BI 20 / subframe 5 / RAR window 5 as compile-time immediates, or runtime values;
    RACH_FIXED=0 forces the runtime view).  Every combination must reproduce the oracle, with and without the per-UE
    dump."""
    cases = [dict(nUE=6000, seed=11, rep=3), dict(nUE=2500, nPreamble=64, backoffIndicator=40, nGrantUL=4, seed=12),
             dict(nUE=3000, distribution=1, nPreamble=3, maxRarWindow=9, accessTime=7, seed=13, geometry=1),
             dict(nUE=9000, maxMsg2TxCount=49, nGrantUL=3, seed=15), dict(nUE=4000, distribution=1, seed=16, geometry=0)]
    for kw in cases:
        res, ue_ref, _ = oracle.run_port(oracle.make_config(**kw))
        for shape in ("huge", "big", "small"):
            for fixed in ("1", "0"):
                monkeypatch.setenv("RACH_BLOCK", shape)
                monkeypatch.setenv("RACH_FIXED", fixed)
                st, ue, _ = _run_gpu(pkg, kw)
                st2, _, _ = _run_gpu(pkg, kw, dump=False)
                for k in KEYS:
                    assert getattr(st, k) == getattr(res, k) == getattr(st2, k), (k, shape, fixed, kw)
                np.testing.assert_array_equal(ue, ue_ref, err_msg="%s %s %s" % (shape, fixed, kw))
    monkeypatch.delenv("RACH_BLOCK")
    monkeypatch.delenv("RACH_FIXED")
    # a point whose tables do not fit 8 times in one SM takes a larger shape by itself
    kw = dict(nUE=4000, nPreamble=64, backoffIndicator=100, seed=14)
    res, ue_ref, _ = oracle.run_port(oracle.make_config(**kw))
    st, ue, _ = _run_gpu(pkg, kw)
    for k in KEYS:
        assert getattr(st, k) == getattr(res, k), (k, kw)
    np.testing.assert_array_equal(ue, ue_ref)


def test_shape_follows_the_job_count(pkg, oracle):
    """Default-family points under load (at least 24 arrivals per occasion at the peak), enough replications for every
    automatic shape choice: 1 per SM (512-thread blocks), 4 per SM (256), 9+ per SM (128).  Same tape ids -> the same
    per-replication counters whatever the shape."""
    p = pkg.default_params(nUE=24000, seed=21)
    ref = None
    for reps in (1400, 600, 100):
        with pkg.RachSim([p], reps=reps, devices=[0], rep_offset=50) as sim:
            sim.run()
            st = sim.stats_all()[0]
        if ref is None:
            ref = st
            for rep in (0, 777, 1399):
                res, _, _ = oracle.run_port(oracle.make_config(nUE=24000, seed=21, rep=50 + rep), per_ue=False)
                for k in KEYS:
                    assert int(st[rep][k]) == getattr(res, k), (rep, k)
        assert (st == ref[:reps]).all(), reps


def test_against_reference_sources_in_tape_mode(pkg, oracle, recorded):
    """Against the tape-mode reference build where it exists, and always against the stored digest of the engine's
    output on the same case (how it was recorded: tests/conftest.py, Recorded)."""
    kw = dict(nUE=8000, seed=31, rep=17)
    st, ue, _ = _run_gpu(pkg, kw)
    recorded.check("gpu_tape_mode_w", recorded.digest(config=kw, ue=ue, **{k: getattr(st, k) for k in KEYS[:8]}))
    if not oracle.ref_available("w"):
        return
    r, ue_ref, _ = oracle.run_ref("w", oracle.make_config(**kw))
    for k in KEYS[:8]:
        assert getattr(st, k) == getattr(r, k), k
    np.testing.assert_array_equal(ue, ue_ref)


def test_full_size_100k_beta(pkg, oracle):
    """BASELINE headline size: one 100k-UE Beta replication, every UE and every counter."""
    kw = dict(nUE=100000, seed=2, rep=5)
    res, ue_ref, _ = oracle.run_port(oracle.make_config(**kw))
    st, ue, _ = _run_gpu(pkg, kw)
    for k in KEYS:
        assert getattr(st, k) == getattr(res, k), k
    np.testing.assert_array_equal(ue, ue_ref)
    assert st.simTimeMs == 10000 and 18000 < st.nSuccess < 20000     # README.md:97: 18.99 %


def test_the_bench_batch_itself(pkg, golden):
    """The headline workload as bench.py launches it (100k UEs x 4096 replications, seed 0, replication ids 0..4095), checked
    through what does not need a CPU run per replication: replication 0 IS the reference's own 100 000-UE run (fixture
    w_default_100000, generated by RandomAccessWithNOMA.c itself in tape mode); a second launch gives the same 4096 x 12
    counters bit for bit (no result depends on the order of atomics or on which block ran what); a 40-replication launch
    reproduces its slice; nobody finishes early, so the update count is exactly nUE x 2000 per replication; and the batch
    means sit on the README row (README.md:97)."""
    stats, _ = golden
    g = stats["w_default_100000"]
    p = pkg.default_params(nUE=100000, seed=0)
    with pkg.RachSim([p], reps=4096, devices=[0]) as sim:
        sim.run()
        a = sim.stats_all().copy()
        sim.run()
        b = sim.stats_all().copy()
    assert (a == b).all()
    for k in KEYS[:8]:
        assert int(a[0, 0][k]) == g["stats"][k], k
    with pkg.RachSim([p], reps=40, devices=[0], rep_offset=1000) as sim:
        sim.run()
        assert (sim.stats_all()[0] == a[0, 1000:1040]).all()
    assert (a["simTimeMs"] == 10000).all() and (a["updates"] == 100000 * 2000).all()
    ns = a["nSuccess"].astype(np.float64)
    assert abs(100.0 * ns.mean() / 100000 - 18.989) < 0.05
    assert abs(a["preambleTxSum"].sum() / ns.sum() - 5.76) < 0.02 and abs(a["delaySum"].sum() / ns.sum() - 96.001) < 0.3


def test_full_size_100k_uniform(pkg, oracle):
    """BASELINE configs[1]: Uniform 60 s, 100k UEs."""
    kw = dict(nUE=100000, distribution=1, seed=3, rep=1)
    res, ue_ref, _ = oracle.run_port(oracle.make_config(**kw))
    st, ue, _ = _run_gpu(pkg, kw)
    for k in KEYS:
        assert getattr(st, k) == getattr(res, k), k
    np.testing.assert_array_equal(ue, ue_ref)
    assert st.nSuccess == 100000 and st.simTimeMs < 60000


def test_beyond_the_reference_sweep_300k(pkg, oracle):
    """Three times the largest size the reference sweeps (W:221), 64 preambles / 16 grants / BI 40 (the corner of
    BASELINE configs[4]): every UE and every counter."""
    kw = dict(nUE=300000, nPreamble=64, nGrantUL=16, backoffIndicator=40, seed=11, rep=2)
    res, ue_ref, _ = oracle.run_port(oracle.make_config(**kw))
    st, ue, _ = _run_gpu(pkg, kw)
    for k in KEYS:
        assert getattr(st, k) == getattr(res, k), k
    np.testing.assert_array_equal(ue, ue_ref)


def test_batch_is_placement_invariant(pkg, oracle):
    """Many replications and two parameter points in one launch == each alone (keyed tape);
    dump on/off and the CTAs-per-SM setting do not change any counter."""
    pa = pkg.default_params(nUE=3000, seed=5)
    pb = pkg.default_params(nUE=1200, seed=6, nPreamble=8, nGrantUL=3)
    with pkg.RachSim([pa, pb], reps=24, devices=[0], rep_offset=100) as sim:
        sim.run()
        allst = sim.stats_all()
    with pkg.RachSim([pa, pb], reps=24, devices=[0], rep_offset=100, dump_ues=True, ctas_per_sm=1) as sim:
        sim.run()
        assert (sim.stats_all() == allst).all()
    for point, kw in ((0, dict(nUE=3000, seed=5)), (1, dict(nUE=1200, seed=6, nPreamble=8, nGrantUL=3))):
        for rep in (0, 7, 23):
            res, _, _ = oracle.run_port(oracle.make_config(rep=100 + rep, **kw), per_ue=False)
            for k in KEYS:
                assert int(allst[point, rep][k]) == getattr(res, k), (point, rep, k)
    assert len({int(x) for x in allst[0]["delaySum"]}) > 20      # replications really differ


def test_streamed_dumps_equal_the_blocking_ones(pkg):
    """ra_sim_run_stream (per-UE logs at scale, the role of saveResult W:797-825): every replication is delivered exactly
    once, while the kernel runs, with the rows ra_sim_dump_ues returns afterwards -- for all three engines."""
    for variant, pts, reps in ((0, [pkg.default_params(nUE=6000, seed=3), pkg.default_params(nUE=2500, seed=4, nPreamble=8)], 300),
                               (2, [pkg.default_params(variant=2, nUE=5000, seed=5)], 64),
                               (1, [pkg.default_params(variant=1, nUE=20000, seed=6)], 40)):
        got = {}

        def on_rep(point, rep, st, rows):
            assert (point, rep) not in got
            got[(point, rep)] = (st, rows)
        with pkg.RachSim(pts, reps=reps, devices=[0], rep_offset=9, dump_ues=True) as sim:
            sim.run_stream(on_rep)
            assert len(got) == len(pts) * reps
            allst = sim.stats_all()
            for (point, rep) in [(0, 0), (len(pts) - 1, reps - 1), (0, reps // 2)]:
                st, rows = got[(point, rep)]
                np.testing.assert_array_equal(rows, sim.dump_ues(point, rep))
                for k in ("simTimeMs", "nSuccess", "preambleTxSum", "delaySum"):
                    assert st[k] == int(allst[point, rep][k]), (variant, k)
            first = sim.stats_all().copy()
            sim.run()                                   # the plain run after a streamed one gives the same counters
            assert (sim.stats_all() == first).all()


def test_error_paths(pkg):
    with pytest.raises(pkg.RachError, match="nPreamble"):
        pkg.RachSim([pkg.default_params(nPreamble=0)], reps=1)
    with pytest.raises(pkg.RachError, match="variant"):
        pkg.RachSim([pkg.default_params(variant=7)], reps=1)
    with pkg.RachSim([pkg.default_params(nUE=10)], reps=1) as sim:
        with pytest.raises(pkg.RachError, match="before ra_sim_run"):
            sim.stats(0, 0)
        sim.run()
        with pytest.raises(pkg.RachError, match="dumpUEs"):
            sim.dump_ues(0, 0)
        with pytest.raises(pkg.RachError, match="out of range"):
            sim.stats(1, 0)


# ---------------------------------------------------------------------------------------------
# variant N (NOMA.c)
# ---------------------------------------------------------------------------------------------
def _run_gpu_n(pkg, kw):
    kw = dict(kw)
    rep = kw.pop("rep", 0)
    for k in ("useTape", "echo", "stopMs", "distribution", "hBS", "hUT"):
        kw.pop(k, None)
    p = pkg.default_params(variant=2, **kw)
    with pkg.RachSim([p], reps=1, devices=[0], rep_offset=rep, dump_ues=True) as sim:
        sim.run()
        return sim.stats(0, 0), sim.dump_ues(0, 0), sim.gains(0, 0)


def _check_gains(g, g_ref):
    """fp64 channel gains: CUDA log/cos/sin vs glibc are within an ulp or two before the float
    roundings of NOMA.c:176-186; tolerance 1e-9 relative (north_star), bit-equal for most."""
    np.testing.assert_allclose(g, g_ref, rtol=1e-9, atol=0)
    return float((g.view(np.uint64) == g_ref.view(np.uint64)).mean())


def test_noma_fixtures_from_the_reference(pkg, golden, oracle):
    stats, ues = golden
    for name, g in stats.items():
        if g["variant"] != "n":
            continue
        st, ue, gain = _run_gpu_n(pkg, g["config"])
        _, ue_ref, gain_ref = oracle.run_port_n(oracle.make_config(**g["config"]))
        assert st.nSuccess == g["stats"]["nSuccess"] and st.preambleTxSum == g["stats"]["preambleTxSum"]
        assert st.delaySum == g["stats"]["delaySum"] and st.continueFailed == g["dropped"]
        # zero decision flips: every integer outcome of every UE equals the reference's
        assert hashlib.sha256(np.ascontiguousarray(ue).tobytes()).hexdigest() == g["ue_sha256"], name
        assert _check_gains(gain, gain_ref) > 0.99


def test_noma_fuzz_against_oracle(pkg, oracle):
    rnd = random.Random(777)
    cases = [dict(nUE=50000, seed=8, rep=3)]            # BASELINE configs[3] size
    for _ in range(25):
        cases.append(dict(nUE=rnd.choice([1, 5, 300, 3000, 9000]), nPreamble=rnd.choice([1, 3, 54, 64]),
                          backoffIndicator=rnd.choice([1, 2, 20, 40]), nGrantUL=rnd.choice([1, 2, 4, 12]),
                          maxMsg2TxCount=rnd.choice([1, 3, 10]), accessTime=rnd.choice([5, 5, 6, 10]),
                          maxRarWindow=rnd.choice([3, 5]), cellRadius=rnd.choice([100.0, 500.0]),
                          seed=rnd.getrandbits(60), rep=rnd.randrange(1000), geometry=rnd.choice([0, 1, 1])))
    for kw in cases:
        res, ue_ref, g_ref = oracle.run_port_n(oracle.make_config_n(**kw))
        st, ue, g = _run_gpu_n(pkg, kw)
        assert (st.simTimeMs, st.nSuccess, st.preambleTxSum, st.delaySum) == \
               (res.simTimeMs, res.nSuccess, res.preambleTxSum, res.delaySum), kw
        np.testing.assert_array_equal(ue, ue_ref, err_msg=str(kw))
        _check_gains(g, g_ref)
        # the pairing test 10*log(h) - 10*log(l) > 15. (NOMA.c:276) is the one fp comparison that decides an integer
        # outcome, and CUDA's log is not glibc's: no comparison of the test set may sit within 1e-9 of the threshold
        # (the two logs differ by a few 1e-14 at these magnitudes), so no decision can flip
        if res.pairTests:
            assert res.minPairMargin > 1e-9, (kw, res.minPairMargin)


def test_noma_points_with_different_cell_radii(pkg, oracle):
    """One ra_sim, three N points that differ in cellRadius (NOMA.c:56 -> activeUE N:168): the radius is a
    per-point value on the device (it was taken from point 0 for the whole launch once)."""
    radii = (100.0, 500.0, 1500.0)
    pts = [pkg.default_params(variant=2, nUE=6000, seed=77, cellRadius=r) for r in radii]
    with pkg.RachSim(pts, reps=2, devices=[0], rep_offset=4, dump_ues=True) as sim:
        sim.run()
        outs = [(sim.stats(k, 1), sim.dump_ues(k, 1), sim.gains(k, 1)) for k in range(len(radii))]
    seen = set()
    for r, (st, ue, g) in zip(radii, outs):
        res, ue_ref, g_ref = oracle.run_port_n(oracle.make_config_n(nUE=6000, seed=77, cellRadius=r, rep=5))
        assert (st.nSuccess, st.preambleTxSum, st.delaySum) == (res.nSuccess, res.preambleTxSum, res.delaySum), r
        np.testing.assert_array_equal(ue, ue_ref, err_msg=str(r))
        _check_gains(g, g_ref)
        seen.add((st.nSuccess, st.delaySum))
    assert len(seen) == len(radii)          # the radius really changes the outcome


def test_noma_batch(pkg, oracle):
    p = pkg.default_params(variant=2, nUE=4000, seed=12)
    with pkg.RachSim([p], reps=40, devices=[0], rep_offset=7) as sim:
        sim.run()
        st = sim.stats_all()
    for rep in (0, 13, 39):
        res, _, _ = oracle.run_port_n(oracle.make_config_n(nUE=4000, seed=12, rep=7 + rep))
        assert int(st[0, rep]["nSuccess"]) == res.nSuccess and int(st[0, rep]["delaySum"]) == res.delaySum


def test_device_list_longer_than_the_job_list(pkg, oracle):
    """ra_sim_create(devices[]) with more device entries than replications (entries may repeat a device id: each entry is
    a shard with its own stream and workspace): the idle entries are skipped, the others give the usual results -- also
    through the streaming run."""
    p = pkg.default_params(nUE=4000, seed=8)
    got = {}
    with pkg.RachSim([p], reps=2, devices=[0, 0, 0, 0], rep_offset=3, dump_ues=True) as sim:
        sim.run_stream(lambda point, rep, st, rows: got.__setitem__(rep, rows))
        st = sim.stats_all()
        for rep in (0, 1):
            res, ue_ref, _ = oracle.run_port(oracle.make_config(nUE=4000, seed=8, rep=3 + rep))
            for k in KEYS:
                assert int(st[0, rep][k]) == getattr(res, k), (rep, k)
            np.testing.assert_array_equal(got[rep], ue_ref)
            np.testing.assert_array_equal(sim.dump_ues(0, rep), ue_ref)


def test_multi_device_in_one_process(pkg):
    """ra_sim_create(devices[]) shards one job list over several GPUs from a single host thread;
    results equal the single-device run (skipped on a 1-GPU box)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    pa = pkg.default_params(nUE=5000, seed=5)
    pb = pkg.default_params(nUE=2000, seed=6, nGrantUL=3)
    with pkg.RachSim([pa, pb], reps=16, devices=[0]) as sim:
        sim.run()
        one = sim.stats_all()
    with pkg.RachSim([pa, pb], reps=16, devices=[0, 1], dump_ues=True) as sim:
        sim.run()
        two = sim.stats_all()
        ue = sim.dump_ues(1, 15)
    assert (one == two).all()
    assert ue.shape == (2000, 16) and (ue[:, 13] == 1).sum() == int(two[1, 15]["nSuccess"])


# ---------------------------------------------------------------------------------------------
# variant U0 (RandomAccessSimulator.c)
# ---------------------------------------------------------------------------------------------
def test_legacy_u0_fixtures_and_fuzz(pkg, golden, oracle):
    """All cases are points of ONE launch (one GPU thread per replication), checked UE by UE."""
    stats, _ = golden
    rnd = random.Random(66)
    cases = [(n, {k: g["config"][k] for k in ("nUE", "nPreamble", "backoffIndicator", "seed")}, g["config"]["rep"], g)
             for n, g in stats.items() if g["variant"] == "u0"]
    rep = cases[0][2]
    assert all(c[2] == rep for c in cases)
    for _ in range(12):
        cases.append((None, dict(nUE=rnd.choice([1, 2, 50, 400, 3000, 9000, 24001]), nPreamble=rnd.choice([1, 2, 3, 8, 64]),
                                 backoffIndicator=rnd.choice([1, 2, 5, 20, 40]), seed=rnd.getrandbits(60)), rep, None))
    pts = [pkg.default_params(variant=1, **kw) for _, kw, _, _ in cases]
    with pkg.RachSim(pts, reps=1, devices=[0], rep_offset=rep, dump_ues=True) as sim:
        sim.run()
        for k, (name, kw, _, g) in enumerate(cases):
            st, ue = sim.stats(k, 0), sim.dump_ues(k, 0)
            res, ue_ref = oracle.run_port_u0(oracle.make_config_u0(rep=rep, **kw))
            for key in ("simTimeMs", "nSuccess", "preambleTxSum", "delaySum", "collisionPreambles", "totalPreambleTxop"):
                assert getattr(st, key) == getattr(res, key), (name, key, kw)
            np.testing.assert_array_equal(ue, ue_ref, err_msg=str(kw))
            if g is not None:
                assert hashlib.sha256(np.ascontiguousarray(ue).tobytes()).hexdigest() == g["ue_sha256"], name


def test_legacy_u0_batch_full_size(pkg, oracle):
    """RandomAccessSimulator.c as shipped at 100 000 UEs (9 arrivals per 5 ms, 64 preambles): 32 replications
    in one launch (one warp each); three of them checked UE by UE."""
    p = pkg.default_params(variant=1, nUE=100000, seed=4)
    with pkg.RachSim([p], reps=32, devices=[0], rep_offset=10, dump_ues=True) as sim:
        sim.run()
        st = sim.stats_all()
        dumps = {r: sim.dump_ues(0, r) for r in (0, 17, 31)}
    assert (st["nSuccess"] == 100000).all()
    for r, ue in dumps.items():
        res, ue_ref = oracle.run_port_u0(oracle.make_config_u0(nUE=100000, seed=4, rep=10 + r))
        assert int(st[0, r]["simTimeMs"]) == res.simTimeMs and int(st[0, r]["delaySum"]) == res.delaySum
        np.testing.assert_array_equal(ue, ue_ref)


def test_legacy_u0_serial_formulation_and_crowded_ms(pkg, oracle, monkeypatch):
    """U0 has two exact formulations of a ms (warp step: one lane per live UE; serial step: lane 0 walks the list,
    used for ms with more than 32 live UEs).  RACH_U0=serial forces the serial one everywhere; a 250 000-UE
    population (21 arrivals per 5 ms) mixes both; an overload with one preamble exercises the phantom calendar."""
    cases = [dict(nUE=9000, seed=21), dict(nUE=250000, nPreamble=64, backoffIndicator=2, seed=22),
             dict(nUE=30000, nPreamble=1, seed=23)]
    refs = []
    for kw in cases:
        p = pkg.default_params(variant=1, **kw)
        p.maxTimeMs = 5000
        refs.append((p, oracle.run_port_u0(oracle.make_config_u0(stopMs=5000, **kw))))
    for mode in ("warp", "serial"):
        monkeypatch.setenv("RACH_U0", mode)
        with pkg.RachSim([p for p, _ in refs], reps=1, devices=[0], dump_ues=True) as sim:
            sim.run()
            for k, (p, (res, ue_ref)) in enumerate(refs):
                st, ue = sim.stats(k, 0), sim.dump_ues(k, 0)
                for key in ("simTimeMs", "nSuccess", "preambleTxSum", "delaySum", "collisionPreambles", "totalPreambleTxop"):
                    assert getattr(st, key) == getattr(res, key), (mode, key, cases[k])
                np.testing.assert_array_equal(ue, ue_ref, err_msg="%s %s" % (mode, cases[k]))
