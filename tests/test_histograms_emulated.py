"""Histograms of the successful UEs (ra_options.histograms, ra_hist_add in rach_core.cuh) on the host emulation of the
engine's phases (tests/emu/rach_emu.cpp, run through tests/emu/rach_emu_hist.cpp with a histogram region): the region is
compared with np.bincount over the oracle's per-UE rows, for W/B, N and U0, and with the counters of the same run.  The
-m gpu file test_gpu_histograms.py checks the kernels."""
import ctypes as C
import importlib
import os
import random
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOP = 256


@pytest.fixture(scope="module")
def emu(oracle, tmp_path_factory):
    so = str(tmp_path_factory.mktemp("emu_hist") / "librach_emu_hist.so")
    subprocess.check_call(["g++", "-O2", "-fPIC", "-shared", "-std=c++17",
                           "-I", os.path.join(ROOT, "include"), "-I", os.path.join(ROOT, "oracle"),
                           "-I", os.path.join(ROOT, "5g-nr-randomaccess_b200", "csrc"),
                           "-I", os.path.join(ROOT, "tests", "emu"),
                           os.path.join(ROOT, "tests", "emu", "rach_emu_hist.cpp"),
                           os.path.join(ROOT, "5g-nr-randomaccess_b200", "csrc", "rach_host.cpp"), "-o", so])
    lib = C.CDLL(so)
    lib.emu_hist_data.restype = C.POINTER(C.c_uint)
    lib.emu_hist_arm.argtypes = [C.c_int]

    class Emu:
        w = oracle._lib(so, "emu_run")
        n = oracle._lib(so, "emu_run_n")
        u0 = oracle._lib(so, "emu_run_u0")
        threads = C.c_int.in_dll(lib, "emu_threads")
        fixed = C.c_int.in_dll(lib, "emu_use_fixed")
        light = C.c_int.in_dll(lib, "emu_light")
        u0_mode = C.c_int.in_dll(lib, "emu_u0_mode")

        @staticmethod
        def arm(horizon):
            """a zeroed region for the next run of a point with this horizon"""
            lib.emu_hist_arm(lib.emu_hist_len(horizon))

        @staticmethod
        def region(horizon):
            n = lib.emu_hist_len(horizon)
            return np.ctypeslib.as_array(lib.emu_hist_data(), shape=(n,)).astype(np.int64)
    yield Emu
    Emu.threads.value, Emu.fixed.value, Emu.light.value, Emu.u0_mode.value = 64, 1, 1, 1


def _horizon(cfg, variant="w"):
    if cfg.stopMs > 0 and variant != "n":
        return cfg.stopMs
    return 60000 if cfg.distribution == 1 else 10000


def _split(region, horizon):
    """delay [horizon + 7], tx [256], fail [256] (the layout of ra_hist_add)"""
    nd = horizon + 7
    assert region.shape == (nd + 2 * TOP,)
    return region[:nd], region[nd:nd + TOP], region[nd + TOP:]


def _bincount(values, n):
    return np.bincount(np.minimum(values, n - 1), minlength=n)


def _check(region, horizon, rows, res, done, timer, tx, fail=None):
    """region against the bincounts of the successful rows, and the identities with the run's counters"""
    delay_h, tx_h, fail_h = _split(region, horizon)
    ok = rows[:, done] == 1
    np.testing.assert_array_equal(delay_h, _bincount(rows[ok, timer], horizon + 7))
    np.testing.assert_array_equal(tx_h, _bincount(rows[ok, tx], TOP))
    if fail is not None:
        np.testing.assert_array_equal(fail_h, _bincount(rows[ok, fail], TOP))
    for h in (delay_h, tx_h) + ((fail_h,) if fail is not None else ()):
        assert h.sum() == res.nSuccess
    assert (np.arange(horizon + 7) * delay_h).sum() == res.delaySum
    if tx_h[-1] == 0:
        assert (np.arange(TOP) * tx_h).sum() == res.preambleTxSum
    if fail is not None and fail_h[-1] == 0:
        assert (np.arange(TOP) * fail_h).sum() == res.failCountSum
    return delay_h, tx_h, fail_h


def _w(oracle, emu, kw):
    cfg = oracle.make_config(**kw)
    _, rows, _ = oracle.run_port(cfg)
    emu.arm(_horizon(cfg))
    res, _, _ = oracle._run(emu.w, cfg, False, False)
    return _check(emu.region(_horizon(cfg)), _horizon(cfg), rows, res, 13, 0, 10, 14)


def test_w_point_views_and_thread_counts(oracle, emu):
    for kw in (dict(nUE=10000, seed=1, rep=2), dict(nUE=3000, distribution=1, seed=3),
               dict(nUE=4000, nPreamble=8, nGrantUL=2, maxMsg2TxCount=49, seed=4),     # failCount and tx well above 0
               dict(nUE=2000, geometry=0, nGrantUL=54, seed=5)):                      # B
        for fixed in (1, 0):
            for threads in (1, 32, 256):
                emu.fixed.value, emu.threads.value = fixed, threads
                _w(oracle, emu, kw)
    emu.fixed.value = 1


def test_w_light_path_on_and_off(oracle, emu):
    emu.threads.value = 128
    for kw in (dict(nUE=20000, distribution=1, seed=3, stopMs=20000), dict(nUE=10000, seed=4)):
        got = []
        for light in (1, 0):
            emu.light.value = light
            got.append(_w(oracle, emu, kw))
        emu.light.value = 1
        for a, b in zip(*got):
            np.testing.assert_array_equal(a, b)


def test_w_fuzz(oracle, emu):
    """cases built as test_engine_emulated.test_fuzz builds them, horizons cut by stopMs included"""
    rnd = random.Random(1907)
    top_tx = 0
    for _ in range(20):
        kw = dict(nUE=rnd.choice([1, 2, 7, 50, 300, 1500, 4000]),
                  distribution=rnd.choice([1, 2, 2, 2]),
                  nPreamble=rnd.choice([1, 2, 3, 8, 54, 64]),
                  backoffIndicator=rnd.choice([1, 2, 5, 20, 40]),
                  nGrantUL=rnd.choice([1, 2, 4, 12, 54]),
                  maxRarWindow=rnd.choice([2, 3, 6, 6, 9]),
                  maxMsg2TxCount=rnd.choice([0, 1, 3, 9, 19]),
                  accessTime=rnd.choice([1, 2, 3, 5, 5, 5, 6, 7, 10]),
                  seed=rnd.getrandbits(64), rep=rnd.randrange(5000),
                  geometry=rnd.choice([0, 1]), stopMs=rnd.choice([0, 0, 0, 777, 3001]))
        emu.threads.value = rnd.choice([1, 32, 256])
        _, tx_h, _ = _w(oracle, emu, kw)
        top_tx = max(top_tx, int(np.nonzero(tx_h)[0].max()) if tx_h.any() else 0)
    assert top_tx >= 3


def test_w_lone_ue_known_answer(oracle, emu, golden):
    """one UE alone: the 18 ms handshake of the reference's timing diagram, first preamble answered"""
    stats, _ = golden
    delay_h, tx_h, fail_h = _w(oracle, emu, {k: v for k, v in stats["w_lone_ue"]["config"].items()})
    assert delay_h.sum() == 1 and delay_h[18] == 1
    assert tx_h.sum() == 1 and tx_h[1] == 1
    assert fail_h.sum() == 1 and fail_h[0] == 1


def test_noma(oracle, emu):
    rnd = random.Random(52)
    cases = [dict(nUE=2000), dict(nUE=20000, seed=4), dict(nUE=8000, geometry=0, seed=6)]
    for _ in range(10):
        cases.append(dict(nUE=rnd.choice([1, 5, 300, 3000, 9000]), nPreamble=rnd.choice([1, 3, 54, 64]),
                          backoffIndicator=rnd.choice([1, 2, 20, 40]), nGrantUL=rnd.choice([1, 2, 4, 12]),
                          maxMsg2TxCount=rnd.choice([1, 3, 10]), accessTime=rnd.choice([5, 5, 6, 10]),
                          maxRarWindow=rnd.choice([3, 5]), cellRadius=rnd.choice([100.0, 500.0]),
                          seed=rnd.getrandbits(60), rep=rnd.randrange(1000), geometry=rnd.choice([0, 1, 1])))
    for kw in cases:
        cfg = oracle.make_config_n(**kw)
        _, rows, _ = oracle.run_port_n(cfg)
        emu.arm(_horizon(cfg, "n"))
        res, _, _ = oracle._run_n(emu.n, cfg)
        _check(emu.region(_horizon(cfg, "n")), _horizon(cfg, "n"), rows, res, 13, 0, 10)


def test_legacy_u0(oracle, emu):
    rnd = random.Random(9)
    cases = [dict(nUE=2000), dict(nUE=20000, seed=2), dict(nUE=40000, nPreamble=1, seed=3, stopMs=20000),
             dict(nUE=250000, nPreamble=64, backoffIndicator=2, seed=327613445147561757, rep=601, stopMs=6000)]
    for _ in range(8):
        cases.append(dict(nUE=rnd.choice([1, 2, 50, 400, 3000, 9000]), nPreamble=rnd.choice([1, 2, 3, 8, 64]),
                          backoffIndicator=rnd.choice([1, 2, 5, 20, 40]), seed=rnd.getrandbits(60),
                          rep=rnd.randrange(1000), stopMs=rnd.choice([0, 3000, 20000])))
    for kw in cases:
        cfg = oracle.make_config_u0(**kw)
        _, rows = oracle.run_port_u0(cfg)
        for mode in (1, 0):
            emu.u0_mode.value = mode
            emu.arm(_horizon(cfg))
            res, _, _ = oracle._run(emu.u0, cfg, False, False)
            _check(emu.region(_horizon(cfg)), _horizon(cfg), rows, res, 10, 0, 7)
    emu.u0_mode.value = 1


def test_hist_bins_host_helper():
    pkg = importlib.import_module("5g-nr-randomaccess_b200")
    pkg.build_lib()
    w = pkg.default_params(nUE=1000)
    assert pkg.hist_bins(w, pkg.HIST_DELAY) == 10000 + 7
    w.maxTimeMs = 777
    assert pkg.hist_bins(w, pkg.HIST_DELAY) == 777 + 7
    assert pkg.hist_bins(w, pkg.HIST_TX) == 256 and pkg.hist_bins(w, pkg.HIST_FAIL) == 256
    assert pkg.hist_bins(w, 3) == -1 and pkg.hist_bins(w, -1) == -1
    u0 = pkg.default_params(variant=1)
    n = pkg.default_params(variant=2)
    assert pkg.hist_bins(u0, pkg.HIST_DELAY) == 60000 + 7 and pkg.hist_bins(n, pkg.HIST_DELAY) == 10000 + 7
    for p in (u0, n):
        assert pkg.hist_bins(p, pkg.HIST_TX) == 256
        assert pkg.hist_bins(p, pkg.HIST_FAIL) == -1          # RA_E_INVAL: no failCount in N or U0
