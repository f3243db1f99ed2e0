"""The CUDA engine's phase functions (5g-nr-randomaccess_b200/csrc/rach_core.cuh) compiled for the
host (tests/emu) and run thread by thread, against the oracle restatement and the reference
fixtures.  Proves the event-driven formulation exact on CPU; the -m gpu tests prove the kernel."""
import ctypes as C
import hashlib
import os
import random
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = ["simTimeMs", "nSuccess", "preambleTxSum", "delaySum", "failCountSum", "continueFailed",
        "collisionPreambles", "totalPreambleTxop", "collisionScans", "totalScans"]


@pytest.fixture(scope="module")
def emu(oracle):
    so = subprocess.check_output([os.path.join(ROOT, "tests", "emu", "build_emu.sh")]).decode().strip()
    f = oracle._lib(so, "emu_run")
    thr = C.c_int.in_dll(C.CDLL(so), "emu_threads")
    return f, thr


def _cmp(oracle, emu, kw, threads=64):
    f, thr = emu
    thr.value = threads
    cfg = oracle.make_config(**kw)
    p, ue, _ = oracle.run_port(cfg)
    e, ue2, _ = oracle._run(f, cfg, True, False)
    for k in KEYS:
        assert getattr(p, k) == getattr(e, k), (k, kw)
    np.testing.assert_array_equal(ue, ue2, err_msg=str(kw))
    return p


def test_defaults(oracle, emu):
    _cmp(oracle, emu, dict(nUE=10000, seed=1, rep=2))
    _cmp(oracle, emu, dict(nUE=20000, seed=5), threads=256)


def test_against_reference_fixtures(oracle, emu, golden):
    stats, _ = golden
    f, thr = emu
    thr.value = 128
    for name, g in stats.items():
        if g["variant"] != "w" or g["config"]["nUE"] > 10000:
            continue
        cfg = oracle.make_config(**g["config"])
        e, ue, _ = oracle._run(f, cfg, True, False)
        for k in KEYS[:8]:
            assert getattr(e, k) == g["stats"][k], (name, k)
        assert hashlib.sha256(np.ascontiguousarray(ue).tobytes()).hexdigest() == g["ue_sha256"], name


def test_fuzz(oracle, emu):
    rnd = random.Random(77)
    late = 0
    for _ in range(60):
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
        late += _cmp(oracle, emu, kw, threads=rnd.choice([1, 3, 32, 64, 256])).lateAbsorbed
    assert late > 0


def test_noma_variant_emulated(oracle, emu):
    """Variant N phases (rach_core_n.cuh) on the host against the N oracle, incl. fp64 gains."""
    so = os.path.join(ROOT, "tests", "emu", "_build", "librach_emu.so")
    f = oracle._lib(so, "emu_run_n")
    rnd = random.Random(31)
    cases = [dict(nUE=2000), dict(nUE=20000, seed=4)]
    for _ in range(40):
        cases.append(dict(nUE=rnd.choice([1, 5, 300, 3000, 9000]), nPreamble=rnd.choice([1, 3, 54, 64]),
                          backoffIndicator=rnd.choice([1, 2, 20, 40]), nGrantUL=rnd.choice([1, 2, 4, 12]),
                          maxMsg2TxCount=rnd.choice([1, 3, 10]), accessTime=rnd.choice([5, 5, 6, 10]),
                          maxRarWindow=rnd.choice([3, 5]), cellRadius=rnd.choice([100.0, 500.0]),
                          seed=rnd.getrandbits(60), rep=rnd.randrange(1000), geometry=rnd.choice([0, 1, 1])))
    # more singles than 32 lanes per sector (non-sector function with 200 preambles), many grants, tiny radius range
    cases += [dict(nUE=30000, nPreamble=200, nGrantUL=7, geometry=0, seed=5), dict(nUE=30000, nPreamble=256, nGrantUL=3, seed=6),
              dict(nUE=12000, nPreamble=100, nGrantUL=40, geometry=0, seed=7), dict(nUE=50000, seed=8, rep=3)]
    import ctypes
    serial_b = ctypes.c_int.in_dll(ctypes.CDLL(so), "emu_n_serialB")
    zomb = 0
    for kw in cases:
        cfg = oracle.make_config_n(**kw)
        p, ue, g = oracle.run_port_n(cfg)
        # the base-station decision of a sector in its two forms: one warp (the kernel's), one thread
        for mode in (0, 1):
            serial_b.value = mode
            e, ue2, g2 = oracle._run_n(f, cfg)
            for k in ("simTimeMs", "nSuccess", "preambleTxSum", "delaySum"):
                assert getattr(p, k) == getattr(e, k), (k, mode, kw)
            np.testing.assert_array_equal(ue, ue2, err_msg="%s mode %d" % (kw, mode))
            np.testing.assert_array_equal(g.view(np.uint64), g2.view(np.uint64))
        serial_b.value = 0
        zomb += int(((ue[:, 1] == 1) & (ue[:, 14] > 0) & (ue[:, 15] == 0) & (ue[:, 2] < p.simTimeMs - 100)).sum())
    assert zomb > 0      # restarts that can never transmit again (NOMA.c:538 + :692) were exercised


def test_legacy_variant_emulated(oracle, emu):
    """Variant U0 (rach_core_u0.cuh) on the host against the U0 oracle: the warp step (one lane per live UE, the 32
    lanes played by a loop over the same source the device compiles; crowded ms fall back to the serial step) and
    the serial step alone."""
    import ctypes
    so = os.path.join(ROOT, "tests", "emu", "_build", "librach_emu.so")
    f = oracle._lib(so, "emu_run_u0")
    mode = ctypes.c_int.in_dll(ctypes.CDLL(so), "emu_u0_mode")
    rnd = random.Random(8)
    cases = [dict(nUE=2000), dict(nUE=20000, seed=2), dict(nUE=40000, nPreamble=1, seed=3),
             dict(nUE=250000, nPreamble=64, backoffIndicator=2, seed=327613445147561757, rep=601, stopMs=6000),   # > 32 live
             dict(nUE=120000, nPreamble=16, backoffIndicator=1, seed=264716576123012100, rep=650, stopMs=3000)]
    for _ in range(25):
        cases.append(dict(nUE=rnd.choice([1, 2, 50, 400, 3000, 9000, 40000]), nPreamble=rnd.choice([1, 2, 3, 8, 64]),
                          backoffIndicator=rnd.choice([1, 2, 5, 20, 40]), seed=rnd.getrandbits(60), rep=rnd.randrange(1000),
                          stopMs=rnd.choice([0, 0, 3000, 20000])))
    for kw in cases:
        cfg = oracle.make_config_u0(**kw)
        p, ue = oracle.run_port_u0(cfg)
        for md in (1, 0):
            mode.value = md
            e, ue2, _ = oracle._run(f, cfg, True, False)
            for k in ("simTimeMs", "nSuccess", "preambleTxSum", "delaySum", "collisionPreambles", "totalPreambleTxop"):
                assert getattr(p, k) == getattr(e, k), (k, md, kw)
            np.testing.assert_array_equal(ue, ue2, err_msg="%s mode %d" % (kw, md))
    mode.value = 1


def test_work_list_overflow_paths(oracle, tmp_path):
    """The singleton scans of a ms keep their first entries in shared memory and the rest in global memory
    (RA_SCAP in rach_core.cuh).  Built here with a capacity of 2 so that every run overflows it, and phase 5
    (the kernel's ra_phase5_warp) and the histogram clear read past the shared-memory front; results must not change."""
    so = str(tmp_path / "librach_emu_small.so")
    subprocess.check_call(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-DRA_SCAP=2",
                           "-DRA_NO_POS_HINT",       # also: granted non-movers always take the search fallback (phase 6b)
                           "-I", os.path.join(ROOT, "include"), "-I", os.path.join(ROOT, "oracle"),
                           "-I", os.path.join(ROOT, "5g-nr-randomaccess_b200", "csrc"),
                           os.path.join(ROOT, "tests", "emu", "rach_emu.cpp"),
                           os.path.join(ROOT, "5g-nr-randomaccess_b200", "csrc", "rach_host.cpp"), "-o", so])
    f = oracle._lib(so, "emu_run")
    rnd = random.Random(5)
    for _ in range(25):
        kw = dict(nUE=rnd.choice([300, 1500, 4000, 9000]), nPreamble=rnd.choice([2, 3, 8, 54]),
                  backoffIndicator=rnd.choice([1, 2, 5, 20]), nGrantUL=rnd.choice([1, 2, 4, 12]),
                  maxRarWindow=rnd.choice([2, 3, 6]), maxMsg2TxCount=rnd.choice([0, 1, 3, 9]),
                  accessTime=rnd.choice([1, 5, 5, 7]), seed=rnd.getrandbits(64), rep=rnd.randrange(5000))
        cfg = oracle.make_config(**kw)
        p, ue, _ = oracle.run_port(cfg)
        e, ue2, _ = oracle._run(f, cfg, True, False)
        for k in KEYS:
            assert getattr(p, k) == getattr(e, k), (k, kw)
        np.testing.assert_array_equal(ue, ue2, err_msg=str(kw))
    # the light-ms path met both of its hand-overs to the general path: a Msg3 restart landing on the ms (code 2) and
    # a granted UE that has to be searched for (code 3, forced by RA_NO_POS_HINT)
    lib = C.CDLL(so)
    assert C.c_longlong.in_dll(lib, "emu_light_code3").value > 0
    assert C.c_longlong.in_dll(lib, "emu_light_ms").value > 0


def test_light_ms_path_against_general_path(oracle, emu):
    """ra_light_ms (one warp, no block barrier, phases 0/1/4/5/6 fused) must give what the general block-wide path gives:
    same runs with the light path switched off, and the share of ms it takes is what makes it worth having."""
    so = os.path.join(ROOT, "tests", "emu", "_build", "librach_emu.so")
    lib = C.CDLL(so)
    light, n_light, n_total, n_code2 = (C.c_int.in_dll(lib, "emu_light"), C.c_longlong.in_dll(lib, "emu_light_ms"),
                                        C.c_longlong.in_dll(lib, "emu_total_ms"), C.c_longlong.in_dll(lib, "emu_light_code2"))
    f, thr = emu
    thr.value = 128
    n_code2.value = 0
    for kw, min_share in ((dict(nUE=100000, distribution=1, seed=3), 0.7), (dict(nUE=10000, seed=4), 0.6),
                          (dict(nUE=40000, seed=5, stopMs=6000), 0.3), (dict(nUE=3000, nPreamble=3, nGrantUL=2, seed=5), 0.4),
                          (dict(nUE=60000, distribution=1, nGrantUL=2, nPreamble=8, seed=6, stopMs=20000), 0.0),
                          (dict(nUE=2500, maxRarWindow=40, seed=7), 0.3),      # a window wider than the 32-bit slot mask
                          (dict(nUE=20000, distribution=1, nPreamble=100, nGrantUL=3, seed=8, stopMs=15000), 0.3)):
        cfg = oracle.make_config(**kw)
        out = []
        for mode in (1, 0):
            light.value = mode
            n_light.value = 0
            n_total.value = 0
            e, ue, _ = oracle._run(f, cfg, True, False)
            out.append((e, ue))
            if mode:
                assert n_light.value >= min_share * n_total.value, (kw, n_light.value, n_total.value)
            else:
                assert n_light.value == 0
        light.value = 1
        for k in KEYS:
            assert getattr(out[0][0], k) == getattr(out[1][0], k), (k, kw)
        np.testing.assert_array_equal(out[0][1], out[1][1], err_msg=str(kw))
    assert n_code2.value > 0


def test_division_free_modulo_is_exact():
    """rand() % backoffIndicator, rand() % nPreamble, subTime % accessTime (W:478,502,514,518) run as multiply-shift with a
    per-divisor magic number (rach_core.cuh: ra_magic / ra_mod_shift / ra_mod).  Exact for every divisor the validator
    admits (<= 4096) and beyond, over the whole 31-bit range of rand(): edge values around multiples + random ones."""
    so = subprocess.check_output([os.path.join(ROOT, "tests", "emu", "build_emu.sh")]).decode().strip()
    lib = C.CDLL(so)
    lib.emu_mod.restype = C.c_uint
    lib.emu_mod.argtypes = [C.c_uint, C.c_uint]
    rnd = random.Random(1)
    top = 2 ** 31 - 1
    for d in list(range(1, 4100)) + [5000, 8191, 8192, 8193, 65535, 65536]:
        xs = [0, 1, d - 1, d, d + 1, 2 * d - 1, 2 * d, top, top - 1, top // d * d, top // d * d - 1]
        xs += [rnd.randrange(2 ** 31) for _ in range(30)]
        for x in xs:
            if 0 <= x <= top:
                assert lib.emu_mod(x, d) == x % d, (x, d)
