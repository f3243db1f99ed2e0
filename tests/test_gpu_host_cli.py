"""The C host program (5g-nr-randomaccess_b200/host/rach_sim.c) against the reference's own
stdout report and result files (RandomAccessWithNOMA.c:354-361, 741-825) produced by the
tape-mode reference build -- byte for byte where that build exists (oracle/_ref), and always against a
stored digest of the host program's reports on the same runs (tests/golden/recorded_outputs.json; how it was
recorded: tests/conftest.py, Recorded)."""
import importlib
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

REF_SCRIPT = r'''
import sys
sys.path.insert(0, %r)
from oracle import oracle as O
cfg = O.make_config(nUE=int(sys.argv[1]), rep=int(sys.argv[2]), echo=2, maxMsg2TxCount=int(sys.argv[3]) - 1,
                    nGrantUL=int(sys.argv[4]), distribution=int(sys.argv[5]))
O.run_ref("w", cfg, per_ue=False)
''' % ROOT


def _outputs(args, out, d):
    """One run of the host program: its arguments, its stdout and every file it wrote under d."""
    got = {"args": args, "stdout": out}
    for f in sorted(d.rglob("*")):
        if f.is_file():
            got[str(f.relative_to(d))] = f.read_bytes()
    return got


def _reference(tmp, nue, rep, retx, grant, dist):
    d = tmp / ("ref_%d_%d" % (nue, rep))
    (d / "NomaBetaResults").mkdir(parents=True)
    (d / "NomaUniformResults").mkdir(parents=True)
    out = subprocess.run([sys.executable, "-c", REF_SCRIPT, str(nue), str(rep), str(retx), str(grant), str(dist)],
                         cwd=d, capture_output=True, text=True, check=True).stdout
    return d, out


@pytest.mark.parametrize("dist,sub", [(0, "NomaBetaResults"), (1, "NomaUniformResults")])
def test_stdout_and_files_match_reference(tmp_path, oracle, recorded, dist, sub):
    pkg = importlib.import_module("5g-nr-randomaccess_b200")
    exe = pkg.build_host()
    nues, retx, grant = [1500, 4000], 5, 7
    args = ["-t", "2", "-d", str(dist), "-mrc", str(retx), "-g", str(grant), "--nue", ",".join(map(str, nues))]
    out = subprocess.run([exe] + args + ["--outdir", str(tmp_path / "ours")],
                         capture_output=True, text=True, check=True).stdout
    recorded.check("cli_w_" + sub, recorded.digest(**_outputs(args, out, tmp_path / "ours")))
    if not oracle.ref_available("w"):
        return
    blocks = out.split("-------- ")
    assert blocks[0] == ("Traffic model: Uniform\n\n" if dist == 1 else "Traffic model: Beta\n\n")
    k = 1
    for seed in (0, 1):
        for nue in nues:
            d, ref_out = _reference(tmp_path, nue, seed, retx, grant, dist if dist == 1 else 0)
            ref_block = ref_out.split("-------- ")[1]
            assert blocks[k] == ref_block, (seed, nue)
            k += 1
            for kind in ("%d_Results.txt" % nue, "UE%05d_Logs.txt" % nue):
                ours = (tmp_path / "ours" / sub / ("%d_54_%s" % (seed, kind))).read_bytes()
                ref = (d / sub / ("0_54_%s" % kind)).read_bytes()
                assert ours == ref, (seed, nue, kind)


def test_cli_errors_match_reference_behaviour():
    pkg = importlib.import_module("5g-nr-randomaccess_b200")
    exe = pkg.build_host()
    r = subprocess.run([exe, "-p", "0"], capture_output=True, text=True)
    assert r.returncode == 255 and r.stdout == "Number of preamble must be greater than zero."     # W:106-108
    r = subprocess.run([exe, "-d", "2"], capture_output=True, text=True)
    assert r.returncode == 255 and r.stdout == "Traffic model just choose 1 or 2"                  # W:100-102
    r = subprocess.run([exe, "--bogus", "1"], capture_output=True, text=True)
    assert r.returncode == 255 and r.stdout.startswith("--times         -t : Simulation times (int)\n")
    assert "--hut           -u : Height of UE from ground (float)\n" in r.stdout                    # W:200


REF_SCRIPT_B = r'''
import sys
sys.path.insert(0, %r)
from oracle import oracle as O
cfg = O.make_config(nUE=int(sys.argv[1]), rep=int(sys.argv[2]), echo=2, nGrantUL=int(sys.argv[3]), geometry=0,
                    distribution=int(sys.argv[4]))
O.run_ref("b", cfg, per_ue=False)
''' % ROOT

REF_SCRIPT_N = r'''
import sys
sys.path.insert(0, %r)
from oracle import oracle as O
O.run_ref_n(O.make_config_n(nUE=int(sys.argv[1]), rep=int(sys.argv[2]), echo=2))
''' % ROOT


def _strip_latency(text):
    return "\n".join(l for l in text.split("\n") if not l.startswith("Latency:"))


@pytest.mark.parametrize("dist,sub", [(0, "BasicBetaSimulationResults"), (1, "BasicUniformSimulationResults")])
def test_format_b_matches_randomaccesssimulatorbeta(tmp_path, oracle, recorded, dist, sub):
    """--format b: stdout block (B:200-209, 440-446) and files (B:460-482, 484-514) of RandomAccessSimulatorBeta.c;
    the clock() latency line / 6th file line is the only thing not compared."""
    pkg = importlib.import_module("5g-nr-randomaccess_b200")
    exe = pkg.build_host()
    nue = 3000
    args = ["--format", "b", "-t", "2", "-d", str(dist), "--nue", str(nue)]
    out = subprocess.run([exe] + args + ["--outdir", str(tmp_path / "ours")],
                         capture_output=True, text=True, check=True).stdout
    got = _outputs(args, _strip_latency(out), tmp_path / "ours")
    for name in got:
        if name.endswith("_Results.txt"):
            lines = got[name].split(b"\n")
            assert len(lines) == 6, name
            got[name] = b"\n".join(lines[:5])
    recorded.check("cli_b_" + sub, recorded.digest(**got))
    if not oracle.ref_available("b"):
        return
    blocks = out.split("-------- ")
    for seed in (0, 1):
        d = tmp_path / ("refb_%d" % seed)
        (d / "BasicBetaSimulationResults").mkdir(parents=True)
        (d / "BasicUniformSimulationResults").mkdir(parents=True)
        ref_out = subprocess.run([sys.executable, "-c", REF_SCRIPT_B, str(nue), str(seed), "54", "1" if dist == 1 else "2"],
                                 cwd=d, capture_output=True, text=True, check=True).stdout
        assert _strip_latency(blocks[1 + seed]) == _strip_latency(ref_out.split("-------- ")[1]), seed
        ours = (tmp_path / "ours" / sub / ("%d_54_%d_Results.txt" % (seed, nue))).read_text().split("\n")
        ref = (d / sub / ("0_54_%d_Results.txt" % nue)).read_text().split("\n")
        assert ours[:5] == ref[:5] and len(ours) == len(ref) == 6
        logname = ("54_Exclude_msg2_failures_UE%05d_Logs.txt" % nue) if dist == 1 else None
        ours_log = (tmp_path / "ours" / sub / (logname or "%d_54_UE%05d_Logs.txt" % (seed, nue))).read_bytes()
        ref_log = (d / sub / (logname or "0_54_UE%05d_Logs.txt" % nue)).read_bytes()
        if dist == 1 and seed == 0:
            continue          # B's Uniform log name has no seed in it: the second seed overwrote the first (B:488)
        assert ours_log == ref_log, seed


def test_format_n_matches_noma_c(tmp_path, oracle, recorded):
    """--format n: NOMA.c's result line (N:598-635) on stdout and appended to TestResults/Sector_<nUE>_Result.txt."""
    pkg = importlib.import_module("5g-nr-randomaccess_b200")
    exe = pkg.build_host()
    nues = [2000, 6000]
    args = ["--format", "n", "-t", "2", "--nue", ",".join(map(str, nues))]
    out = subprocess.run([exe] + args + ["--outdir", str(tmp_path / "ours")],
                         capture_output=True, text=True, check=True).stdout
    recorded.check("cli_n", recorded.digest(**_outputs(args, out, tmp_path / "ours")))
    if not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libref_n.so")):
        return
    exp = ""
    files = {n: "" for n in nues}
    for seed in (0, 1):
        for n in nues:
            d = tmp_path / ("refn_%d_%d" % (seed, n))
            (d / "TestResults").mkdir(parents=True)
            ref_out = subprocess.run([sys.executable, "-c", REF_SCRIPT_N, str(n), str(seed)], cwd=d, capture_output=True,
                                     text=True, check=True).stdout
            line = ref_out.split("\n")[0] + "\n"
            assert ref_out == line + "Done\n"
            exp += line
            files[n] += (d / "TestResults" / ("Sector_%d_Result.txt" % n)).read_text()
        exp += "Done\n"
    assert out == exp
    for n in nues:
        assert (tmp_path / "ours" / "TestResults" / ("Sector_%d_Result.txt" % n)).read_text() == files[n]


REF_SCRIPT_U0 = r'''
import sys
sys.path.insert(0, %r)
from oracle import oracle as O
r, _ = O.run_ref_u0(O.make_config_u0(nUE=int(sys.argv[1]), rep=0, echo=2))
print("COUNTERS %%d %%d %%d %%d" %% (r.collisionPreambles, r.totalPreambleTxop, r.preambleTxSum, r.nSuccess))
''' % ROOT


def test_format_u_matches_random_access_simulator_c(tmp_path, oracle, recorded):
    """--format u: the report of RandomAccessSimulator.c (U0:69-70, 141-143, 277-345): stdout, *_Results.txt and
    *_Logs.txt byte for byte against the tape-mode build of that file; its collision / tx-opportunity counters are
    globals that accumulate over the nUE sweep (U0:36-37), so the second point's two ratio lines are checked
    against the sums."""
    import numpy as np
    pkg = importlib.import_module("5g-nr-randomaccess_b200")
    exe = pkg.build_host()
    nues = [20000, 30000]
    args = ["--format", "u", "--nue", ",".join(map(str, nues))]
    out = subprocess.run([exe] + args + ["--outdir", str(tmp_path / "ours")],
                         capture_output=True, text=True, check=True).stdout
    recorded.check("cli_u", recorded.digest(**_outputs(args, out, tmp_path / "ours")))
    if not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libref_u0.so")):
        return
    refs = []
    for n in nues:
        d = tmp_path / ("refu_%d" % n)
        (d / "2_SimulationResults").mkdir(parents=True)
        ro = subprocess.run([sys.executable, "-c", REF_SCRIPT_U0, str(n)], cwd=d, capture_output=True, text=True, check=True).stdout
        body, counters = ro.rsplit("COUNTERS ", 1)
        refs.append((d, body, [int(x) for x in counters.split()]))
    # first point: everything identical
    assert out.startswith(refs[0][1])
    for kind in ("Results", "Logs"):
        name = "2_Exclude_msg2_failures_UE%05d_%s.txt" % (nues[0], kind)
        assert (tmp_path / "ours" / "2_SimulationResults" / name).read_bytes() == (refs[0][0] / "2_SimulationResults" / name).read_bytes(), name
    # second point: the per-UE log is identical; the report differs only in the two lines fed by the global counters
    ours2 = out[len(refs[0][1]):].split("\n")
    ref2 = refs[1][1].split("\n")
    (c1, t1, _, _), (c2, t2, tx2, ns2) = refs[0][2], refs[1][2]
    f32 = np.float32
    exp = list(ref2)
    for i, line in enumerate(ref2):
        if line.startswith("Number of collision preambles:"):
            exp[i] = "Number of collision preambles: %f" % float(f32(c1 + c2) / f32(tx2))
        if line.startswith("Average preamble tx count:"):
            exp[i] = "Average preamble tx count: %f" % float(f32(t1 + t2) / f32(ns2))
    assert ours2 == exp
    name = "2_Exclude_msg2_failures_UE%05d_Logs.txt" % nues[1]
    assert (tmp_path / "ours" / "2_SimulationResults" / name).read_bytes() == (refs[1][0] / "2_SimulationResults" / name).read_bytes()


def test_binary_logs_and_device_list(tmp_path):
    """--binlog writes the 14 saveResult fields (W:812-819) per UE as int32 after a 32-byte header; the numbers equal the
    text log's; --devices takes a list (all GPUs of the box) and changes nothing in the output."""
    import re
    import numpy as np
    import torch
    pkg = importlib.import_module("5g-nr-randomaccess_b200")
    exe = pkg.build_host()
    common = ["-t", "3", "--nue", "1200,5000", "-g", "5"]
    subprocess.run([exe] + common + ["--outdir", str(tmp_path / "txt")], capture_output=True, text=True, check=True)
    devs = ",".join(str(i) for i in range(torch.cuda.device_count()))
    out_b = subprocess.run([exe] + common + ["--binlog", "--devices", devs, "--outdir", str(tmp_path / "bin")],
                           capture_output=True, text=True)
    assert out_b.returncode == 0, out_b.stderr
    assert ("on %d device(s)" % torch.cuda.device_count()) in out_b.stderr
    for seed in range(3):
        for nue in (1200, 5000):
            raw = (tmp_path / "bin" / "NomaBetaResults" / ("%d_54_UE%05d_Logs.bin" % (seed, nue))).read_bytes()
            assert raw[:8] == b"RAUELOG1"
            hdr = np.frombuffer(raw[8:32], dtype="<i4")
            assert list(hdr[:4]) == [nue, 14, seed, 54] and len(raw) == 32 + nue * 14 * 4
            rows = np.frombuffer(raw[32:], dtype="<i4").reshape(nue, 14)
            txt = (tmp_path / "txt" / "NomaBetaResults" / ("%d_54_UE%05d_Logs.txt" % (seed, nue))).read_text().splitlines()
            assert len(txt) == nue
            for i in (0, 1, nue // 2, nue - 1):
                vals = [int(x) for x in re.findall(r": (-?\d+)", txt[i])]
                assert vals[0] == i and vals[1:] == list(rows[i]), (seed, nue, i)
            a = (tmp_path / "txt" / "NomaBetaResults" / ("%d_54_%d_Results.txt" % (seed, nue))).read_bytes()
            b = (tmp_path / "bin" / "NomaBetaResults" / ("%d_54_%d_Results.txt" % (seed, nue))).read_bytes()
            assert a == b
