"""Cost of ra_options.histograms: each workload runs with histograms off and on, alternating in one process (the order
flips every round), and the medians of the rounds are compared.  A round creates the handle, runs it once to warm up and
times --steps runs by the CUDA events inside the library (ra_sim_kernel_ms) and by the host clock around ra_sim_run.
Prints the GPU's name and power limit first: the numbers belong to that card.

    python tools/bench_histograms.py [--rounds 5] [--steps 2] [--only NAME]
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# (name, point, replications): the bench.py headline, Uniform traffic (long light-loaded horizon: the largest region to
# flush per replication), and the N and U0 engines with their own success sites
WORKLOADS = [("headline Beta 100k x 4096", dict(nUE=100000), 4096),
             ("Uniform 100k x 256", dict(nUE=100000, distribution=1), 256),
             ("N 50k x 1024", dict(variant=2, nUE=50000), 1024),
             ("U0 100k x 1024", dict(variant=1, nUE=100000), 1024)]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        out = ""
    return out or "unknown (nvidia-smi unavailable)"


def one_round(pkg, point, reps, hist, steps):
    with pkg.RachSim([point], reps=reps, devices=[0], histograms=hist) as sim:
        sim.run()
        kern, wall = [], []
        for _ in range(steps):
            t0 = time.perf_counter()
            sim.run()
            wall.append((time.perf_counter() - t0) * 1e3)
            kern.append(sim.kernel_ms)
        return statistics.mean(kern), statistics.mean(wall)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--only", default=None, help="run the workloads whose name contains this string")
    args = ap.parse_args()
    if args.rounds < 3:
        ap.error("--rounds must be at least 3 (medians)")
    pkg = importlib.import_module("5g-nr-randomaccess_b200")
    pkg.load_lib()
    print(json.dumps({"gpu": gpu_info(), "rounds": args.rounds, "steps": args.steps}), flush=True)
    for name, kw, reps in WORKLOADS:
        if args.only and args.only not in name:
            continue
        point = pkg.default_params(**kw)
        res = {False: [], True: []}
        for r in range(args.rounds):
            for hist in ((False, True) if r % 2 == 0 else (True, False)):
                res[hist].append(one_round(pkg, point, reps, hist, args.steps))
        med = {h: (statistics.median(k for k, _ in v), statistics.median(w for _, w in v)) for h, v in res.items()}
        print(json.dumps({"workload": name, "kernel_ms_off": round(med[False][0], 2), "kernel_ms_on": round(med[True][0], 2),
                          "cost_pct": round(100.0 * (med[True][0] / med[False][0] - 1.0), 2),
                          "wall_ms_off": round(med[False][1], 2), "wall_ms_on": round(med[True][1], 2),
                          "kernel_ms_rounds_off": [round(k, 2) for k, _ in res[False]],
                          "kernel_ms_rounds_on": [round(k, 2) for k, _ in res[True]]}), flush=True)


if __name__ == "__main__":
    main()
