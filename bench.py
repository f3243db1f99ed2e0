#!/usr/bin/env python
"""bench.py -- the headline measurement: UE*RACH-occasion updates/s of the RACH step on B200.

Workload (BASELINE.json `metric`): 100 000 UEs x 4096 replications per GPU, Beta traffic over
10 s, RandomAccessWithNOMA.c defaults (54 preambles, BI 20, 12 grants, RAR window 5, max retx
10).  Nobody finishes early at 100k UEs, so every replication is exactly 2000 occasions and one
step (= one pass of the hot path over the batch) is 8.192e11 updates per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W]            our arm (CUDA, librach_gpu)
    python bench.py ... --dump-outputs DIR                         also write the last step's outputs as DIR/*.npy
    python bench.py --impl reference [--steps K] [--warmup W]      the reference's own CPU code

One JSON line on stdout (rank 0).  See DESIGN.md section 6 for what each key means.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ALGO_BYTES_PER_UPDATE = 32          # SURVEY section 8(d): one 128-bit read + one 128-bit write
METRIC = "UE*RACH-occasion updates/s"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_traffic():
    """dram bytes per launch of ra_step_kernel from the committed ncu capture, if any."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f)
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); power.append(float(r[3]))
            except ValueError:
                continue
            for n, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
# CPU baseline: the REFERENCE's own code (oracle/_ref/libref_w.so, compiled from
# /root/reference/RandomAccessWithNOMA.c by oracle/build_ref.sh) with its own libc rand().
# ------------------------------------------------------------------------------------------------
SAMPLE_MS = 1000        # the ONE prefix length of every CPU sample at the headline size (both arms, any --steps)
FULL_NUE = 30000        # a complete replication is affordable on the CPU at this size (about a minute per core)


def _ref_worker(args):
    nue, stop_ms, seed = args
    from oracle import oracle as O
    kind = "reference" if O.ref_available("w") else "port"
    cfg = O.make_config(nUE=nue, useTape=0 if kind == "reference" else 1, seed=seed, stopMs=stop_ms)
    t = time.perf_counter()
    if kind == "reference":
        r, _, _ = O.run_ref("w", cfg, per_ue=False)
    else:
        r, _, _ = O.run_port(cfg, per_ue=False)
    dt = time.perf_counter() - t
    ms_done = stop_ms if stop_ms > 0 else r.simTimeMs
    return kind, nue * ((ms_done + 4) // 5), dt, r.nSuccess


def cpu_reference_sample(nue, stop_ms, procs):
    """The reference's own code (libc rand()), one process per core, distinct seeds; each process runs the first
    `stop_ms` ms of a replication, or a complete replication when stop_ms == 0."""
    import multiprocessing as mp
    from oracle import oracle as O
    O.build()
    t = time.perf_counter()
    with mp.get_context("fork").Pool(procs) as pool:
        out = pool.map(_ref_worker, [(nue, stop_ms, 1000 + i) for i in range(procs)])
    wall = time.perf_counter() - t
    updates = sum(o[1] for o in out)
    kind = out[0][0]
    if stop_ms > 0:
        what = ("first %d ms (%d occasions) of a %d-UE Beta replication (a complete one takes ~14 min per core); the "
                "prefix is the cheap part of the run (before the Beta peak), so this number FLATTERS the CPU"
                % (stop_ms, (stop_ms + 4) // 5, nue))
    else:
        what = "one COMPLETE %d-UE Beta replication (10 000 ms, %d occasions)" % (nue, 2000)
    return {"value": updates / wall, "unit": "updates/s", "cores": procs, "kind": kind,
            "sample": "%s; one process per core, %d replications, libc rand()" % (what, procs),
            "wall_s": wall, "single_thread_value": max(o[1] / o[2] for o in out),
            "mean_success": sum(o[3] for o in out) / len(out)}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    procs = os.cpu_count() or 1
    total = args.steps + args.warmup
    vals = []
    for i in range(total):
        s = cpu_reference_sample(args.nue, SAMPLE_MS, procs)
        if i >= args.warmup:
            vals.append(s)
    updates_per_s = sum(v["value"] for v in vals) / len(vals)
    ms = 1000.0 * sum(v["wall_s"] for v in vals) / len(vals)
    line = {"impl": "reference", "metric": METRIC, "value": updates_per_s, "unit": "updates/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32",
            "data": "synthetic",
            "config": {"workload": "100k UEs, Beta 10 s, W defaults (54 preambles, BI 20, 12 grants, RAR 5, retx 10)",
                       "nUE": args.nue, "sample_ms": SAMPLE_MS, "replications_per_step": procs,
                       "same_work_as_gpu_arm": False,
                       "note": "a step here is the first %d ms of one replication per host core (bounded sample, the cheap "
                               "prefix); the GPU arm's step is 4096 complete replications.  The like-for-like CPU/GPU "
                               "pair is cpu_baseline.full_replication in the GPU arm's line" % SAMPLE_MS},
            "cpu_baseline": {"value": updates_per_s, "unit": "updates/s", "cores": procs,
                             "kind": vals[0]["kind"], "sample": vals[0]["sample"]},
            "e2e": {"value": updates_per_s, "unit": "updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def full_replication_pair(pkg, device, procs):
    """The like-for-like CPU/GPU pair: COMPLETE replications at a size the CPU can finish (FULL_NUE UEs, Beta 10 s,
    W defaults, overloaded regime: ~60 % success), the reference's code on every host core and the engine on the GPU."""
    cpu = cpu_reference_sample(FULL_NUE, 0, procs)
    reps = 2048
    p = pkg.default_params(nUE=FULL_NUE)
    with pkg.RachSim([p], reps=reps, devices=[device]) as sim:
        sim.run()
        sim.run()
        st = sim.stats_all()
        kms = sim.kernel_ms
    gpu_val = float(st["updates"].sum()) / (kms / 1e3)
    return {"nUE": FULL_NUE, "what": "complete replications on both sides (no prefix): the apples-to-apples CPU/GPU point",
            "cpu": {"value": cpu["value"], "unit": "updates/s", "cores": procs, "kind": cpu["kind"],
                    "single_thread_value": cpu["single_thread_value"], "replications": procs, "wall_s": cpu["wall_s"],
                    "mean_success_pct": 100.0 * cpu["mean_success"] / FULL_NUE},
            "gpu": {"value": gpu_val, "unit": "updates/s", "replications": reps, "kernel_ms": kms,
                    "mean_success_pct": 100.0 * float(st["nSuccess"].mean()) / FULL_NUE},
            "ratio_gpu_over_cpu_all_cores": gpu_val / cpu["value"],
            "ratio_gpu_over_cpu_one_core": gpu_val / cpu["single_thread_value"]}


# ------------------------------------------------------------------------------------------------
DUMP_LIMIT_BYTES = 64 << 20
DUMP_SKIP = ("updates", "recordMoves")      # engine work counters: how the engine scheduled its work, not results


def dump_outputs(out_dir, st, suffix="", limit=DUMP_LIMIT_BYTES):
    """What the last timed step returned to its caller: the per-replication counters of the simulation
    (ra_sim_stats_all), one float64 array per counter, indexed [point, replication] -- 11 x 4096 x 8 B at the headline
    size.  Above `limit` bytes a fixed, seeded sample of replications is written, and replication.npy holds their
    indices.  Two builds run with the same arguments see the same inputs (seeded tape, fixed replication ids), so
    their files compare value for value."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    names = [n for n in st.dtype.names if n not in DUMP_SKIP]
    reps = st.shape[1]
    keep = max(1, min(reps, limit // (8 * len(names) * st.shape[0] + 8)))
    if keep < reps:
        idx = np.sort(np.random.default_rng(0).choice(reps, keep, replace=False))
        st = st[:, idx]
        np.save(os.path.join(out_dir, "replication" + suffix + ".npy"), idx.astype(np.float64))
    for name in names:
        np.save(os.path.join(out_dir, name + suffix + ".npy"), st[name].astype(np.float64))


def run_our_arm(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; librach_gpu has no CPU path")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    pkg = importlib.import_module("5g-nr-randomaccess_b200")
    pkg.load_lib()

    reps_local, rep_offset = pkg.shard_plan(args.reps, world, rank, args.scaling)
    p = pkg.default_params(nUE=args.nue, seed=args.seed)
    if args.distribution == "uniform":
        p.distribution = 1
    sim = pkg.RachSim([p], reps=reps_local, devices=[local], rep_offset=rep_offset, ctas_per_sm=args.ctas_per_sm)

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        sim.run()
    sampler = ClockSampler(local)
    sync()
    sampler.start()
    t0 = time.perf_counter()
    kernel_ms = 0.0
    launches = 0
    for _ in range(args.steps):
        sim.run()                       # C-ABI call: kernel + D2H of the per-replication counters
        kernel_ms += sim.kernel_ms      # CUDA events on the launching stream, inside the library
        launches += sim.gpu_launches
    sync()
    wall_ms = (time.perf_counter() - t0) * 1e3
    clocks = sampler.stop()

    st = sim.stats_all()
    stats_bytes = st.nbytes
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, st, "_rank%d" % rank if world > 1 else "", DUMP_LIMIT_BYTES // world)
    t = torch.tensor([kernel_ms, wall_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)            # max over ranks of the device time
    # the one small all-reduce of the per-replication counters (NCCL over NVLink when world > 1)
    tot = pkg.allreduce_counters(pkg.local_counter_vector(st), dist if world > 1 else None, device="cuda")
    kernel_ms, wall_ms = float(t[0]), float(t[1])
    updates, n_succ, tx_sum, delay_sum, reps_total = (tot["updates"], tot["nSuccess"], tot["preambleTxSum"],
                                                      tot["delaySum"], tot["replications"])

    if rank == 0:
        peak, peak_src = peaks()
        value = updates * args.steps / (kernel_ms / 1e3)
        e2e = updates * args.steps / (wall_ms / 1e3)
        per_gpu = value / world
        achieved = per_gpu * ALGO_BYTES_PER_UPDATE / 1e9
        traffic = measured_traffic()
        same_workload = bool(traffic) and args.nue == 100000 and args.reps == 4096 and args.distribution == "beta" and args.scaling == "weak"
        line = {"metric": METRIC, "value": value, "unit": "updates/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": wall_ms / args.steps, "higher_is_better": True,
                "scaling": args.scaling, "vs_baseline": None, "dtype": "int32", "data": "synthetic",
                "config": {"workload": "100k UEs x 4096 replications per GPU, Beta 10 s, W defaults "
                                       "(54 preambles, BI 20, 12 grants, RAR 5, retx 10)",
                           "nUE": args.nue, "replications_per_gpu": args.reps if args.scaling == "weak" else None,
                           "replications_total": reps_total, "distribution": args.distribution,
                           "l2": "working set per step (calendar records of ~600 concurrent replications, >0.5 GB) exceeds the 126 MB L2",
                           "success_ratio_pct": 100.0 * n_succ / (reps_total * args.nue),
                           "mean_preamble_tx": tx_sum / max(n_succ, 1), "mean_delay_ms": delay_sum / max(n_succ, 1)},
                "e2e": {"value": e2e, "unit": "updates/s", "h2d_bytes_per_step": 8 + 0,
                        "d2h_bytes_per_step": stats_bytes + 4},
                "gpu_launches": launches * world,
                # BASELINE.md section 1 has no published throughput; the only timing the reference ships is
                # results.csv column 6 (unknown hardware, -O0): 370.5 s for the 100k-UE point = 5.4e5 updates/s
                "vs_results_csv_derived": value / world / 5.4e5,
                "kernel_ms_per_step": kernel_ms / args.steps,
                "replications_per_s": reps_total * args.steps / (kernel_ms / 1e3),
                "clocks": clocks,
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                             "frac": achieved / peak,
                             "traffic": traffic["dram_bytes_per_launch"] if same_workload else None,
                             "note": "achieved = updates/s/GPU x 32 B (SURVEY 8d contract); the engine is event-driven and "
                                     "moves fewer bytes than that model, so frac > 1 means avoided traffic -- see "
                                     "`traffic` (ncu dram bytes per launch) and DESIGN.md section 5; peak " + peak_src}}
        # the same kernel against the bytes it REALLY moves.  Counted live by the engine in this very run: every calendar
        # record it read at its event time (ra_stats.recordMoves), 16 B in + 16 B out each; next to it the DRAM bytes ncu
        # measured for this workload (profiles/traffic.json, written by tools/ncu_onepager.py from a capture of this round)
        moved = 32.0 * tot["recordMoves"] * args.steps / world            # bytes per GPU over the timed region
        real = moved / (kernel_ms / 1e3) / 1e9
        line["roofline_measured_traffic"] = {
            "bound": "hbm", "achieved": real, "peak": peak, "unit": "GB/s", "frac": real / peak,
            "bytes_per_launch_counted_live": 32.0 * tot["recordMoves"] / world,
            "bytes_per_launch_ncu": traffic["dram_bytes_per_launch"] if same_workload else None,
            "note": "achieved = engine-counted record traffic of this run (recordMoves x 32 B) / CUDA-event kernel time; the "
                    "event-driven engine moves a 16-B record only when a UE has an event, so this is the physical HBM "
                    "fraction.  The kernel is issue/latency-bound, not DRAM-bound (profiles/r02*_ncu_w*.md)"}
        if world == 1 and not args.no_cpu_baseline:
            procs = os.cpu_count() or 1
            cb = cpu_reference_sample(args.nue, SAMPLE_MS, procs)         # the same sample the --impl reference arm times
            cb["what"] = ("`value` = prefix sample at the headline size (same sample as the --impl reference arm); "
                          "`full_replication` = complete replications at %d UEs on both CPU and GPU" % FULL_NUE)
            if not args.no_full_replication:
                cb["full_replication"] = full_replication_pair(pkg, local, procs)
            line["cpu_baseline"] = cb
        print(json.dumps(line), flush=True)
    sim.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--reps", type=int, default=4096, help="replications per GPU (weak) or in total (strong)")
    ap.add_argument("--nue", type=int, default=100000)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--distribution", default="beta", choices=["beta", "uniform"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--ctas-per-sm", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-full-replication", action="store_true", help="skip the ~1-2 min complete-replication CPU/GPU pair")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's per-replication counters to DIR/<counter>.npy (float64, at most "
                         "64 MB: a seeded sample of replications above that); with several ranks each writes "
                         "DIR/<counter>_rank<r>.npy.  bench_outputs/ is git-ignored")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU arm's outputs (--impl ours)")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_our_arm(args)


if __name__ == "__main__":
    main()
