"""Cost of ticking some robots of a running batch on their own (hsddp_batch_*_problems) on the bench's config-3 workload.

  (a) one robot's tick inside a 4,096-robot handle -- mpc_update, set_initial_condition, solve (2 AL x 1 DDP) and mpc_command
      of that robot only -- against the same tick of a handle that holds that one robot;
  (b) 8 cohorts of 512 robots ticking in turn (one cohort per call, the 4,096 robots once per round of 8) against the
      whole-batch tick of all 4,096.
Variants run round-robin (one block of ticks of every variant per round).  Per tick: host wall clock of the four calls (the
command read-out ends in a device synchronise) and device time between CUDA events from before the update to after the
solve.  The card's name, power limit and maximum SM clock are read in the same process.
Usage: python tools/subset_tick.py [--robots 4096] [--cohorts 8] [--rounds 5] [--ticks 8] [--out profiles/r03e_subset_tick.json]"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
pkg = importlib.import_module("hkd-mpc_b200")
wl = importlib.import_module("hkd-mpc_b200.workloads")


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # the numbers are still device times; the card line is then missing
        return f"nvidia-smi unavailable: {e}"


def tick(B, opt, problems):
    """One tick; returns (wall ms, device ms from before the update to after the solve)."""
    x = B.get_rows("Xbar", 1, 1)[:, 0, :]
    x = x[problems].copy() if problems is not None else x.copy()
    B.sync()
    t0 = time.perf_counter()
    B.event_record(0)
    B.mpc_update(problems=problems)
    B.set_initial_condition(x, problems=problems)
    B.solve(opt, problems=problems)
    B.event_record(1)
    B.mpc_command(8, problems=problems)
    t1 = time.perf_counter()
    return (t1 - t0) * 1e3, B.event_elapsed_ms(0, 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--robots", type=int, default=4096)
    ap.add_argument("--cohorts", type=int, default=8)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--ticks", type=int, default=8, help="timed ticks per variant and round (after one untimed tick)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03e_subset_tick.json"))
    args = ap.parse_args()
    plan = 0.6
    total_ticks = args.rounds * (args.ticks + 1)  # (ticks of one robot: every variant ticks each of its robots once per timed tick)
    _, e = wl.define("config3", 2 * args.robots, plan)
    e = wl.with_room_for_ticks(e, total_ticks + 2, plan)[:args.robots]
    w = wl.from_entries(pkg, "subset tick batch", e, plan)
    w1 = wl.from_entries(pkg, "one robot", e[:1], plan)
    opt = pkg.Options(max_AL_iter=2, max_DDP_iter=1)
    C = args.cohorts
    cohort = [np.arange(c, w.n, C, dtype=np.int32) for c in range(C)]  # (interleaved: every cohort spans the gaits and windows)
    # variant: (batch, list of problem lists ticked in turn; None = the whole batch)
    variants = {"one robot in a %d-robot handle" % w.n: (wl.gait_batch(pkg, w), [np.array([0], np.int32)]),
                "1-robot handle": (wl.gait_batch(pkg, w1), [None]),
                "%d cohorts of %d robots, one per tick" % (C, w.n // C): (wl.gait_batch(pkg, w), cohort),
                "whole %d-robot batch" % w.n: (wl.gait_batch(pkg, w), [None])}
    res = {}
    for name, (B, lists) in variants.items():
        B.solve(pkg.Options())
        res[name] = dict(wall_ms=[], device_ms=[])
    for rnd in range(args.rounds):
        for name, (B, lists) in variants.items():
            for t in range(args.ticks + 1):
                for p in lists:
                    wall, dev = tick(B, opt, p)
                    if t > 0:
                        res[name]["wall_ms"].append(wall)
                        res[name]["device_ms"].append(dev)
    out = dict(card=card(), robots=w.n, cohorts=C, rounds=args.rounds, ticks_per_round=args.ticks,
               what="per call: wall_ms = host clock of mpc_update + set_initial_condition + solve (2 x 1) + mpc_command of the listed "
                    "robots (or all), ending in a device synchronise; device_ms = CUDA events from before the update to after the solve; "
                    "p50 over all timed calls, spread = min / max of the per-round medians.  The cohort variant ticks each cohort once per "
                    "timed tick, so its calls are cohorts x ticks per round",
               variants=[])
    for name in variants:
        row = dict(variant=name)
        for key, vals in res[name].items():
            a = np.asarray(vals, np.float64)
            med = np.median(a.reshape(args.rounds, -1), axis=1)
            row[key] = dict(p50=float(np.median(a)), max=float(a.max()), round_median_min=float(med.min()), round_median_max=float(med.max()))
        out["variants"].append(row)
        print(json.dumps(row))
    print("card:", out["card"])
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
