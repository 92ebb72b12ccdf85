#!/usr/bin/env python3
"""One cold solve of a small batch — the target of `ncu` captures (profiles/)."""
import importlib, os, sys
import numpy as np
ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
pkg = importlib.import_module("hkd-mpc_b200")
wl = importlib.import_module("hkd-mpc_b200.workloads")
n = int(sys.argv[1]) if len(sys.argv) > 1 else 296
cfg = sys.argv[2] if len(sys.argv) > 2 else "config2"
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 1
mode = int(sys.argv[4]) if len(sys.argv) > 4 else 0  # solve mode: 0 auto, 1 persistent, 2 phased
w = getattr(wl, cfg)(pkg, n)
B = pkg.MultiPhaseDDPBatch(0)
B.set_solve_mode(mode)
B.set_problems(w.schedules, w.schedule_id)
B.set_initial_condition(w.x0)
for _ in range(reps):
    B.reset(); B.solve()
    info = B.info()
    print(f"{cfg} n={n}: kernel {B.last_solve_ms():.2f} ms, {n / B.last_solve_ms() * 1e3:.0f} solves/s, mean iters {info['n_iter'].mean():.2f}, sweeps {info['n_sweeps'].sum()}")
prof = B.profile()
if any(prof):
    names = ["rollout:U=K dx", "rollout:dynamics", "rollout:commit", "cost", "LQ approx", "sweep:phase init", "sweep:P1 Y,Z", "sweep:P2 Q",
             "sweep:P3 GJ", "sweep:P4 H'", "GJ:publish cols (or Px)", "GJ:pivot math (or linear rec)", "GJ:eliminate (or dV pass)", "P3:load tableau", "P3:gauss-jordan", "P3:stores"]
    tot = sum(prof)
    for nm, v in zip(names, prof):
        print(f"  {nm:22s} {v:>14d} cyc  {100.0 * v / tot:5.1f}%")
    print("  total cycles (thread 0 of all blocks)", tot)
