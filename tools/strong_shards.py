#!/usr/bin/env python3
"""The eight 2,048-problem shards of BASELINE config 3 (16,384 problems in total, strong scaling on 8 GPUs) on ONE GPU, one after
the other: kernel time and reset + solve time per shard and solve mode.  The 8-GPU strong line is bounded by the slowest shard."""
import importlib, os, sys, time
import numpy as np
ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
pkg = importlib.import_module("hkd-mpc_b200")
wl = importlib.import_module("hkd-mpc_b200.workloads")
n = int(sys.argv[1]) if len(sys.argv) > 1 else 2048
modes = [int(m) for m in (sys.argv[2] if len(sys.argv) > 2 else "1,2").split(",")]
interleaved = len(sys.argv) > 3 and sys.argv[3] == "interleaved"  # shard r = problems r, r + R, r + 2 R, ... instead of a contiguous range
R = 16384 // n
for first in (range(R) if interleaved else range(0, 16384, n)):
    w = wl.config3(pkg, n, 0.6, first=first, stride=R if interleaved else 1)
    B = pkg.MultiPhaseDDPBatch(0)
    B.set_problems(w.schedules, w.schedule_id)
    B.set_initial_condition(w.x0)
    line = f"first {first:6d}:"
    for m in modes:
        B.set_solve_mode(m)
        for _ in range(2):
            B.reset(); B.solve()
        B.event_record(0)
        for _ in range(3):
            B.reset(); B.solve_async()
        B.event_record(1); B.sync()
        info = B.info()
        line += f"  mode {m}: kernel {B.last_solve_ms():6.2f} ms, reset+solve {B.event_elapsed_ms(0, 1) / 3:6.2f} ms"
    print(line + f"  mean iters {info['n_iter'].mean():.2f}, at 50: {(info['n_iter'] >= 50).sum()}", flush=True)
    del B
