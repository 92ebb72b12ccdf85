"""Cost of restarting problems inside a running MPC batch (hsddp_batch_restart_problems) on the bench's 4,096-robot config-3
tick loop: per tick  mpc_update -> set_initial_condition -> restart_problems(k robots) -> solve(2 AL x 1 DDP).

Variants, each on its own batch, run round-robin (one block of ticks of every variant per round) so that the spread between
rounds covers the same host / GPU conditions for all of them:
  k = 0, 1, 16, 256 restarts per tick, the restarted robots' next solve with first_solve = 5 x 10 ("cold") or with the tick's
  own budget ("tick"); and, for comparison, rebuilding the whole batch (set_problems_from_gaits + set_initial_condition) and
  its cold solve, which is what a fleet had to do before restarts existed.
Per tick: host wall clock of the whole tick (ends with a device synchronise), device time between CUDA events around the
update, the restart call and the solve, and the host wall clock of the restart call alone (it contains one host synchronise).
Usage: python tools/restart_tick.py [--robots 4096] [--rounds 5] [--ticks 8] [--out profiles/r03a_restart_tick.json]"""
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
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        return q
    except Exception as e:  # the numbers are still device times; the card line is then missing
        return f"nvidia-smi unavailable: {e}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--robots", type=int, default=4096)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--ticks", type=int, default=8, help="timed ticks per variant and round (after one untimed tick)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03a_restart_tick.json"))
    args = ap.parse_args()
    plan, order = 0.6, list(wl.GAITS)
    total_ticks = args.rounds * (args.ticks + 1)
    _, e = wl.define("config3", 2 * args.robots, plan)
    w = wl.from_entries(pkg, "restart tick batch", wl.with_room_for_ticks(e, total_ticks + 2, plan)[:args.robots], plan)
    refs = [pkg.QuadReference(wl.gait_path(g)) for g in order]
    tick_opt, cold_opt = pkg.Options(max_AL_iter=2, max_DDP_iter=1), pkg.Options()
    rng = np.random.default_rng(0)
    # restart targets: random robots to random windows near the start of a random gait table (room for every later tick)
    n_win = 100

    def restart_list(k):
        p = rng.choice(w.n, size=k, replace=False).astype(np.int32)
        g = rng.integers(0, 3, size=k).astype(np.int32)
        win = rng.integers(0, n_win, size=k).astype(np.int32)
        x0 = wl.initial_states([(order[gi], int(wi), "reference", 7 + j) for j, (gi, wi) in enumerate(zip(g, win))], pkg.compute_hkd_state)
        return p, g, win, x0

    variants = [(0, None)] + [(k, b) for k in (1, 16, 256) for b in ("cold", "tick")] + [("rebuild", None)]
    batches, res = {}, {}
    for v in variants:
        B = wl.gait_batch(pkg, w)
        B.solve(cold_opt)
        batches[v] = B
        res[v] = dict(wall_ms=[], update_ms=[], restart_dev_ms=[], solve_dev_ms=[], restart_wall_ms=[], iters_max=[])
    for rnd in range(args.rounds):
        for v in variants:
            B = batches[v]
            k, budget = v
            for t in range(args.ticks + 1):
                x = B.get_rows("Xbar", 1, 1)[:, 0, :].copy()
                lists = restart_list(k) if isinstance(k, int) and k > 0 else None
                B.sync()
                t0 = time.perf_counter()
                B.event_record(0)
                if k == "rebuild":
                    B.set_problems_from_gaits(refs, [order.index(g) for g, _ in w.keys], [kk for _, kk in w.keys], w.plan, w.schedule_id)
                    B.event_record(1)
                    B.set_initial_condition(x)
                else:
                    B.mpc_update()
                    B.event_record(1)
                    B.set_initial_condition(x)
                B.event_record(2)
                tr0 = time.perf_counter()
                if lists is not None:
                    B.restart(*lists, first_solve=cold_opt if budget == "cold" else None)
                    B.sync()
                tr1 = time.perf_counter()
                B.event_record(3)
                B.solve(cold_opt if k == "rebuild" else tick_opt)
                B.event_record(4)
                B.sync()
                t1 = time.perf_counter()
                if t == 0:
                    continue  # (first tick of a block: untimed)
                r = res[v]
                r["wall_ms"].append((t1 - t0) * 1e3)
                r["update_ms"].append(B.event_elapsed_ms(0, 1))
                r["restart_dev_ms"].append(B.event_elapsed_ms(2, 3))
                r["restart_wall_ms"].append((tr1 - tr0) * 1e3)
                r["solve_dev_ms"].append(B.event_elapsed_ms(3, 4))
                r["iters_max"].append(int(B.info()["n_iter"].max()))
    out = dict(card=card(), robots=w.n, schedules=len(w.keys), rounds=args.rounds, ticks_per_round=args.ticks,
               what="per tick: wall_ms = host clock of update (or rebuild) + set_initial_condition + restart + solve, ending in a device "
                    "synchronise; update_ms, restart_dev_ms, solve_dev_ms = CUDA events; restart_wall_ms = host clock of the restart call "
                    "and a device synchronise; p50 over all timed ticks, spread = min / max of the per-round medians",
               variants=[])
    for v in variants:
        r = res[v]
        row = dict(restarts=v[0], first_solve=v[1] or ("5x10 (all robots)" if v[0] == "rebuild" else "-"))
        for key, vals in r.items():
            a = np.asarray(vals, np.float64)
            per_round = a.reshape(args.rounds, args.ticks)
            med = np.median(per_round, axis=1)
            row[key] = dict(p50=float(np.median(a)), max=float(a.max()), round_median_min=float(med.min()), round_median_max=float(med.max()))
        out["variants"].append(row)
        print(json.dumps(row))
    print("card:", out["card"])
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
