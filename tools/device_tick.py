"""What the host round trips of an MPC tick cost: the host-I/O tick against the device-I/O tick on the bench's config-3 workload.

Two handles hold the same 4,096 robots (built as bench.py's mpc_batch builds them).  Every tick's "measured" state (the plan's
next node) is prepared before the timed window: in pinned host memory for one handle, as a CUDA tensor for the other.
  host-I/O tick:   mpc_update, set_initial_condition (pinned NumPy view), solve, mpc_command into pinned host memory;
  device-I/O tick: mpc_update, set_initial_condition (CUDA tensor, hsddp_batch_set_initial_condition_dev), solve_async,
                   mpc_command into a CUDA tensor (hsddp_batch_get_mpc_command_dev), then one synchronise of the caller's stream.
The two variants alternate tick by tick, for the whole batch, one robot of the handle and one cohort of 512 robots (the 8
cohorts in turn).  Every tick's command records of the two handles are compared byte for byte.  Per tick: host wall clock of
the four calls (ending in a synchronise either way) and device time between CUDA events on the handle's stream from before the
update to after the solve.  The card's name, power limit and maximum SM clock are read in the same process.
Usage: python tools/device_tick.py [--robots 4096] [--cohorts 8] [--rounds 5] [--ticks 8] [--out profiles/r03g_device_tick.json]"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

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


def host_tick(B, opt, p, x_pin, cmd_pin):
    """(wall ms, device ms, command records) of a tick whose states come from and commands go to pinned host memory."""
    n = len(x_pin)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    B.event_record(0)
    B.mpc_update(problems=p)
    B.set_initial_condition(x_pin.numpy(), problems=p)
    B.solve(opt, problems=p)
    B.event_record(1)
    out = B.mpc_command(8, out=cmd_pin.numpy().view(pkg.CMD_DTYPE).reshape(n), problems=p)
    t1 = time.perf_counter()
    return (t1 - t0) * 1e3, B.event_elapsed_ms(0, 1), out.tobytes()


def device_tick(B, opt, p, x_dev, cmd_dev):
    """The same tick with the states in and the commands out through CUDA tensors, ordered on the current stream."""
    stream = torch.cuda.current_stream()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    B.event_record(0)
    B.mpc_update(problems=p)
    B.set_initial_condition(x_dev, problems=p)
    B.solve_async(opt, problems=p)
    B.event_record(1)
    B.mpc_command(8, out=cmd_dev, problems=p)
    stream.synchronize()
    t1 = time.perf_counter()
    return (t1 - t0) * 1e3, B.event_elapsed_ms(0, 1), cmd_dev.cpu().numpy().tobytes()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--robots", type=int, default=4096)
    ap.add_argument("--cohorts", type=int, default=8)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--ticks", type=int, default=8, help="timed ticks per variant and round (after one untimed tick)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03g_device_tick.json"))
    args = ap.parse_args()
    plan = 0.6
    per_variant = args.rounds * (args.ticks + 1)
    _, e = wl.define("config3", 2 * args.robots, plan)
    e = wl.with_room_for_ticks(e, 3 * per_variant + 4, plan)[:args.robots]  # (robot 0 ticks in all three variants)
    w = wl.from_entries(pkg, "device tick batch", e, plan)
    H, D = wl.gait_batch(pkg, w), wl.gait_batch(pkg, w)
    for B in (H, D):
        B.solve(pkg.Options())
    opt = pkg.Options(max_AL_iter=2, max_DDP_iter=1)
    C = args.cohorts
    cohort = [np.arange(c, w.n, C, dtype=np.int32) for c in range(C)]
    variants = {"whole %d-robot batch" % w.n: [None],
                "one robot of the %d-robot handle" % w.n: [np.array([0], np.int32)],
                "one cohort of %d robots (%d cohorts in turn)" % (w.n // C, C): cohort}
    itemsize = pkg.CMD_DTYPE.itemsize
    res = {name: {io: dict(wall_ms=[], device_ms=[]) for io in ("host", "device")} for name in variants}
    mismatches = 0
    for rnd in range(args.rounds):
        for name, lists in variants.items():
            for t in range(args.ticks + 1):
                p = lists[(rnd * (args.ticks + 1) + t) % len(lists)]
                x = H.get_rows("Xbar", 1, 1)[:, 0, :]
                x = (x if p is None else x[p]).copy()
                n = len(x)
                x_pin = torch.from_numpy(x).pin_memory()
                cmd_pin = torch.zeros((n, itemsize), dtype=torch.uint8).pin_memory()
                x_dev = torch.from_numpy(x).cuda()
                cmd_dev = torch.zeros((n, itemsize), dtype=torch.uint8, device="cuda")
                hw, hd, hc = host_tick(H, opt, p, x_pin, cmd_pin)
                dw, dd, dc = device_tick(D, opt, p, x_dev, cmd_dev)
                mismatches += hc != dc
                if t > 0:
                    for io, (wall, dev) in (("host", (hw, hd)), ("device", (dw, dd))):
                        res[name][io]["wall_ms"].append(wall)
                        res[name][io]["device_ms"].append(dev)
    out = dict(card=card(), robots=w.n, cohorts=C, rounds=args.rounds, ticks_per_round=args.ticks,
               command_record_bytes=itemsize, command_mismatches=int(mismatches),
               what="per tick: wall_ms = host clock of mpc_update + initial states + solve (2 x 1) + commands, ending in a "
                    "synchronise (host-I/O: the command copy's; device-I/O: one synchronise of the caller's stream); device_ms = CUDA "
                    "events on the handle's stream from before the update to after the solve.  Host-I/O: states from and commands "
                    "into pinned host memory; device-I/O: CUDA tensors through the _dev entry points.  The variants alternate tick "
                    "by tick; p50 over all timed ticks, spread = min / max of the per-round medians.  command_mismatches counts ticks "
                    "whose command records of the two handles differ",
               variants=[])
    for name in variants:
        for io in ("host", "device"):
            row = dict(variant=name, io=io)
            for key, vals in res[name][io].items():
                a = np.asarray(vals, np.float64)
                med = np.median(a.reshape(args.rounds, -1), axis=1)
                row[key] = dict(p50=float(np.median(a)), max=float(a.max()), round_median_min=float(med.min()), round_median_max=float(med.max()))
            out["variants"].append(row)
            print(json.dumps(row))
    print("card:", out["card"], "command mismatches:", mismatches)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    if mismatches:
        sys.exit(1)


if __name__ == "__main__":
    main()
