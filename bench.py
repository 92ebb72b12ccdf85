#!/usr/bin/env python3
"""bench.py — batched HS-DDP solves/s on B200 (BASELINE.json metric).

A "step" is one cold solve of the whole batch: reset to the reference's cold-start
guess + MultiPhaseDDP::solve for every problem of the rank's shard.

  python bench.py --gpus N --steps K --warmup W            # our arm (CUDA path through the C ABI)
  python bench.py --impl reference --gpus N --steps K ...  # CPU arm: the reference's HS-DDP path on host cores
  python bench.py ... --dump-outputs DIR                   # also write what the last timed step computed (DIR/<name>.npy)

Workload: SURVEY.md §8(d) config 3 — 16,384 mixed-gait Mini Cheetah problems
(trot / bound / pronk with flight phases and reset maps), plan 0.6 s, dt 0.01, ReB+AL.
  * headline `value` / `e2e`: 16,384 problems PER GPU ("weak" scaling: problems are sharded by global index,
    no data-path collective);
  * `strong`: the same run also times BASELINE config 3 as written — 16,384 problems IN TOTAL, index-sharded
    over the N ranks (2,048 per GPU at N = 8).
Timing: CUDA events on the solver handle's stream, barrier + synchronise on both sides,
MAX over ranks.  The per-GPU workspace (~4 GB) is far larger than L2, so no explicit L2
flush is needed between timed steps.

The CPU arm never loads the CUDA library: it builds the same inputs from the workload definition
(hkd-mpc_b200/workloads.py is pure NumPy for that) and the oracle's own compute_hkd_state.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# ---- work model (DESIGN.md §5) ----
F_STAGE = 203904.0               # ALGORITHMIC FLOP of one dense 24x24 Riccati stage (SURVEY.md §8d)
F_ITER_STAGE = 3600.0 + 5000.0   # LQ approximation + linear rollout, per stage per DDP iteration
F_TRIAL_STAGE = 2100.0           # one line-search trial, per stage
BYTES_STAGE = 6400.0             # minimum HBM bytes per stage per iteration (fused), SURVEY.md §8d
# FLOP the sweep kernel actually EXECUTES per stage (structure exploited: A = I + 12 dense rows, 12 coupled controls;
# DESIGN.md §4.3): 37 output tiles x 3 DMMA m8n8k4 (512 FLOP each) + the 12x12 block Gauss-Jordan on 49 tableau columns
# (6 steps x (20 eliminate + 8 pivot) DFMA per column) + ~1.5k FLOP of vector work
F_STAGE_EXECUTED = 120.5 * 512.0 + 49 * 6 * 28 * 2.0 + 1500.0  # (120.5 DMMA per stage executed: profiles/r02_sweep_sass_dmma.txt)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--problems", type=int, default=16384, help="problems per GPU (weak) = problems in total (strong block)")
    ap.add_argument("--config", default="config3", choices=["config2", "config3", "config4"])
    ap.add_argument("--plan", type=float, default=0.6)
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target wall time of ONE pass of the CPU sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--no-generic", action="store_true", help="skip the generic SinglePhase<12,12,0> / <36,12,12> sweep timing")
    ap.add_argument("--no-latency", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy (float64, "
                    "at most 64 MB; with several ranks, DIR/rank<r>/); the inputs depend only on the arguments")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    return args


def dump_outputs(pkg, B, out_dir, seed=0):
    """What a caller reads back after a solve of the batch, as float64 .npy files of at most 64 MB in all: the result
    record of every problem (info_<field>; a seeded sample beyond ~190k problems, indices in info_problem) and, for a
    seeded sample of at most 128 problems (indices in sample_problem), the trajectories Xbar / Ubar, the feed-forward
    dU and the gains K [stage, row, col] of every stage."""
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(seed)
    fields = [f for f in pkg.INFO_DTYPE.names if f != "_pad"]
    rows = {"Xbar": B.max_nodes, "Ubar": B.max_stages, "dU": B.max_stages, "K": B.max_stages}
    cols = {"Xbar": 24, "Ubar": 24, "dU": 24, "K": 576}
    n_info = min(B.n, (16 << 20) // (8 * (len(fields) + 1)))
    n_traj = min(B.n, 128, (44 << 20) // (8 * sum(rows[k] * cols[k] for k in rows)))
    pick_info = np.sort(rng.choice(B.n, n_info, replace=False))
    pick = np.sort(rng.choice(B.n, n_traj, replace=False))
    info = B.info()[pick_info]
    out = {"info_problem": pick_info, "sample_problem": pick}
    out.update({"info_" + f: info[f] for f in fields})
    for name, nr in rows.items():
        buf = np.zeros((B.n, 1, cols[name]))
        a = np.stack([B.get_rows(name, r, 1, out=buf)[pick, 0] for r in range(nr)], axis=1)  # row by row: K of a batch is GBs
        out[name] = np.swapaxes(a.reshape(n_traj, nr, 24, 24), -1, -2) if name == "K" else a  # K: column-major on the device
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, np.float64))


def config_block(args, world, name, n_schedules):
    """Identical in both arms (the driver compares them)."""
    return {"workload": name, "problems_per_gpu": args.problems, "problems_total": args.problems * world, "schedules_per_gpu": n_schedules,
            "plan_duration_s": args.plan, "dt": 0.01, "stages": int(round(args.plan / 0.01)),
            "options": "ddp_setting.info as consumed (alpha .1, gamma .01, 5 AL x 10 DDP, ReB+AL, MS)",
            "cache": "inputs larger than L2: %.1f GB workspace per GPU, no flush" % (args.problems * 0.23e6 / 1e9),
            "step": "cold-start reset + solve of every problem",
            "cpu_arm": "times a bounded sample of the same workload (first problems of rank 0's shard; see cpu_baseline.sample)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, power = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(smax)) if smax else None,
                "power_w_max": float(max(power)) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------
# CPU side (the only place bench.py executes oracle/): the reference's HS-DDP path on the host cores
# ---------------------------------------------------------------------------
def load_oracle():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_py as orc
    import parity_check as pc
    orc.lib()
    return orc, pc


def cpu_workload(orc, wl, args, first=0):
    hk = lambda e, p, q, c: orc.model_hkd_state(orc.default_model(), e, p, q, c)
    return wl.build_cpu(args.config, hk, args.problems, args.plan, first)


def cpu_problem_lists(orc, wl, w, idx, tables):
    for g in wl.GAITS:
        if g not in tables:
            tables[g] = orc.GaitTable(wl.gait_path(g))
    tabs = [tables[w.keys[w.schedule_id[i]][0]] for i in idx]
    k0 = [w.keys[w.schedule_id[i]][1] for i in idx]
    return tabs, k0


def cpu_sample_size(orc, wl, w, seconds, tables):
    """Pilot run -> number of problems that take about `seconds` on all host threads."""
    cores = orc.hardware_concurrency()
    pilot = max(2 * cores, 16)
    idx = np.arange(pilot) % w.n
    tabs, k0 = cpu_problem_lists(orc, wl, w, idx, tables)
    wall, _ = orc.batch_solve(tabs, k0, w.x0[idx], plan=w.plan, n_threads=cores)
    count = int(max(pilot, min(w.n, pilot / wall * seconds)))
    return max(cores, (count // cores) * cores), cores


def cpu_baseline_block(r, cores, count, orc, extra=None):
    s = r["summary"]
    out = {"value": count / r["wall"], "unit": "solves/s", "cores": cores, "kind": "port",
           "detail": ("reference-model+port-solver" if orc.ref_available() else "port-model+port-solver"),
           "model": "reference CasADi C compiled unmodified (oracle/_ref)" if orc.ref_available() else "oracle model port",
           "build": "-O3, no -march, no FMA contraction (the reference's CMakeLists.txt:7)",
           "sample": f"first {count} problems of the workload, one problem per std::thread on {cores} threads, {r['wall']:.1f} s; "
                     f"mean iterations {s[:, 1].mean():.2f}"}
    if extra:
        out.update(extra)
    return out


def cpu_native_rate(orc, tabs, k0, x0, plan, cores):
    """The same oracle compiled -O3 -march=native ON THIS HOST (SURVEY.md §8d: reported separately); best effort."""
    try:
        import ctypes as C
        with tempfile.TemporaryDirectory() as tmp:  # private to this run: the tree may be read-only, /tmp is shared
            so = os.path.join(tmp, "liboracle_hsddp_native.so")
            src = [os.path.join(ROOT, "oracle", f) for f in ("hsddp_oracle.cpp", "oracle_capi.cpp")]
            subprocess.check_call(["g++", "-O3", "-march=native", "-std=c++17", "-fPIC", "-pthread", "-w", "-shared", "-o", so] + src + ["-ldl"],
                                  stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, timeout=300)
            L = C.CDLL(so)
        L.orc_batch_solve.restype = C.c_double
        L.orc_batch_solve.argtypes = orc.lib().orc_batch_solve.argtypes
        L.orc_load_ref.argtypes = [C.c_char_p]
        ref = os.path.join(ROOT, "oracle", "_ref", "libhkd_casadi_ref.so")
        if os.path.exists(ref):
            L.orc_load_ref(ref.encode())
        n = len(tabs)
        tp = (C.c_void_p * n)(*[t.handle for t in tabs])
        k0a = np.ascontiguousarray(k0, np.int32); x0a = np.ascontiguousarray(x0, np.float64)
        o = orc.options_array(); cp = orc.cparams_array()
        dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
        wall = L.orc_batch_solve(tp, k0a.ctypes.data_as(C.POINTER(C.c_int)), dp(x0a), n, C.c_float(plan), orc.default_model(), dp(o), dp(cp), cores, None)
        return n / wall
    except Exception:
        return None


def reference_arm(args):
    """bench.py --impl reference: rank 0 alone, no CUDA library in the process."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    wl = importlib.import_module("hkd-mpc_b200.workloads")  # (workload definition only: pure NumPy, the .so is not loaded)
    orc, pc = load_oracle()
    w = cpu_workload(orc, wl, args)
    tables = {}
    count, cores = cpu_sample_size(orc, wl, w, args.cpu_seconds, tables)
    idx = np.arange(count)
    tabs, k0 = cpu_problem_lists(orc, wl, w, idx, tables)
    walls, summ = [], None
    for it in range(min(args.warmup, 1) + max(1, args.steps)):
        wall, summ = orc.batch_solve(tabs, k0, w.x0[idx], plan=w.plan, n_threads=cores)
        if it >= min(args.warmup, 1):
            walls.append(wall)
    value = count * len(walls) / sum(walls)
    r = {"wall": sum(walls) / len(walls), "summary": summ}
    line = {"impl": "reference", "metric": "batched HS-DDP solves/sec", "value": value, "unit": "solves/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(walls) / len(walls),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_block(args, args.gpus, w.name, len(w.keys)),
            "cpu_baseline": cpu_baseline_block(r, cores, count, orc, {"value": value, "passes": len(walls)}),
            "e2e": {"value": value, "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------
def main():
    args = parse()
    if args.impl == "reference":
        return reference_arm(args)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    pkg = importlib.import_module("hkd-mpc_b200")
    wl = importlib.import_module("hkd-mpc_b200.workloads")
    sh = importlib.import_module("hkd-mpc_b200.sharding")

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the solver has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL's init lines (rank / nranks, transports) must reach the launcher's record, and stdout must stay ONE JSON line:
        # NCCL writes them to a per-process file, which every rank copies to its stderr at the end of the run
        os.environ["NCCL_DEBUG"] = os.environ.get("HSDDP_NCCL_DEBUG", "INFO")
        os.environ["NCCL_DEBUG_SUBSYS"] = os.environ.get("HSDDP_NCCL_DEBUG_SUBSYS", "INIT")
        nccl_log = "/tmp/hsddp_nccl_%d_%d.log" % (os.getpid(), rank)
        os.environ["NCCL_DEBUG_FILE"] = nccl_log
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    opt = pkg.Options()
    n_cmd = 8  # controls / gains shipped per MPC update (HKDMPC.cpp:245-248)

    def time_batch(w, steps, warmup, want_e2e, dump_dir=None):
        """Resident and end-to-end timing of one workload on this rank's GPU; returns a dict (times are max over ranks)."""
        B = pkg.MultiPhaseDDPBatch(local_rank)
        B.set_problems(w.schedules, w.schedule_id)
        x0_pin = torch.from_numpy(w.x0.copy()).pin_memory()
        cmd_pin = torch.zeros((w.n, pkg.CMD_DTYPE.itemsize), dtype=torch.uint8).pin_memory()
        cmd_view = cmd_pin.numpy().view(pkg.CMD_DTYPE).reshape(w.n)

        def step_resident():
            B.reset()
            B.solve_async(opt)

        def step_e2e():
            B.set_initial_condition(x0_pin.numpy())
            B.reset()
            B.solve_async(opt)
            B.mpc_command(n_cmd, out=cmd_view)
            return B.info()

        B.set_initial_condition(w.x0)
        for _ in range(warmup):
            step_resident()
        B.sync()
        B.reset_counters()
        sampler = ClockSampler(local_rank)
        barrier()
        sampler.start()
        B.event_record(0)
        for _ in range(steps):
            step_resident()
        B.event_record(1)
        B.sync()
        barrier()
        clocks = sampler.stop()
        ms_total = sh.max_over_ranks(B.event_elapsed_ms(0, 1), dev)
        info = B.info()
        cnt = B.counters()
        if dump_dir:
            dump_outputs(pkg, B, dump_dir)
        out = dict(B=B, ms_total=ms_total, info=info, clocks=clocks, launches=cnt["solve_launches"] + cnt["step_launches"],
                   sweep_stages_per_step=cnt["sweep_stages"] / max(1, steps), kernel_ms=B.last_solve_ms())
        if want_e2e:
            for _ in range(min(warmup, 2)):
                step_e2e()
            barrier()
            t0 = time.perf_counter()
            B.event_record(4)
            for _ in range(steps):
                step_e2e()
            B.event_record(5)
            B.sync()
            barrier()
            e2e_wall_ms = (time.perf_counter() - t0) * 1e3
            out["e2e_ms"] = sh.max_over_ranks(max(B.event_elapsed_ms(4, 5), e2e_wall_ms), dev)
            out["h2d"] = w.x0.nbytes
            out["d2h"] = cmd_pin.numel() + w.n * pkg.INFO_DTYPE.itemsize
        return out

    # ---- weak: args.problems per GPU ----
    w = getattr(wl, args.config)(pkg, args.problems, args.plan, **({"first": rank * args.problems} if args.config == "config3" else {}))
    dump_dir = args.dump_outputs and (os.path.join(args.dump_outputs, "rank%d" % rank) if world > 1 else args.dump_outputs)
    t = time_batch(w, args.steps, args.warmup, True, dump_dir)
    B = t["B"]
    g = sh.gather_stats(sh.local_stats(t["info"], t["sweep_stages_per_step"]), dev)
    tot = sh.reduce_stats(g)
    n_total = int(tot["n_problems"])
    value = n_total * args.steps / (t["ms_total"] * 1e-3)
    e2e_value = n_total * args.steps / (t["e2e_ms"] * 1e-3)

    # ---- strong: args.problems IN TOTAL, index-sharded over the ranks (BASELINE config 3 as written) ----
    strong = None
    if not args.no_strong:
        if world == 1:
            strong = {"value": value, "ms_per_step": t["ms_total"] / args.steps, "problems_total": n_total, "problems_per_gpu": w.n,
                      "efficiency_vs_n1": 1.0, "e2e_value": e2e_value, "note": "N = 1: identical to the headline measurement"}
        else:
            lo, hi = sh.shard_range(args.problems, rank, world)
            ws = getattr(wl, args.config)(pkg, hi - lo, args.plan, **({"first": lo} if args.config == "config3" else {}))
            ts = time_batch(ws, args.steps, max(3, args.warmup), True)
            # every rank's weak shard is a 16,384-problem batch on one GPU: its time is this run's own N = 1 reference
            strong = {"value": args.problems * args.steps / (ts["ms_total"] * 1e-3), "ms_per_step": ts["ms_total"] / args.steps,
                      "problems_total": args.problems, "problems_per_gpu": hi - lo,
                      "efficiency_vs_n1": (t["ms_total"] / args.steps) / (world * ts["ms_total"] / args.steps),
                      "e2e_value": args.problems * args.steps / (ts["e2e_ms"] * 1e-3), "e2e_ms_per_step": ts["e2e_ms"] / args.steps,
                      "gpu_launches": int(ts["launches"]), "scaling": "strong",
                      "note": "16,384 problems in total, contiguous index ranges per rank, no data-path collective; "
                              "efficiency = (ms of 16,384 problems on ONE GPU, measured in this run) / (N x ms of the sharded batch)"}
            del ts

    # ---- single-solve latency (BASELINE.json: "single-solve p50 latency"): batch = 1, config 1, 101 cold solves ----
    latency = None
    if rank == 0 and not args.no_latency:
        w1 = wl.config1(pkg, args.plan)
        B1 = pkg.MultiPhaseDDPBatch(local_rank)
        B1.set_problems(w1.schedules, w1.schedule_id)
        B1.set_initial_condition(w1.x0)
        dev_ms, wall_ms = [], []
        for rep in range(104):
            t1 = time.perf_counter()
            B1.reset()
            B1.solve(opt)
            i1 = B1.info()
            t2 = time.perf_counter()
            if rep >= 3:
                dev_ms.append(B1.last_solve_ms()); wall_ms.append((t2 - t1) * 1e3)
        latency = {"p50_ms": float(np.median(dev_ms)), "p50_wall_ms": float(np.median(wall_ms)), "p99_ms": float(np.percentile(dev_ms, 99)),
                   "reps": len(dev_ms), "iterations": int(i1["n_iter"][0]),
                   "what": "one cold Mini Cheetah trot solve (config 1), batch 1: p50_ms = solve kernel on the device (CUDA events), "
                           "p50_wall_ms = host wall clock of reset + solve + info read-back"}
        # the reference's MPC tick (HKDMPC.cpp:97-166): shift the horizon by one step (HKDProblem::update), take the "measured"
        # state (here: the plan's next node), warm re-solve with 2 AL x 1 DDP iterations, ship the command
        tick_opt = pkg.Options(max_AL_iter=2, max_DDP_iter=1)
        Bt = wl.gait_batch(pkg, w1, local_rank)
        Bt.solve(opt)
        tick_ms, tick_wall = [], []
        for rep in range(43):
            x_next = Bt.get_rows("Xbar", 1, 1)[:, 0, :].copy()
            t1 = time.perf_counter()
            Bt.mpc_update()
            Bt.set_initial_condition(x_next)
            Bt.solve(tick_opt)
            Bt.mpc_command(n_cmd)
            t2 = time.perf_counter()
            if rep >= 3:
                tick_ms.append(Bt.last_solve_ms() + Bt.last_update_ms()); tick_wall.append((t2 - t1) * 1e3)
        latency["mpc_tick_p50_ms"] = float(np.median(tick_ms))
        latency["mpc_tick_p50_wall_ms"] = float(np.median(tick_wall))
        latency["mpc_tick_what"] = ("one robot, one MPC step: HKDProblem::update on the device (receding-horizon shift) + warm re-solve, 2 AL x 1 DDP "
                                    "iteration; p50_ms = device time of the update and solve kernels, p50_wall_ms = host wall clock incl. the "
                                    "initial-state upload and the command read-back")
        del Bt
        # the same tick for a batch of robots: 4,096 config-3 problems (or the batch, if smaller)
        nb = min(4096, w.n)
        _, eb = wl.define(args.config, 2 * nb, args.plan)
        wb = wl.from_entries(pkg, "mpc tick batch", wl.with_room_for_ticks(eb, 16, args.plan)[:nb], args.plan)
        Bb = wl.gait_batch(pkg, wb, local_rank)
        Bb.solve(opt)
        cmd_b = np.zeros(wb.n, dtype=pkg.CMD_DTYPE)
        walls = []
        for rep in range(13):
            x_next = Bb.get_rows("Xbar", 1, 1)[:, 0, :].copy()
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            Bb.mpc_update()
            Bb.set_initial_condition(x_next)
            Bb.solve(tick_opt)
            Bb.mpc_command(n_cmd, out=cmd_b)
            t2 = time.perf_counter()
            if rep >= 3:
                walls.append(t2 - t1)
        latency["mpc_batch"] = {"robots": wb.n, "tick_ms": float(np.median(walls) * 1e3), "ticks_per_s": float(wb.n / np.median(walls)),
                                "update_ms": Bb.last_update_ms(), "solve_ms": Bb.last_solve_ms(),
                                "what": "wall clock of one MPC step of every robot: update + initial states from the host + re-solve + commands to the host"}
        del Bb
        del B1

    # ---- the reference's other instantiations (SURVEY.md 8f N4): generic sweeps on synthetic plug-in outputs, 4,096 phases x 60 stages ----
    other = None
    if rank == 0 and not args.no_generic:
        other = []
        for xs, us, ys in ((12, 12, 0), (36, 12, 12)):
            ng, Ng = 4096, 60
            one = wl.random_phase(xs, us, ys, Ng, 1, n=8)
            Bg = pkg.SinglePhaseBatch(xs, us, ys, Ng, ng, local_rank)
            for nm in Bg.INPUTS:
                Bg.set(nm, np.ascontiguousarray(np.broadcast_to(one[nm][None], (ng // 8,) + one[nm].shape).reshape((ng,) + one[nm].shape[1:])))
            ts = []
            for _ in range(5):
                ok = Bg.backward_sweep(1e-3)
                ts.append(Bg.last_ms())
            ms = float(np.median(ts[2:]))
            Fg = wl.generic_flop_per_stage(xs, us, ys)
            other.append({"instantiation": "SinglePhase<double,%d,%d,%d>" % (xs, us, ys), "phases": ng, "horizon": Ng, "sweeps_ok": int(ok.sum()),
                          "backward_sweep_ms": ms, "stages_per_s": ng * Ng / (ms * 1e-3), "flop_per_stage": Fg, "tflops": ng * Ng * Fg / (ms * 1e-3) / 1e12})
            del Bg

    if rank == 0:
        mean_stages = float(np.mean([w.schedules[s].n_stages for s in w.schedule_id]))
        info = t["info"]
        kernel_ms = t["ms_total"] / args.steps   # one solve of the batch = one step of the timed region (reset + solve kernels)
        flop_launch = (t["sweep_stages_per_step"] * F_STAGE + float(info["n_iter"].sum()) * mean_stages * F_ITER_STAGE
                       + float(info["n_trials"].sum()) * mean_stages * F_TRIAL_STAGE)
        flop_exec = (t["sweep_stages_per_step"] * F_STAGE_EXECUTED + float(info["n_iter"].sum()) * mean_stages * F_ITER_STAGE
                     + float(info["n_trials"].sum()) * mean_stages * F_TRIAL_STAGE)
        peak_dfma = pkg.fp64_peak_tflops(local_rank, 0)
        peak_dmma = pkg.fp64_peak_tflops(local_rank, 1)
        peak = max(peak_dfma, peak_dmma)
        achieved = flop_launch / (kernel_ms * 1e-3) / 1e12
        bytes_launch = float(info["n_iter"].sum()) * mean_stages * BYTES_STAGE
        try:
            hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
            hbm_src = "MEASURED_PEAKS.json"
        except Exception:
            hbm_peak, hbm_src = 6650.0, "fallback (B200_PROFILING.md)"
        hbm_ach = bytes_launch / (kernel_ms * 1e-3) / 1e9
        # DRAM bytes of one solve from the committed ncu launch list of this workload (profiles/)
        traffic, traffic_src, shares = None, None, None
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "k_solve_traffic.json")))
            if tr.get("config") == args.config and int(tr.get("problems", 0)) == w.n and abs(tr.get("plan", 0.6) - args.plan) < 1e-9:
                traffic, traffic_src = float(tr["dram_bytes_read"]) + float(tr["dram_bytes_write"]), tr.get("source")
                shares = tr.get("kernel_shares")
        except Exception:
            pass
        line = {
            "metric": "batched HS-DDP solves/sec", "value": value, "unit": "solves/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": t["ms_total"] / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_block(args, world, w.name, len(w.schedules)),
            "gpu_launches": int(t["launches"]),
            "e2e": {"value": e2e_value, "unit": "solves/s", "h2d_bytes_per_step": int(t["h2d"]), "d2h_bytes_per_step": int(t["d2h"]),
                    "ms_per_step": t["e2e_ms"] / args.steps,
                    "what": "set_initial_condition(x0 from pinned host) + reset + solve + copy-out to pinned host of the result record and the MPC command of every problem (hkd_command_lcmt payload: 8 controls, body states, 12x12 feedback blocks, foot placements; HKDMPC.cpp:207-298)"},
            "strong": strong,
            "roofline": {"bound": "tensor", "pipe": "FP64 (DFMA / DMMA m8n8k4)", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": achieved / peak, "dense_equivalent": True,
                         "executed": {"tflops": flop_exec / (kernel_ms * 1e-3) / 1e12, "frac": flop_exec / (kernel_ms * 1e-3) / 1e12 / peak,
                                      "flop_per_stage": F_STAGE_EXECUTED, "executed_over_algorithmic": flop_exec / flop_launch,
                                      "what": "FLOP the kernels execute (structure of A, B exploited: 111 DMMA + a 12x12 block elimination per stage) over the same time; `achieved`/`frac` divide the ALGORITHMIC dense 24x24 count (SURVEY.md §8d) by it and are dense-equivalent"},
                         "traffic": traffic, "traffic_unit": "bytes per solve (dram__bytes_read.sum + dram__bytes_write.sum over its launches)",
                         "traffic_source": traffic_src, "kernel_shares": shares,
                         "kernel": "one solve of the batch = the launches of one timed step; the backward-sweep kernel is the dominant one (kernel_shares)",
                         "kernel_ms": kernel_ms,
                         "flop_per_launch": flop_launch,
                         "peak_source": "measured in this run by hsddp_fp64_peak_tflops: DFMA %.1f, DMMA %.1f TFLOP/s "
                                        "(MEASURED_PEAKS.json has no FP64 entry)" % (peak_dfma, peak_dmma),
                         "hbm": {"achieved": hbm_ach, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_ach / hbm_peak,
                                 "bytes_per_launch": bytes_launch, "peak_source": hbm_src}},
            "latency": latency,
            "other_instantiations": other,
            "convergence": {k: float(v) for k, v in tot.items()},
            "clocks": t["clocks"],
        }
        if world == 1 and not args.no_cpu_baseline:
            # CPU baseline + parity of the SAME problems: the oracle solves the first `count` problems of the batch (timed),
            # then again under perturbed arithmetic to classify each problem, and the GPU results of those problems are compared
            orc, pc = load_oracle()
            tables = {}
            count, cores = cpu_sample_size(orc, wl, w, args.cpu_seconds, tables)
            idx = np.arange(count)
            tabs, k0 = cpu_problem_lists(orc, wl, w, idx, tables)
            base, others = pc.oracle_runs(orc, tabs, k0, w.x0[idx], B.max_nodes, B.max_stages, w.plan, k_rows=n_cmd, n_threads=cores)
            well, sens = pc.classify(base, others)
            B.reset(); B.solve(opt)
            gpu = dict(info=B.info()[:count], Xbar=B.get_rows("Xbar", 0, B.max_nodes)[:count], Ubar=B.get_rows("Ubar", 0, B.max_stages)[:count],
                       K=np.ascontiguousarray(np.swapaxes(B.get_rows("K", 0, n_cmd)[:count].reshape(count, n_cmd, 24, 24), -1, -2)))
            rep, _ = pc.compare_gpu(base, well, gpu)
            rep["variants"] = ["ref"] + list(others.keys())
            rep["what"] = ("first %d problems of the batch: oracle (reference CasADi model + restated solver) vs the CUDA path; a problem is "
                           "well-posed when the oracle's own arithmetic variants (model port, FMA-contracted build) take the same decisions "
                           "and agree to 1e-11; on those the CUDA path must take the same decisions (status, iterations, outer iterations, "
                           "backward sweeps, line-search trials) and agree to 1e-9 per row on cost, Xbar, Ubar and the first 8 gain matrices" % count)
            line["parity"] = rep
            extra = {}
            if "fma" in others:
                extra["value_fma_build"] = count / others["fma"]["wall"]
            nat = cpu_native_rate(orc, tabs, k0, w.x0[idx], w.plan, cores)
            if nat:
                extra["value_march_native"] = nat
            line["cpu_baseline"] = cpu_baseline_block(base, cores, count, orc, extra)
            if latency is not None:  # CPU single-solve latency beside the GPU's (config 1, one thread)
                hk = lambda e, p, q, c: orc.model_hkd_state(orc.default_model(), e, p, q, c)
                wc = wl.build_cpu("config1", hk, None, args.plan)
                tb, kk = cpu_problem_lists(orc, wl, wc, [0], tables)
                ts_ = []
                for _ in range(7):
                    wall, _s = orc.batch_solve(tb, kk, wc.x0[:1], plan=wc.plan, n_threads=1)
                    ts_.append(wall * 1e3)
                latency["cpu_single_ms"] = float(np.median(ts_))
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
        try:
            with open(nccl_log) as f:
                sys.stderr.write(f.read())
            os.remove(nccl_log)
        except OSError:
            pass
    return 0


if __name__ == "__main__":
    sys.exit(main())
