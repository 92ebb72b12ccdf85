"""Backward-sweep time per round and group of one phased solve (torch.profiler, CUDA activities).

Solves the benchmark's config-3 batch once to warm up, then profiles one solve and attributes every sweep launch
(k_sweep_w1 and k_phase<2>: both are launched every round, one leaves at once) to its group stream and round.  Prints one
JSON line per run and writes it to --out.  The sweep variant comes from the environment (HSDDP_SWEEP_SPEC, ...), which the
library reads when the handle is created.

    HSDDP_SWEEP_SPEC=4 python tools/tail_rounds.py --label spec4 --out tail_spec4.json
"""
import argparse
import importlib
import json
import os
import re
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--problems", type=int, default=16384)
    ap.add_argument("--label", default="")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    pkg = importlib.import_module("hkd-mpc_b200")
    wl = importlib.import_module("hkd-mpc_b200.workloads")
    w = wl.config3(pkg, args.problems)
    B = pkg.MultiPhaseDDPBatch(0)
    B.set_problems(w.schedules, w.schedule_id)
    B.set_initial_condition(w.x0)
    opt = pkg.Options()
    B.reset()
    B.solve(opt)
    B.reset()
    B.reset_counters()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        B.solve(opt)
        torch.cuda.synchronize()
    spec = B.speculation() if hasattr(B, "speculation") else None
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    kernels = [e for e in events if e.get("cat") == "kernel" and "k_" in e.get("name", "")]
    streams = {}
    for e in kernels:
        streams.setdefault(e["args"].get("stream"), []).append(e)
    groups = []
    for sid, ev in streams.items():
        ev.sort(key=lambda e: e["ts"])
        if not any("k_phase<1>" in e["name"] for e in ev):
            continue
        rounds, cur = [], None
        for e in ev:
            if "k_phase<1>" in e["name"]:
                cur = {"w1_us": 0.0, "block_us": 0.0, "round_us": 0.0, "t0": e["ts"]}
                rounds.append(cur)
            if cur is None:
                continue
            if "k_sweep_w1" in e["name"]:
                cur["w1_us"] += e["dur"]
            elif re.search(r"k_phase<2>", e["name"]):
                cur["block_us"] += e["dur"]
            cur["round_us"] = e["ts"] + e["dur"] - cur["t0"]
        for r in rounds:
            del r["t0"]
        tail = [r for r in rounds if r["block_us"] > r["w1_us"]]
        groups.append({"stream": sid, "rounds": len(rounds), "tail_rounds": len(tail),
                       "tail_sweep_ms": round(sum(r["block_us"] for r in tail) / 1e3, 3),
                       "sweep_ms": round(sum(r["w1_us"] + r["block_us"] for r in rounds) / 1e3, 3),
                       "kernel_span_ms": round((ev[-1]["ts"] + ev[-1]["dur"] - ev[0]["ts"]) / 1e3, 3),
                       "per_round": [{k: round(v, 1) for k, v in r.items()} for r in rounds]})
    groups.sort(key=lambda g: -g["kernel_span_ms"])
    res = {"label": args.label, "problems": args.problems, "gpu": torch.cuda.get_device_name(0),
           "HSDDP_SWEEP_SPEC": os.environ.get("HSDDP_SWEEP_SPEC"), "speculation": spec, "groups": groups}
    line = json.dumps(res)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    summary = [{k: g[k] for k in ("rounds", "tail_rounds", "tail_sweep_ms", "sweep_ms", "kernel_span_ms")} for g in groups]
    print(json.dumps({"label": args.label, "speculation": spec, "groups": summary}))


if __name__ == "__main__":
    main()
