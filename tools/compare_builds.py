#!/usr/bin/env python
"""Runs bench.py for several builds of libmrsb.so, alternating them round by round in one process tree, and reports per build
the headline value and where the tick's time went: the stepping kernel alone, the list-only tick, the rebuild pass alone and the
average tick, with the rebuild fraction, the state checksum, the parity record and the secondaries, plus the card name and power
limit read in the same run.

    python tools/compare_builds.py parent=path/a.so new=path/b.so --rounds 3 [--out FILE] [-- <bench.py arguments>]

A build is LABEL=PATH: a library (MRSB_LIB_PATH of its runs), or the directory of another checkout, built, whose own bench.py and
library run (for builds whose C ABI differs from this tree's); LABEL=default runs this tree as built."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def one_run(path, bench_args):
    env = dict(os.environ)
    env.pop("MRSB_LIB_PATH", None)
    root = ROOT
    if os.path.isdir(path):
        root = os.path.abspath(path)
    elif path != "default":
        env["MRSB_LIB_PATH"] = os.path.abspath(path)
    p = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1"] + bench_args, capture_output=True, text=True, env=env, cwd=root)
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    if p.returncode != 0 or not lines:
        raise SystemExit(f"bench.py failed for {path} (exit {p.returncode}):\n{p.stderr[-3000:]}")
    d = json.loads(lines[-1])
    roof, coll = d["roofline"], d["roofline"]["collision_pass"]
    r = {"value": d["value"], "tick_us": d["ms_per_step"] * 1e3, "step_kernel_us": roof["launch_ms"] * 1e3, "list_only_tick_us": coll["ms_list_only_tick"] * 1e3,
         "rebuild_pass_us": coll["ms_rebuild_pass_alone"] * 1e3, "rebuild_fraction": coll["rebuild_fraction"], "roofline_frac": roof["frac"],
         "x_u64_sum": d["state_checksum"]["x_u64_sum"]}
    if d.get("parity"):
        r["parity"] = {"within_tolerance": d["parity"]["within_tolerance"], "pairs_equal": d["parity"]["pairs_equal"]}
    for s in d.get("secondary") or []:
        r[s["config"][:2]] = s["value"]
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("builds", nargs="+", help="LABEL=PATH")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out")
    args, rest = ap.parse_known_args()
    bench_args = [a for a in rest if a != "--"]
    builds = [b.split("=", 1) for b in args.builds]
    runs = {label: [] for label, _ in builds}
    for rnd in range(args.rounds):
        for label, path in builds:
            runs[label].append(one_run(path, bench_args))
            print(json.dumps({"round": rnd, "build": label, **runs[label][-1]}), flush=True)
    summary = {}
    for label, rs in runs.items():
        s = {k: float(np.median([r[k] for r in rs])) for k in rs[0] if isinstance(rs[0][k], float)}
        s["values"] = [r["value"] for r in rs]
        s["x_u64_sum"] = sorted({r["x_u64_sum"] for r in rs})
        if "parity" in rs[0]:
            s["parity_ok"] = all(r["parity"]["within_tolerance"] and r["parity"]["pairs_equal"] for r in rs)
        summary[label] = s
    out = {"card": card(), "bench_args": ["--gpus", "1"] + bench_args, "rounds": args.rounds, "median": summary, "runs": runs}
    print(json.dumps(out["median"]), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
