"""A/B probe of the one-hot execute: `bench.py` over several builds of the library, alternated in one process tree.

    python profiles/probe_oh_exec.py [--workloads cfg3,cfg2] [--reps 3] [--steps 640] [--tracks] [--out FILE] LIB [LIB ...]
    python profiles/probe_oh_exec.py --default [--reps 3] [--out FILE] LIB [LIB ...]

Every LIB is a file name under genvarloader_b200/_lib/ (the library is chosen with GVL_LIB_NAME; nothing is rebuilt on
import, so variant builds sit there side by side, for example the parent commit built as `libgvl_base.so`).  For each
repetition and workload the libraries run one after the other, so drifts of the shared host and of the card's clocks fall
on all of them alike.  Each run is `python bench.py --workload W --steps S --no-tracks --cpu-seconds 0.2`; its `value`
(whole-step bp/s) and `roofline.launch_ms` (one execute launch over a ring of batches, device events) are kept.  With
`--default` each run is plain `python bench.py` (cfg3, 640 steps, tracks leg, CPU baseline), the benchmark as shipped.  The same
call also runs the store-bandwidth microbenchmark (profiles/microbench/fill.py) and reads the card's name, power limit and
maximum SM clock, read-only, so that every number in the JSON comes with the ceiling and the card it was measured on."""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent


def card() -> dict:
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                         check=True).stdout.strip().splitlines()[0]
    return dict(zip(q.split(","), (x.strip() for x in out.split(","))))


def fill_ceiling() -> dict:
    """Pure-store rates of profiles/microbench/fill.py (GB/s), keyed by the line of its output they come from."""
    lib = ROOT / "profiles" / "microbench" / "libfill.so"
    if not lib.exists():
        subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-shared", "-Xcompiler", "-fPIC",
                        "-o", str(lib), str(lib.with_name("fill.cu"))], check=True)
    out = subprocess.run([sys.executable, str(lib.with_name("fill.py"))], capture_output=True, text=True, check=True).stdout
    rates = {}
    for line in out.splitlines():
        m = re.findall(r"(\d+) GB/s", line)
        if m:
            rates[line.split(":")[0].strip()] = int(m[-1])  # (the copy line: bytes written)
    return {"lines": out.splitlines(), "gb_s": rates}


def bench_run(lib: str, workload: str, steps: int, tracks: bool, default: bool = False) -> dict:
    cmd = [sys.executable, str(ROOT / "bench.py")]
    if not default:
        cmd += ["--workload", workload, "--steps", str(steps), "--cpu-seconds", "0.2"] + ([] if tracks else ["--no-tracks"])
    env = dict(os.environ, GVL_LIB_NAME=lib)
    p = subprocess.run(cmd, capture_output=True, text=True, env=env, cwd=ROOT)
    lines = [x for x in p.stdout.splitlines() if x.startswith("{")]
    if p.returncode != 0 or not lines:
        raise RuntimeError(f"{lib} {workload}: bench.py exited {p.returncode}\n{p.stderr[-3000:]}")
    j = json.loads(lines[-1])
    rl = j["roofline"]
    bp_per_step = j["value"] * j["ms_per_step"] * 1e-3
    res = {"value": j["value"], "launch_ms": rl["launch_ms"], "alg_bytes_per_launch": rl["alg_bytes_per_launch"],
           # output bytes only (4 B/bp one-hot): what a store ceiling compares against
           "written_bytes_per_launch": j["output_GBps"] * 1e9 / j["value"] * bp_per_step * rl["batches_per_launch"],
           "kernel": rl["kernel"], "clocks": j.get("clocks")}
    if (tracks or default) and j.get("tracks"):
        res["tracks_value"] = j["tracks"]["value"]
    return res


def summary(runs: list[dict]) -> dict:
    v = np.array([r["value"] for r in runs])
    ms = np.array([r["launch_ms"] for r in runs])
    s = {"value_mean": float(v.mean()), "value_min": float(v.min()), "value_max": float(v.max()),
         "value_spread": float((v.max() - v.min()) / v.mean()),
         "launch_ms_mean": float(ms.mean()), "launch_ms_min": float(ms.min()), "launch_ms_max": float(ms.max()),
         "launch_alg_tb_s": float(runs[0]["alg_bytes_per_launch"] / (ms.mean() * 1e-3) / 1e12),
         "launch_written_tb_s": float(runs[0]["written_bytes_per_launch"] / (ms.mean() * 1e-3) / 1e12)}
    if all("tracks_value" in r for r in runs):
        s["tracks_value_mean"] = float(np.mean([r["tracks_value"] for r in runs]))
    return s


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("libs", nargs="+")
    ap.add_argument("--workloads", default="cfg3")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--steps", type=int, default=640)
    ap.add_argument("--tracks", action="store_true", help="keep bench.py's cfg3t leg (realigned tracks)")
    ap.add_argument("--default", action="store_true", help="plain `python bench.py` (ignores --workloads / --steps / --tracks)")
    ap.add_argument("--no-fill", action="store_true", help="skip the store-bandwidth microbenchmark")
    ap.add_argument("--out", type=Path, default=ROOT / "profiles" / "probe_oh_exec.json")
    args = ap.parse_args()
    for lib in args.libs:
        if not (ROOT / "genvarloader_b200" / "_lib" / lib).exists():
            sys.exit(f"genvarloader_b200/_lib/{lib} is not built")
    if args.default:
        args.workloads, args.steps = "cfg3", 640
    res = {"card": card(), "steps": args.steps, "default_bench": args.default, "libs": args.libs, "runs": {}, "summary": {}}
    if not args.no_fill:
        res["fill"] = fill_ceiling()
    workloads = args.workloads.split(",")
    for rep in range(args.reps):
        for w in workloads:
            for lib in args.libs:
                r = bench_run(lib, w, args.steps, args.tracks, args.default)
                res["runs"].setdefault(w, {}).setdefault(lib, []).append(r)
                print(f"rep {rep} {w:6s} {lib:24s} value {r['value']:.4e}  launch {r['launch_ms']:.4f} ms", flush=True)
    for w in workloads:
        res["summary"][w] = {lib: summary(res["runs"][w][lib]) for lib in args.libs}
        base = res["summary"][w][args.libs[0]]
        for lib in args.libs:
            s = res["summary"][w][lib]
            s["value_gain"] = s["value_mean"] / base["value_mean"] - 1
            s["launch_gain"] = base["launch_ms_mean"] / s["launch_ms_mean"] - 1
            print(f"{w:6s} {lib:24s} value {s['value_mean']:.4e} ({s['value_gain']:+.1%}, spread {s['value_spread']:.1%})  "
                  f"launch {s['launch_ms_mean']:.4f} ms ({s['launch_gain']:+.1%}) = {s['launch_written_tb_s']:.2f} TB/s written, "
                  f"{s['launch_alg_tb_s']:.2f} TB/s algorithmic" + (f", tracks leg {s['tracks_value_mean']:.4e}" if "tracks_value_mean" in s else ""))
    args.out.parent.mkdir(parents=True, exist_ok=True)
    args.out.write_text(json.dumps(res, indent=1) + "\n")
    print(f"card {res['card']}")
    print(f"wrote {args.out}")


if __name__ == "__main__":
    main()
