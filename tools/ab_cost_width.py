#!/usr/bin/env python
"""A/B of the materialised pass's cost-tile width on the flagship workload (bench.py, cfg3, one GPU).

    python tools/ab_cost_width.py [--runs 3] [--steps 20] [--warmup 5] [--out FILE] [--shapes FILE]

Alternates bench.py --no-cpu --no-extras runs of the default build (16-bit price words when every worker price fits)
with PM_TUNE_COST=8 (the int64 tile), --runs times each, in one process tree on one card.  Each arm's last run dumps its
outputs (--dump-outputs); they must be equal array for array.  Writes each arm's values, spread and kernel time per
step with the card's name, power limit and max SM clock (nvidia-smi, read-only).  --shapes adds one run per kernel
shape of the 16-bit arm (PM_TUNE_ARGMIN / PM_TUNE_BUILD) and writes their kernel times.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

ARMS = {"u16 (default)": {}, "int64 (PM_TUNE_COST=8)": {"PM_TUNE_COST": "8"}}
# shapes of the 16-bit kernels: pm_argmin16<S, RPW> and rows per CTA of pm_build_cost_fast (see launch_argmin/launch_build)
SHAPES = {"argmin16 S=4 RPW=2, build 512 rows (default)": {},
          "argmin16 S=2 RPW=4": {"PM_TUNE_ARGMIN": "1"}, "argmin16 S=4 RPW=1": {"PM_TUNE_ARGMIN": "2"},
          "argmin16 S=8 RPW=1": {"PM_TUNE_ARGMIN": "3"}, "argmin16 S=4 RPW=4": {"PM_TUNE_ARGMIN": "4"},
          "argmin16 S=8 RPW=2": {"PM_TUNE_ARGMIN": "5"},
          "build 128 rows": {"PM_TUNE_BUILD": "5"}, "build 256 rows": {"PM_TUNE_BUILD": "6"}}


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:   # noqa: BLE001
        return f"nvidia-smi unavailable ({e})"


def bench(env_extra, steps, warmup, dump=None):
    env = dict(os.environ)
    for k in ("PM_TUNE_COST", "PM_TUNE_ARGMIN", "PM_TUNE_BUILD"):
        env.pop(k, None)
    env.update(env_extra)
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--no-cpu", "--no-extras", "--steps", str(steps),
           "--warmup", str(warmup)]
    if dump:
        cmd += ["--dump-outputs", dump]
    p = subprocess.run(cmd, env=env, capture_output=True, text=True, cwd=ROOT)
    if p.returncode != 0:
        raise SystemExit(f"bench.py failed ({env_extra}):\n{p.stderr[-4000:]}")
    return json.loads(p.stdout.strip().splitlines()[-1])


def summary(name, lines):
    vals = [ln["value"] for ln in lines]
    med = statistics.median(vals)
    ker = {k: statistics.median(ln["kernel_ms_per_step"][k] for ln in lines) for k in ("ms_build", "ms_argmin", "ms_resolve")}
    rf = lines[-1]["roofline"] or {}
    return med, (f"{name}: values {[f'{v:.4g}' for v in vals]}  median {med:.4g} evals/s  spread (max-min)/median "
                 f"{(max(vals) - min(vals)) / med:.2%}  ms/step median {statistics.median(ln['ms_per_step'] for ln in lines):.2f}\n"
                 f"    kernel ms/step (median): build {ker['ms_build']:.2f}  argmin {ker['ms_argmin']:.2f}  resolve "
                 f"{ker['ms_resolve']:.2f};  {rf.get('kernel')} {rf.get('achieved', 0):.0f} GB/s, "
                 f"{rf.get('other', {}).get('kernel')} {rf.get('other', {}).get('achieved', 0):.0f} GB/s (engine byte counters)")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_cost_width_ab.txt"))
    ap.add_argument("--shapes", default=None, help="also run each 16-bit kernel shape once and write the times here")
    args = ap.parse_args()
    facts = card()
    out = [f"card: {facts}",
           f"bench.py --no-cpu --no-extras --steps {args.steps} --warmup {args.warmup} (cfg3: 100k asks x 1M workers), "
           f"arms alternated, {args.runs} runs each"]
    res = {k: [] for k in ARMS}
    with tempfile.TemporaryDirectory() as tmp:
        dumps = {k: os.path.join(tmp, f"arm{i}") for i, k in enumerate(ARMS)}
        for r in range(args.runs):
            for k, env in ARMS.items():
                res[k].append(bench(env, args.steps, args.warmup, dumps[k] if r == args.runs - 1 else None))
                print(k, res[k][-1]["value"], file=sys.stderr, flush=True)
        a, b = dumps.values()
        names = sorted(f for f in os.listdir(a) if f.endswith(".npy"))
        assert names == sorted(f for f in os.listdir(b) if f.endswith(".npy")), "the arms dumped different arrays"
        diff = [n for n in names if not np.array_equal(np.load(os.path.join(a, n)), np.load(os.path.join(b, n)))]
    meds = {}
    for k in ARMS:
        meds[k], text = summary(k, res[k])
        out.append(text)
    m16, m64 = meds.values()
    out.append(f"outputs ({', '.join(n[:-4] for n in names)}): {'identical' if not diff else 'DIFFER: ' + ', '.join(diff)}")
    out.append(f"median ratio u16 / int64: {m16 / m64:.3f}")
    text = "\n".join(out) + "\n"
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    open(args.out, "w").write(text)
    print(text)
    if args.shapes:
        lines = [f"card: {facts}", f"16-bit kernel shapes, one bench.py --no-cpu --no-extras --steps 10 --warmup 3 run each (cfg3)"]
        for name, env in SHAPES.items():
            ln = bench(env, 10, 3)
            k = ln["kernel_ms_per_step"]
            lines.append(f"{name}: value {ln['value']:.4g}  build {k['ms_build']:.2f} ms  argmin {k['ms_argmin']:.2f} ms")
            print(lines[-1], file=sys.stderr, flush=True)
        open(args.shapes, "w").write("\n".join(lines) + "\n")
    if diff:
        raise SystemExit(1)


if __name__ == "__main__":
    main()
