#!/usr/bin/env python
"""A/B of the tree's library against another build of it (for instance the parent commit's), in one call.

    python tools/lib_ab.py BASE_LIB [--compare C2,C2f32,C3,C4,C5,K1,K2,K3,K6] [--workloads C2,C3,C5,K1,K6]
                           [--rounds 5] [--steps 3] [--warmup 2] [--out FILE]

1. Builds the tree's library (csrc/Makefile).
2. Outputs: bench.py --dump-outputs of every --compare workload with each library; every array must be bit-identical
   (a change that moves no floating-point operation changes no output).
3. Speed: `PMC_LIB_PATH=… python bench.py --workload W --no-extras --no-cpu-baseline --no-e2e`, the two libraries
   alternating (the order flips every round); median and spread (min … max) of each workload's updates/s, and whether
   the tree's median lies within the base's spread.
The card name and power limit are read in the same call.  Exit status 1 when an output differs.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "polymer-stats_b200", "csrc")
TREE_LIB = os.path.join(ROOT, "polymer-stats_b200", "libpolymc_b200.so")
FAST = ["--no-extras", "--no-cpu-baseline", "--no-e2e"]


def bench(lib, args_):
    env = dict(os.environ, PMC_LIB_PATH=lib)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1"] + args_, env=env, cwd=ROOT,
                         capture_output=True, text=True)
    if out.returncode != 0:
        raise RuntimeError(f"bench.py {args_} failed:\n{out.stderr[-4000:]}")
    return json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])


def compare_outputs(libs, workload, tmp, log):
    dirs = {}
    for name, lib in libs.items():
        dirs[name] = os.path.join(tmp, f"dump_{workload}_{name}")
        bench(lib, ["--workload", workload, "--steps", "1", "--warmup", "1", "--dump-outputs", dirs[name]] + FAST)
    a, b = dirs["base"], dirs["tree"]
    files = sorted(set(os.listdir(a)) | set(os.listdir(b)))
    bad = []
    for f in files:
        if not (os.path.exists(os.path.join(a, f)) and os.path.exists(os.path.join(b, f))):
            bad.append(f"{f} (missing)")
            continue
        x, y = np.load(os.path.join(a, f)), np.load(os.path.join(b, f))
        if x.shape != y.shape or not np.array_equal(x, y, equal_nan=True):
            bad.append(f[:-4])
    log(f"  {workload:6s} {len(files)} arrays: " + ("all bit-identical" if not bad else "DIFFER: " + ", ".join(bad)))
    return not bad


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("base_lib", help="the library to compare against (another build of libpolymc_b200.so)")
    ap.add_argument("--compare", default="C2,C2f32,C3,C4,C5,K1,K2,K3,K6")
    ap.add_argument("--workloads", default="C2,C3,C5,K1,K6")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    log(f"card (name, power limit, max SM clock): {smi}")
    subprocess.check_call(["make", "-C", CSRC, "-s"], stdout=subprocess.DEVNULL)
    libs = {"base": os.path.abspath(args.base_lib), "tree": TREE_LIB}
    ok = True
    with tempfile.TemporaryDirectory() as tmp:
        log("outputs (bench.py --dump-outputs, 1 step after 1 warm-up step), base against tree:")
        for w in [w for w in args.compare.split(",") if w]:
            ok &= compare_outputs(libs, w, tmp, log)
    wls = [w for w in args.workloads.split(",") if w]
    res = {(w, k): [] for w in wls for k in libs}
    for r in range(args.rounds):
        order = list(libs) if r % 2 == 0 else list(reversed(libs))
        for w in wls:
            for k in order:
                j = bench(libs[k], ["--workload", w, "--steps", str(args.steps), "--warmup", str(args.warmup)] + FAST)
                res[(w, k)].append(j["value"])
                log(f"round {r} {w} {k}: {j['value']:.4e} {j['unit']} ({j['ms_per_step']:.2f} ms/step)")
    log("")
    log(f"{'workload':8s} {'build':5s} {'median':>11s} {'min':>11s} {'max':>11s}   tree vs base median")
    for w in wls:
        b = res[(w, "base")]
        for k in libs:
            v = res[(w, k)]
            g = statistics.median(v) / statistics.median(b) - 1.0
            log(f"{w:8s} {k:5s} {statistics.median(v):11.4e} {min(v):11.4e} {max(v):11.4e}   {100 * g:+.2f} %")
        inside = min(b) <= statistics.median(res[(w, "tree")]) <= max(b)
        log(f"{w:8s} tree median within the base's min … max: {inside}")
    log(f"all compared outputs bit-identical: {ok}")
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
