#!/usr/bin/env python
"""A/B of the two forms of the rectangle's |r'|² (cta_kernels.cuh, PMC_RECT_Q2): the product build (Q2 = 1, from the
projections on the move) against a build with -DPMC_RECT_Q2=0 (r' formed and squared), in one call.

    python tools/rect_q2_ab.py [--rounds 5] [--workloads C2,C3,C5,K1] [--steps 3] [--warmup 2] [--out FILE]

1. Builds both libraries: the product one in the tree (csrc/Makefile), the Q2 = 0 one under a temporary directory.
2. Outputs: bench.py --dump-outputs of C2 with each library; chain states, acceptance rates and normalisers must be
   bit-identical, and the largest relative difference of every other array is printed.
3. Speed: `PMC_LIB_PATH=… python bench.py --workload W --no-extras --no-cpu-baseline --no-e2e`, the two libraries
   alternating (the order flips every round), median and spread (min … max) of each workload's updates/s.
The card name and power limit are read in the same call.
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
EXACT = ("phi", "theta", "acc_rate", "normalizer", "chain_index")


def build(tmp):
    subprocess.check_call(["make", "-C", CSRC, "-s"])
    q0 = os.path.join(tmp, "libpolymc_b200_q0.so")
    subprocess.check_call(["make", "-C", CSRC, "-s", "DEFINES=-DPMC_RECT_Q2=0", f"BUILD={tmp}/build_q0", f"OUT={q0}"])
    return {"q2=0": q0, "q2=1": os.path.join(ROOT, "polymer-stats_b200", "libpolymc_b200.so")}


def bench(lib, args_):
    env = dict(os.environ, PMC_LIB_PATH=lib)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1"] + args_, env=env, cwd=ROOT,
                         capture_output=True, text=True)
    if out.returncode != 0:
        raise RuntimeError(f"bench.py {args_} failed:\n{out.stderr[-4000:]}")
    return json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])


def compare_outputs(libs, tmp, log):
    dirs = {}
    for name, lib in libs.items():
        d = os.path.join(tmp, "dump_" + name.replace("=", ""))
        bench(lib, ["--workload", "C2", "--steps", "1", "--warmup", "1", "--no-extras", "--no-cpu-baseline",
                    "--no-e2e", "--dump-outputs", d])
        dirs[name] = d
    a, b = dirs["q2=0"], dirs["q2=1"]
    ok = True
    for f in sorted(os.listdir(a)):
        x, y = np.load(os.path.join(a, f)), np.load(os.path.join(b, f))
        key = f[:-4]
        if x.shape != y.shape:
            log(f"  {key}: shapes differ {x.shape} {y.shape}"); ok = False; continue
        if key in EXACT:
            same = np.array_equal(x, y, equal_nan=True)
            ok &= same
            log(f"  {key:28s} bit-identical: {same}")
        else:
            d = np.abs(x - y)
            den = np.maximum(np.abs(x), np.abs(y))
            rel = np.where(den > 0, d / np.where(den > 0, den, 1), 0.0)
            # per column: the largest difference against the column's largest magnitude (averages of quantities that
            # sum to about zero, such as transverse components, have large element-wise relative differences)
            xc, dc = x.reshape(len(x), -1), d.reshape(len(d), -1)
            scale = np.abs(xc).max(axis=0)
            colrel = np.where(scale > 0, dc.max(axis=0) / np.where(scale > 0, scale, 1), 0.0)
            worst = int(np.argmax(colrel))
            log(f"  {key:28s} max relative difference {np.nanmax(rel) if rel.size else 0.0:.3e} (element-wise), "
                f"{colrel[worst]:.3e} of the column's largest magnitude (column {worst})")
    return ok


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--workloads", default="C2,C3,C5,K1")
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
    log(f"card: {smi}")
    with tempfile.TemporaryDirectory() as tmp:
        libs = build(tmp)
        log("outputs of C2 (bench.py --dump-outputs, 1 step of 500 trials after 1 warm-up step), q2=0 against q2=1:")
        ok = compare_outputs(libs, tmp, log)
        log(f"  exact arrays identical: {ok}")
        res = {(w, k): [] for w in args.workloads.split(",") for k in libs}
        for r in range(args.rounds):
            order = list(libs) if r % 2 == 0 else list(reversed(libs))
            for w in args.workloads.split(","):
                for k in order:
                    j = bench(libs[k], ["--workload", w, "--steps", str(args.steps), "--warmup", str(args.warmup),
                                        "--no-extras", "--no-cpu-baseline", "--no-e2e"])
                    res[(w, k)].append(j["value"])
                    log(f"round {r} {w} {k}: {j['value']:.4e} {j['unit']} ({j['ms_per_step']:.2f} ms/step)")
        log("")
        log(f"{'workload':8s} {'build':6s} {'median':>11s} {'min':>11s} {'max':>11s}   gain of the median")
        for w in args.workloads.split(","):
            m0 = statistics.median(res[(w, "q2=0")])
            for k in libs:
                v = res[(w, k)]
                g = statistics.median(v) / m0 - 1.0
                log(f"{w:8s} {k:6s} {statistics.median(v):11.4e} {min(v):11.4e} {max(v):11.4e}   {100 * g:+.2f} %")
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
