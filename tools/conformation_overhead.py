#!/usr/bin/env python
"""What conformation sampling costs: pmc_run(N) against pmc_run_sampled(N, K) on the same handle, and k_conformation
alone.

    python tools/conformation_overhead.py [--reps 5] [--out FILE]

Workloads (bench.py's parameters):
  C2  interacting dielectric n = 512, 4096 chains (64 cases × 64 replicas), N = 500 trials per call
  K1  clustering driver, all pairs + bending, n = 100, 4096 chains, N = 500
  K6  the same as K1 with 100 chains, N = 4000
For K = 100 and 1000 (K6: 100 and 1000; C2 and K1 with N = 1000 for K = 1000): A = pmc_run(N) (pmc_run_ex for the
clustering driver), B = pmc_run_sampled(N, K), C = N / K pmc_run(K) calls.  Each call is timed with CUDA events on the
handle's stream (the calls end in a stream synchronise); A, B and C alternate after a warm-up.  B does what
`pmc_run(K); pmc_sample_conformation()` repeated does, so B − C is the sampling itself and C − A is the per-chunk
re-synchronisation of the running scalars (DESIGN.md §12), plus for C the host round trips B avoids.
k_conformation alone: pmc_sample_conformation repeated, per call, with its FP64 operations (n(n+1)/2 three-term dot
products per chain, 5 FP64 operations each counting an FMA as 2) and bytes (records read, sums read and written).  Each
call ends in a host stream synchronise, so the per-call time is an upper bound on the kernel's and the rates derived
from it are lower bounds; B − C above is the in-stream cost of the same kernel without that synchronise.  The card
name and power limit are read in the same call.
"""
import argparse
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "polymer-stats_b200"))
sys.dont_write_bytecode = True

import polymc as pm  # noqa: E402

C2_KW = dict(n=512, E0=1.0, K1=1.0, K2=0.0, b=1.0, Fx=0.0, chain_type="dielectric", energy_type="interacting")
K_KW = dict(n=100, E0=1.0, K1=1.0, K2=0.0, b=1.0, Fx=0.0, chain_type="dielectric", energy_type="interacting",
            kappa=0.5, clustering=True, adj_ub=0.40)
HBM = 7.7e12
BINS = 100

# (case fields, cases, replicas, clustering driver, trials per timed call)
WORKLOADS = {
    "C2": (C2_KW, 64, 64, False, 500),
    "K1": (K_KW, 64, 64, True, 500),
    "K6": (K_KW, 4, 25, True, 4000),
}


def measure(name, reps):
    import torch
    kw, ncases, R, cluster, n_trials = WORKLOADS[name]
    cases = [pm.make_case(**kw, Fz=0.25 * (1 + j % 8), kT=1.1 ** (j // 8)) for j in range(ncases)]
    stream = torch.cuda.Stream()
    lines = []
    with pm.Ensemble(cases, replicas=R, seed=20260101) as ens:
        ens.set_stream(stream.cuda_stream)
        ens.set_conformation(BINS)
        if cluster:
            ens.begin_stage(1.0)

        def timed(f):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            f()
            e1.record(stream)
            e1.synchronize()
            return e0.elapsed_time(e1)

        run = ens.run_ex if cluster else ens.run
        sampled = ens.run_sampled_ex if cluster else ens.run_sampled
        kname = ens.kernel_name()
        threads = ens.block_threads()
        for every in (100, 1000):
            N = max(n_trials, every)
            a = lambda: run(N, 0, fetch_rows=False)                      # noqa: E731
            b = lambda: sampled(N, every, 0, fetch_rows=False)           # noqa: E731

            def c():
                for _ in range(N // every):
                    run(every, 0, fetch_rows=False)
            for f in (a, b, c, a, b, c):   # warm-up: module loads, buffers, launch shapes
                timed(f)
            ta, tb, tc = [], [], []
            for _ in range(reps):
                ta.append(timed(a))
                tb.append(timed(b))
                tc.append(timed(c))
            ma, mb, mc = statistics.median(ta), statistics.median(tb), statistics.median(tc)
            chunks = N // every
            lines += [
                f"  K = {every}, N = {N}:",
                f"    A pmc_run{'_ex' if cluster else ''}({N})  ms: " + " ".join(f"{t:.3f}" for t in ta) + f"   median {ma:.3f}",
                f"    B pmc_run_sampled{'_ex' if cluster else ''}({N}, {every})  ms: " + " ".join(f"{t:.3f}" for t in tb)
                + f"   median {mb:.3f}",
                f"    C {chunks} x pmc_run{'_ex' if cluster else ''}({every})  ms: " + " ".join(f"{t:.3f}" for t in tc)
                + f"   median {mc:.3f}",
                f"    B - C (the sampling): {(mb - mc) / chunks * 1e3:.1f} us per sample = {100.0 * (mb - mc) / ma:+.2f} % of A; "
                f"C - A (re-synchronisation per chunk): {100.0 * (mc - ma) / ma:+.2f} % of A; B over A: "
                f"{100.0 * (mb - ma) / ma:+.2f} %",
            ]
        L = pm.load()
        calls = 50
        tk = timed(lambda: [L.pmc_sample_conformation(ens._h) for _ in range(calls)]) / calls
        n, c = kw["n"], ens.nchains
        flops = c * (n * (n + 1) / 2) * 5.0
        cols = 8 + 3 * n + BINS
        nbytes = c * (n * 48 + 2 * cols * 8)
    head = [f"{name}: {ncases} cases x {R} replicas = {c} chains, n = {n}, run kernel {kname}, block {threads}"]
    tail = [f"  k_conformation per pmc_sample_conformation call, incl. its host stream synchronise (an upper bound on the "
            f"kernel's time): {tk * 1e3:.1f} us; {flops / 1e9:.3f} GFLOP FP64, at least "
            f"{flops / (tk * 1e-3) / 1e12:.2f} TFLOP/s; {nbytes / 1e6:.2f} MB, at least {nbytes / (tk * 1e-3) / 1e9:.1f} GB/s "
            f"= {100.0 * nbytes / (tk * 1e-3) / HBM:.2f} % of 7.7 TB/s"]
    return head + lines + tail


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if pm.device_count() < 1:
        raise SystemExit("conformation_overhead.py needs a CUDA device")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    out = [f"card: {card}", "timer: CUDA events on the handle's stream; A, B and C alternate, medians of "
           f"{args.reps} triples after two warm-up triples", ""]
    for name in WORKLOADS:
        out += measure(name, args.reps) + [""]
    text = "\n".join(out)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
