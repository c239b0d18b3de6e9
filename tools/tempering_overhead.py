#!/usr/bin/env python
"""What replica exchange costs: pmc_run(N) against pmc_run_tempering(N, 100) on the same handle, and k_exchange alone.

    python tools/tempering_overhead.py [--reps 5] [--out FILE]

Workloads (bench.py's parameters, chains arranged as kT ladders):
  C2  interacting dielectric n = 512, 4096 chains = 8 ladders (Fz = 0.25 … 2.0) of 8 kT rungs (1.0 … 1.1^7) × 64 replicas
  K1  clustering driver, all pairs + bending, n = 100, 4096 chains arranged the same way
  K6  the same as K1 with 100 chains: one ladder of 4 kT rungs × 25 replicas
Each call is timed with CUDA events on the handle's stream (the calls end in a stream synchronise); A (pmc_run /
pmc_run_ex, N = 500 trials; 4000 for K6, as bench.py's steps), B (the tempering twin, an exchange round every 100
trials) and C (N / 100 pmc_run(100) calls, no exchange) alternate after a warm-up.  The tempering call does what
`pmc_run(100); pmc_exchange()` N / 100 times does — a re-synchronisation of the running energies (one full energy evaluation per chain), the run kernel
and one exchange round per chunk — so B − A splits into C − A, the extra re-synchronisations that cutting the
run into chunks costs (plus, for C, the host round trips that B avoids), and what is left, the exchange rounds.
k_exchange alone: pmc_exchange without the host copy of the flags, per round, with the bytes its accepted swaps move
(both chains' records read and written: 4 · n · 48 B per accepted pair) against 7.7 TB/s.  The card name and power
limit are read in the same call.
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


def ladder_cases(kw, nladders, nrungs):
    cases = [pm.make_case(**kw, Fz=0.25 * (1 + j), kT=1.1 ** k) for j in range(nladders) for k in range(nrungs)]
    ladders = [list(range(j * nrungs, (j + 1) * nrungs)) for j in range(nladders)]
    return cases, ladders


# (case fields, ladders, rungs, replicas, clustering driver, trials per timed call = bench.py's step of the workload)
WORKLOADS = {
    "C2": (C2_KW, 8, 8, 64, False, 500),
    "K1": (K_KW, 8, 8, 64, True, 500),
    "K6": (K_KW, 1, 4, 25, True, 4000),
}


def measure(name, reps, every=100):
    import torch
    kw, nl, nr, R, cluster, n_trials = WORKLOADS[name]
    cases, ladders = ladder_cases(kw, nl, nr)
    stream = torch.cuda.Stream()
    with pm.Ensemble(cases, replicas=R, seed=20260101) as ens:
        ens.set_stream(stream.cuda_stream)
        ens.set_ladders(ladders)
        if cluster:
            ens.begin_stage(1.0)
        a = (lambda: ens.run_ex(n_trials, 0, fetch_rows=False)) if cluster else (lambda: ens.run(n_trials, 0, fetch_rows=False))
        b = ((lambda: ens.run_tempering_ex(n_trials, every, 0, fetch_rows=False)) if cluster
             else (lambda: ens.run_tempering(n_trials, every, 0, fetch_rows=False)))

        def timed(f):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            f()
            e1.record(stream)
            e1.synchronize()
            return e0.elapsed_time(e1)

        def c():
            for _ in range(n_trials // every):
                a_chunk()
        a_chunk = ((lambda: ens.run_ex(every, 0, fetch_rows=False)) if cluster
                   else (lambda: ens.run(every, 0, fetch_rows=False)))
        for f in (a, b, c, a, b, c):   # warm-up: module loads, buffers, launch shapes
            timed(f)
        ta, tb, tc = [], [], []
        for _ in range(reps):
            ta.append(timed(a))
            tb.append(timed(b))
            tc.append(timed(c))
        # k_exchange alone (pmc_exchange without copying the flags back)
        L = pm.load()
        rounds = 40
        st0 = ens.exchange_stats()
        tx = timed(lambda: [L.pmc_exchange(ens._h, None) for _ in range(rounds)]) / rounds
        st1 = ens.exchange_stats()
        acc = int((st1["accepts"] - st0["accepts"]).sum()) / rounds
        att = int((st1["attempts"] - st0["attempts"]).sum()) / rounds
        nbytes = acc * 4 * kw["n"] * 48
        kname = ens.kernel_name()
    ma, mb, mc = statistics.median(ta), statistics.median(tb), statistics.median(tc)
    chunks = n_trials // every
    lines = [
        f"{name}: {len(cases)} cases x {R} replicas = {len(cases) * R} chains, n = {kw['n']}, run kernel {kname}",
        f"  A pmc_run{'_ex' if cluster else ''}({n_trials})  ms: " + " ".join(f"{t:.3f}" for t in ta)
        + f"   median {ma:.3f}",
        f"  B pmc_run_tempering{'_ex' if cluster else ''}({n_trials}, {every})  ms: " + " ".join(f"{t:.3f}" for t in tb)
        + f"   median {mb:.3f}",
        f"  C {chunks} x pmc_run{'_ex' if cluster else ''}({every}), no exchange  ms: " + " ".join(f"{t:.3f}" for t in tc)
        + f"   median {mc:.3f}",
        f"  overhead of B over A (medians): {100.0 * (mb - ma) / ma:+.2f} %  ({(mb - ma) / chunks:.4f} ms per chunk); "
        f"C over A: {100.0 * (mc - ma) / ma:+.2f} %; B over C: {100.0 * (mb - mc) / ma:+.2f} % of A",
        f"  k_exchange alone: {tx * 1e3:.1f} us per round (pmc_exchange incl. the flag memset), {att:.0f} pairs attempted, "
        f"{acc:.1f} accepted; {nbytes / 1e6:.3f} MB of records moved = {nbytes / (tx * 1e-3) / 1e9:.2f} GB/s = "
        f"{100.0 * nbytes / (tx * 1e-3) / HBM:.3f} % of 7.7 TB/s",
    ]
    return lines


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if pm.device_count() < 1:
        raise SystemExit("tempering_overhead.py needs a CUDA device")
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
