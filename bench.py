#!/usr/bin/env python
"""bench.py — monomer MC updates/s of the fixed-force MCMC hot path on B200.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on host cores

A "step" is one pass of the hot path over one batch: S trials (default 500 = one --stepout
interval) on every chain of the workload.  The headline is workload C2 (BASELINE.json configs[1]):
interacting dielectric chains, n=512, 4096 independent replicas PER GPU (weak scaling), E0=1, K1=1,
K2=0, kT=1, b=1, Fz=0.5, default step sizes with adaptation on, stepout=500 (SURVEY.md §8d).

One JSON line is printed by rank 0.  Besides the headline keys of the contract it carries
  "workloads": short runs of the other BASELINE configs — C3 (polar n=512, a real (mu, E0, Fz) sweep),
               C4 (the 32 × 32 × 16 (Fz, E0, kT) grid of n=100 non-interacting chains, sharded over the GPUs),
               C5 (n=4096) — and K1 (n=100 all-pairs clustering driver, the reference's most common study),
               each with value, e2e, roofline, clocks;
  "strong":    C2 with 4096 chains in total and C5 with 1184 chains in total over the N GPUs;
  "multi_abi": the same C2 ensemble driven by ONE process over all N GPUs through pmc_multi_* (rank 0 only, after the
               per-rank measurements): one host thread per device inside the library, one NCCL all-gather.
Under torchrun each rank drives one GPU; chains are sharded by global chain id with no data-path
collective; the only collective is the final gather of the per-chain averages (NCCL), inside the e2e region.
`--workload X` runs a single workload as the headline instead (development).
`--dump-outputs DIR` writes what the headline's last timed step left for a caller (rank 0's chains) as DIR/<name>.npy,
so that two builds can be compared output for output on identical, seeded inputs.
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "polymer-stats_b200"))
sys.dont_write_bytecode = True   # the tree may be read-only; the benchmark writes nothing into it

METRIC = "monomer MC updates/sec (whole box), interacting n=512 dielectric chains"
UNIT = "updates/s"
SEED = 20260101

C2_KW = dict(n=512, E0=1.0, K1=1.0, K2=0.0, kT=1.0, b=1.0, Fz=0.5, Fx=0.0, chain_type="dielectric",
             energy_type="interacting")
C5_KW = dict(C2_KW, n=4096)
K_KW = dict(n=100, E0=1.0, K1=1.0, K2=0.0, kT=1.0, b=1.0, Fz=0.25, Fx=0.0, chain_type="dielectric", kappa=0.5,
            clustering=True, adj_ub=0.40)


def c3_grid():
    """SURVEY §8d C3: polar n=512, mu × E0 × Fz grid (64 points); replicas fill 4096 chains per GPU."""
    return [dict(n=512, mu=mu, E0=E0, Fz=Fz, Fx=0.0, kT=1.0, b=1.0, chain_type="polar", energy_type="interacting")
            for mu in (0.01, 0.1, 0.5, 1.0) for E0 in (0.0, 0.1, 1.0, 10.0) for Fz in (-1.0, 0.0, 1.0, 5.0)]


def c4_grid():
    """SURVEY §8d C4: n=100 non-interacting dielectric, 32 Fz × 32 E0 × 16 kT = 16384 points (Fz, E0 in [0,5] linear,
    kT in [0.1,10] log-spaced) — the shape of run/phases-kT-small-n_2023-09-09.jl's grids."""
    Fz = [5.0 * i / 31 for i in range(32)]
    E0 = [5.0 * i / 31 for i in range(32)]
    kT = [0.1 * (100.0 ** (i / 15)) for i in range(16)]
    return [dict(n=100, E0=e, K1=1.0, K2=0.0, kT=t, b=1.0, Fz=f, Fx=0.0, chain_type="dielectric",
                 energy_type="noninteracting") for f in Fz for e in E0 for t in kT]


# name: dict(cases=[kwargs...], replicas (per case, per GPU for weak / total for strong), S trials per step, stepout,
#            scaling: "weak" (replicas per GPU fixed) | "strong" (the case list is split over the GPUs), e2e: "state"
#            (host state in, host rows out) | "sweep" (polymc.sweep.run_sweep: case table in, gathered averages out))
WORKLOADS = {
    "C2": dict(cases=[C2_KW], replicas=4096, S=500, stepout=500, scaling="weak", e2e="state",
               desc="C2: interacting dielectric chains n=512, 4096 replicas per GPU"),
    # opt-in precision of north_star's "ΔU in fp64, or in fp32 with a stated tolerance" (pmc_set_pair_precision): the
    # rectangle of every trial in FP32, state / row / acceptance / accumulators FP64.  Never the headline.
    "C2f32": dict(cases=[C2_KW], replicas=4096, S=500, stepout=500, scaling="weak", e2e="state", precision="fp32",
                  desc="C2 with the FP32 rectangle (stated tolerance: include/polymc.h pmc_set_pair_precision)"),
    "C3": dict(cases=c3_grid(), replicas=64, S=500, stepout=500, scaling="weak", e2e="sweep",
               desc="C3: polar chains n=512 with dipole-dipole coupling, 4 mu x 4 E0 x 4 Fz sweep (64 points) x 64 replicas "
                    "per GPU"),
    "C4": dict(cases=c4_grid(), replicas=1, S=100000, stepout=500, scaling="strong", e2e="sweep",
               desc="C4: phase-diagram sweep, 32 Fz x 32 E0 x 16 kT = 16384 points x n=100 non-interacting chains, 1e5 "
                    "trials per point (SURVEY 8d), grid split over the GPUs"),
    "C5": dict(cases=[C5_KW], replicas=148, S=200, stepout=200, scaling="weak", e2e="state",
               desc="C5: long interacting dielectric chains n=4096, 148 chains per GPU"),
    # the clustering driver (mcmc_clustering_eap_chain.jl; SURVEY §8f rank 1-2), shapes of its launchers:
    # run/phases-kT-small-n_2023-09-09.jl (all-pairs, bending), run/Ising_2025-12-17.jl, run/phases-big_2023-05-18.jl
    "K1": dict(cases=[dict(K_KW, energy_type="interacting")], replicas=4096, S=500, stepout=250, scaling="weak",
               e2e="state", desc="K1: clustering driver, all-pairs + bending, n=100, 4096 chains per GPU"),
    "K2": dict(cases=[dict(K_KW, energy_type="Ising")], replicas=65536, S=2000, stepout=250, scaling="weak", e2e="state",
               desc="K2: clustering driver, Ising + bending, n=100, 65536 chains per GPU"),
    "K3": dict(cases=[dict(K_KW, n=400, energy_type="cutoff", cutoff_radius=7.5)], replicas=2368, S=200, stepout=100,
               scaling="weak", e2e="state", desc="K3: clustering driver, cut-off + bending, n=400, 2368 chains per GPU"),
    # the size of the reference's own studies: 20 cases × 25 runs (run/Ising_2025-12-17.jl)
    "K4": dict(cases=[dict(K_KW, energy_type="Ising")], replicas=500, S=20000, stepout=2500, scaling="weak", e2e="state",
               desc="K4: clustering driver, Ising + bending, n=100, 500 chains"),
    "K5": dict(cases=[dict(K_KW, energy_type="interacting")], replicas=500, S=2000, stepout=250, scaling="weak",
               e2e="state", desc="K5: clustering driver, all-pairs + bending, n=100, 500 chains"),
    "K6": dict(cases=[dict(K_KW, energy_type="interacting")], replicas=100, S=4000, stepout=500, scaling="weak",
               e2e="state", desc="K6: clustering driver, all-pairs + bending, n=100, 100 chains per GPU — the size of one study "
                                 "of the reference (a handful of cases x 25 runs); eight one-warp teams per chain on different trials"),
    # strong scaling: the TOTAL is fixed and split over the GPUs
    "C2s": dict(cases=[C2_KW], replicas=4096, S=500, stepout=500, scaling="strong", e2e="state",
                desc="C2 strong: interacting dielectric n=512, 4096 chains in total"),
    "C5s": dict(cases=[C5_KW], replicas=1184, S=50, stepout=50, scaling="strong", e2e="state",
                desc="C5 strong: interacting dielectric n=4096, 1184 chains in total (8 x 148 SMs)"),
}
# ncu `--set full` capture of the headline launch (dram__bytes_read.sum + dram__bytes_write.sum per launch), from the
# profile named here; other workloads: null unless listed
TRAFFIC = {"C2": (1.136e8, "profiles/r02a_ncu_full_k_run_cta_win_C2.txt: 104.9 MB read (the chain records, once per launch) + 8.7 MB written"),
           "C5": (2.93e7, "profiles/r02a_ncu_full_k_run_cta_pair_C5.txt (captured at 50 trials per launch; the records are read once per launch whatever its length)")}


def flops_per_update(n: int, energy_type: str) -> float:
    """Algorithmic FP64 flop per update (SURVEY.md §8d / BASELINE.md §3)."""
    if energy_type in ("interacting", "cutoff"):
        return 2.0 * 34.0 * ((n - 1) * (n - 2) / 6.0 + (n - 1))
    return 210.0 if energy_type == "Ising" else 66.0


class ClockSampler:
    """nvidia-smi clocks / throttle reasons for the whole run (B200_PROFILING.md recipe), time-stamped on arrival so
    that every workload reports the samples of its own timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, device: int):
        self.device = device
        self.proc = None
        self.samples = []   # (t, sm, smmax, power, [reasons])

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                self.samples.append((time.perf_counter(), float(f[0]), float(f[1]), float(f[2]),
                                     [nm for nm, v in zip(self.NAMES, f[3:7]) if v.lower().startswith("active")]))
            except ValueError:
                continue

    def window(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)   # let the sample that covers the end of the window arrive
        inside = [s for s in self.samples if t0 <= s[0] <= t1 + 0.15]
        if not inside and self.samples:     # a region shorter than the sampling period: the nearest sample
            inside = [min(self.samples, key=lambda s: abs(s[0] - 0.5 * (t0 + t1)))]
        if not inside:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no sample"]}
        return {"sm_mhz": statistics.median(s[1] for s in inside), "sm_max_mhz": max(s[2] for s in inside),
                "power_w_max": max(s[3] for s in inside), "samples": len(inside),
                "reasons": sorted({r for s in inside for r in s[4]})}

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()


def metric_of(name, kw):
    if name == "C2":
        return METRIC
    drv = "clustering driver, " if kw.get("clustering") else ""
    return f"monomer MC updates/sec (whole box), {drv}{kw['energy_type']} n={kw['n']} {kw['chain_type']} chains"


def make_config(name, W, per_gpu, S, stepout, world):
    """The `config` object — identical for both arms."""
    kw = W["cases"][0]
    cfg = {"workload": f"{W['desc']}, {S} trials per step, stepout={stepout}",
           "chains_per_gpu": per_gpu, "trials_per_step": S, "seed": SEED, "scaling": W["scaling"],
           "l2": "flushed between timed steps (256 MiB write)"}
    if len(W["cases"]) == 1:
        cfg.update(kw)
    else:
        cfg.update({k: v for k, v in kw.items() if all(c[k] == v for c in W["cases"])})
        cfg["sweep_points"] = len(W["cases"])
    return cfg


# ------------------------------------------------------------------------------------------------------------------
# CPU arm
# ------------------------------------------------------------------------------------------------------------------
def cpu_reference_run(kw, n_chains, trials, threads, algo=0):
    """The reference algorithm (deep-copy-free full energy recompute per trial, oracle algo 0) on host threads, one
    chain per thread at a time, timed with the `-O3 -march=native` build compiled on this host (BASELINE.md §4)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle as O
    okw = {k: v for k, v in kw.items()}
    oc = O.make_case(**okw)
    secs = O.bench(oc, SEED, algo, n_chains, trials, threads, native=True)
    return n_chains * trials / secs, secs


def cpu_build_flags():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle as O
    return O.native_lib()[1]


def sized_cpu_sample(kw, threads, target_s, algo=0):
    """Pick trials/chain so that `threads` chains take about target_s seconds."""
    probe_trials = 20 if kw["energy_type"] == "interacting" and kw["n"] >= 512 else 2000
    if kw["n"] >= 4096:
        probe_trials = 2
    ups, secs = cpu_reference_run(kw, threads, probe_trials, threads, algo)
    per_thread_rate = ups / threads
    return max(probe_trials, int(per_thread_rate * target_s))


def run_reference_arm(args, rank, world):
    """`--impl reference`: the reference's own CPU algorithm for the path on the box's host cores.
    Julia is not installable here, so the timed code is the oracle's C restatement of the reference
    algorithm (kind "port"): full O(n²) energy recompute per trial, one chain per thread."""
    if rank != 0:
        return 0
    W = WORKLOADS[args.workload]
    kw = W["cases"][0]
    per_gpu = args.chains_per_gpu or W["replicas"] * (len(W["cases"]) if W["scaling"] == "weak" else 1)
    S = args.trials_per_step or W["S"]
    stepout = min(W["stepout"], S)
    threads = os.cpu_count() or 1
    trials = sized_cpu_sample(kw, threads, target_s=args.ref_step_seconds)
    for _ in range(args.warmup):
        cpu_reference_run(kw, threads, max(1, trials // 10), threads)
    t_total, updates = 0.0, 0
    for _ in range(args.steps):
        ups, secs = cpu_reference_run(kw, threads, trials, threads)
        t_total += secs
        updates += threads * trials
    value = updates / t_total
    sample = (f"{threads} chains x {trials} trials per step (one chain per thread), n={kw['n']} "
              f"{kw['energy_type']} {kw['chain_type']}, same parameters as the GPU arm")
    line = {
        "impl": "reference", "metric": metric_of(args.workload, kw), "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": make_config(args.workload, W, per_gpu, S, stepout, world),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                         "build": cpu_build_flags(),
                         "note": "C restatement of the reference algorithm (oracle/polymc_oracle.c, algo 0); "
                                 "Julia is not installed in this image"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)
    return 0


_REAL_STDOUT = None


def emit(line: dict):
    """Exactly one JSON line on the real stdout (libraries such as NCCL may print to fd 1; everything
    else is redirected to stderr for the duration of the run)."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, data)
    else:
        sys.stdout.write(data.decode())
        sys.stdout.flush()


# ------------------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------------------
class Ctx:
    pass


def shard_of(W, rank, world, chains_override=None):
    """(case kwargs list of this rank, replicas per case, chain_id_base, chains on this rank, chains on all ranks).
    weak: every rank runs the whole case list with `replicas` replicas (global replica index = rank·replicas + r);
    strong: the chains (case-major, cases × replicas) are split into contiguous blocks of whole cases or, for a
    single-case workload, of replicas."""
    cases, rep = W["cases"], W["replicas"]
    if chains_override:
        rep = max(1, chains_override // len(cases))
    if W["scaling"] == "weak":
        per = len(cases) * rep
        return cases, rep, rank * per, per, per * world
    if len(cases) == 1:
        lo, hi = rep * rank // world, rep * (rank + 1) // world
        return cases, hi - lo, lo, hi - lo, rep
    lo, hi = len(cases) * rank // world, len(cases) * (rank + 1) // world
    return cases[lo:hi], rep, lo * rep, (hi - lo) * rep, len(cases) * rep


DUMP_BYTES = 63_000_000   # array data of one dump; with the .npy headers it stays below 64 MB


def dump_outputs(ens, clustering: bool, out_dir: str):
    """Write what a caller of the timed path receives after its last step, as float64 .npy files: the chain states
    (phi, theta), the per-chain averages, acceptance rates, normalisers and step diagnostics, and for the clustering
    driver its extra averages and cluster statistics.  When all of it exceeds DUMP_BYTES, the same fixed, seeded sample
    of chains is taken from every array; chain_index.npy names the chains written."""
    import numpy as np
    phi, theta = ens.get_state_all()
    avg, ar, nrm = ens.averages()
    arrays = {"phi": phi, "theta": theta, "averages": avg, "acc_rate": ar, "normalizer": nrm,
              "diagnostics": ens.diagnostics()}
    if clustering:
        arrays.update(extra_averages=ens.extra_averages(), cluster_stats=ens.cluster_stats())
    per_chain = 8 * (1 + sum(a[0].size for a in arrays.values()))
    keep = min(ens.nchains, DUMP_BYTES // per_chain)
    idx = np.arange(ens.nchains)
    if keep < ens.nchains:
        idx = np.sort(np.random.default_rng(SEED).choice(ens.nchains, keep, replace=False))
    arrays["chain_index"] = idx
    os.makedirs(out_dir, exist_ok=True)
    for nm, a in arrays.items():
        a = a if nm == "chain_index" else a[idx]
        np.save(os.path.join(out_dir, nm + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def measure(cx: Ctx, name: str, steps: int, warmup: int, want_e2e=True, chains_override=None, S_override=None,
            dump_dir=None):
    """One workload on this rank's GPU: device-timed resident `value`, e2e through the public API, roofline;
    with dump_dir, the outputs of the last timed step are written there (dump_outputs)."""
    import numpy as np
    import torch
    import torch.distributed as dist
    pm = cx.pm
    W = WORKLOADS[name]
    S = S_override or W["S"]
    stepout = min(W["stepout"], S)
    my_cases, rep, base, mine, total = shard_of(W, cx.rank, cx.world, chains_override)
    kw0 = W["cases"][0]
    n = kw0["n"]
    clustering = bool(kw0.get("clustering"))
    cases = [pm.make_case(**kw) for kw in my_cases]
    ens = pm.Ensemble(cases, replicas=rep, seed=SEED, device=cx.local_rank, chain_id_base=base)
    ens.set_stream(cx.stream.cuda_stream)
    fp32 = W.get("precision") == "fp32"
    if fp32:
        ens.set_pair_precision("fp32")
    kernel = ens.kernel_name()
    if clustering:
        ens.begin_stage(1.0)   # a fresh mcmc(nsteps, pargs, chain) call (mcmc_clustering_eap_chain.jl:171-265)

    def run_resident():
        if clustering:
            ens.run_ex(S, stepout, fetch_rows=False)
        else:
            ens.run(S, stepout, fetch_rows=False)

    for _ in range(max(warmup, 0)):
        run_resident()
    launches0 = ens.launch_count()
    cx.barrier()
    t_w0 = time.perf_counter()
    step_ms, kernel_ms = [], []
    for _ in range(steps):
        cx.flush.fill_(1.0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(cx.stream)
        run_resident()
        e1.record(cx.stream)
        e1.synchronize()
        step_ms.append(e0.elapsed_time(e1))
        kernel_ms.append(ens.last_run_ms())
    cx.barrier()
    t_w1 = time.perf_counter()
    launches = ens.launch_count() - launches0
    if dump_dir and cx.rank == 0:
        dump_outputs(ens, clustering, dump_dir)
    total_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device=cx.dev)
    if cx.world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms.item())
    value = total * S * steps / (total_ms * 1e-3)
    clocks = cx.sampler.window(t_w0, t_w1)

    # ---- roofline of the MCMC kernel (this rank's launch) ----------------------------------------------------------
    F = flops_per_update(n, kw0["energy_type"])
    if clustering and kw0["energy_type"] in ("interacting", "cutoff"):
        # changed pair terms of a composite trial: segment×everything + heads×tails, from the measured cluster sizes
        cs = ens.cluster_stats()
        trials = ens.diagnostics()[:, 5].sum()
        mean_seg = 1.0 + (cs[:, 1].sum() - cs[:, 0].sum()) / max(1.0, trials)
        F = 2.0 * 34.0 * ((n - mean_seg) * (n - mean_seg - 1) / 6.0 + mean_seg * (n - 1))
    kavg_ms = sum(kernel_ms) / len(kernel_ms)
    achieved_tf = mine * S * F / (kavg_ms * 1e-3) / 1e12
    pair_bound = kw0["energy_type"] in ("interacting", "cutoff")
    traffic = TRAFFIC.get(name) if (not chains_override and not S_override and cx.world == 1) else None
    roofline = {
        "bound": "fp64", "kernel": kernel, "kernel_source": "pmc_kernel_name (the library's own launch decision)",
        "achieved": achieved_tf, "peak": cx.probe_tf, "unit": "TFLOP/s",
        "frac": achieved_tf / cx.probe_tf, "traffic": traffic[0] if traffic else None,
        "traffic_source": traffic[1] if traffic else None,
        "peak_source": "measured in this run: DFMA-only microbenchmark pmc_fp64_peak_probe (MEASURED_PEAKS.json "
                       "holds no FP64 figure)",
        "peak_derived": cx.derived_tf, "frac_of_derived": achieved_tf / cx.derived_tf,
        "flop_per_update": F, "updates_per_launch": mine * S, "kernel_ms_avg": kavg_ms,
        "kernel_share_of_step": kavg_ms * len(kernel_ms) / sum(step_ms),
    }
    if fp32:   # the rectangle runs on the FP32 pipe: 128 FMA per clock per SM (no measured FP32 figure in MEASURED_PEAKS.json)
        peak32 = 148 * 128 * 2 * 1.965e9 / 1e12
        roofline.update({"bound": "fp32", "peak": peak32, "frac": achieved_tf / peak32, "peak_derived": peak32,
                         "frac_of_derived": achieved_tf / peak32,
                         "peak_source": "derived: 148 SMs x 128 FP32 FMA per clock x 1.965 GHz",
                         "tolerance": "relative error <= 5e-7 (1 + amplification) per pair term, include/polymc.h; "
                                      "tests/test_gpu_fp32.py"})
    if not pair_bound:
        roofline["note"] = ("O(1)-energy chains are latency / transcendental bound (2 Philox, 2 sincos, log, exp per trial): "
                            "the flop fraction is informational, updates/s is the figure (SURVEY §8d)")

    # ---- e2e through the public API --------------------------------------------------------------------------------
    e2e = None
    if want_e2e and W["e2e"] == "state":
        phi_h = torch.empty((mine, n), dtype=torch.float64).pin_memory()
        th_h = torch.empty((mine, n), dtype=torch.float64).pin_memory()
        p0, t0 = ens.get_state_all()
        phi_h.numpy()[:] = p0
        th_h.numpy()[:] = t0
        rows = max(1, S // stepout) if stepout > 0 else 0
        cols = 19 if clustering else 17
        traj_h = torch.empty((mine, rows, 8), dtype=torch.float64).pin_memory()
        roll_h = torch.empty((mine, rows, cols), dtype=torch.float64).pin_memory()
        L = pm.load()
        from polymc.lib import _check, _dp

        def e2e_step():
            ens.set_state_all(phi_h.numpy(), th_h.numpy())                 # H2D + cache rebuild
            if clustering:                                                 # hot loop + D2H rows
                _check(L.pmc_run_ex(ens._h, S, stepout, _dp(traj_h.numpy()), _dp(roll_h.numpy()), None))
            else:
                ens.run(S, stepout, traj=traj_h.numpy(), roll=roll_h.numpy())
            avg, ar, nrm = ens.averages()                                  # D2H results
            if cx.world > 1:                                               # final gather of averages (NCCL)
                t = torch.from_numpy(np.concatenate([avg, ar[:, None], nrm[:, None]], axis=1)).to(cx.dev)
                pad = torch.zeros((cx.max_over_ranks(mine), t.shape[1]), dtype=t.dtype, device=cx.dev)
                pad[: t.shape[0]] = t
                outs = [torch.empty_like(pad) for _ in range(cx.world)]
                dist.all_gather(outs, pad)
                torch.cuda.synchronize(cx.dev)
            return avg
        e2e_step()
        cx.barrier()
        t0w = time.perf_counter()
        for _ in range(steps):
            e2e_step()
        cx.barrier()
        dt = torch.tensor([time.perf_counter() - t0w], dtype=torch.float64, device=cx.dev)
        if cx.world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        h2d = phi_h.numel() * 8 + th_h.numel() * 8
        d2h = traj_h.numel() * 8 + roll_h.numel() * 8 + mine * (16 + 2) * 8
        e2e = {"value": total * S * steps / float(dt.item()), "unit": UNIT,
               "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "ms_per_step": 1e3 * float(dt.item()) / steps,
               "api": "polymc.Ensemble.set_state_all + run(host traj/roll) + averages (C ABI pmc_*), pinned host buffers"}
    ens.close()
    if want_e2e and W["e2e"] == "sweep":
        # the call a study makes: polymc.sweep.run_sweep — case table in (H2D of the per-chain constants, chains drawn
        # on the device), S trials, per-chain averages + raw sums out (D2H), gathered over the ranks (NCCL all_gather)
        from polymc import sweep
        all_cases = pm.CaseTable([pm.make_case(**kw) for kw in W["cases"]])   # the host-resident case table
        reps = rep * cx.world if W["scaling"] == "weak" else rep

        def sweep_step():
            return sweep.run_sweep(all_cases, reps, S, 0, SEED, cx.local_rank, cx.dev if cx.world > 1 else None)
        sweep_step()
        cx.barrier()
        t0w = time.perf_counter()
        for _ in range(steps):
            res = sweep_step()
        cx.barrier()
        dt = torch.tensor([time.perf_counter() - t0w], dtype=torch.float64, device=cx.dev)
        if cx.world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        assert res["avg"].shape[0] == total
        e2e = {"value": total * S * steps / float(dt.item()), "unit": UNIT,
               "h2d_bytes_per_step": int(mine * 160), "d2h_bytes_per_step": int(mine * (16 + 2 + 17 + 8) * 8),
               "ms_per_step": 1e3 * float(dt.item()) / steps,
               "api": "polymc.sweep.run_sweep: handle creation (case table H2D, chains drawn on device) + S trials + "
                      "averages/sums D2H + all_gather over the ranks; no per-case rows"}
    return {"metric": metric_of(name, kw0), "value": value, "unit": UNIT, "ms_per_step": total_ms / steps,
            "steps": steps, "warmup": warmup, "scaling": W["scaling"], "chains_total": total, "chains_per_gpu": mine,
            "config": make_config(name, W, mine, S, stepout, cx.world), "gpu_launches": int(launches),
            "clocks": clocks, "e2e": e2e, "roofline": roofline, "wall_s_timed_region": t_w1 - t_w0}


def measure_multi_abi(cx: Ctx, steps: int, warmup: int):
    """C2 (4096 chains per GPU) driven by ONE process over all the box's GPUs through pmc_multi_* — what a Julia host
    calls (julia/polymc_host.jl `--devices`).  Rank 0 only; the other ranks wait at the barrier with idle GPUs."""
    import numpy as np
    import torch
    pm = cx.pm
    G = cx.world
    if pm.device_count() < G:
        return {"skipped": f"only {pm.device_count()} device(s) visible to rank 0"}
    W = WORKLOADS["C2"]
    S, stepout, per = W["S"], W["stepout"], W["replicas"]
    case = pm.make_case(**W["cases"][0])
    with pm.MultiEnsemble(case, replicas=per * G, seed=SEED, ndevices=G) as m:
        n, R = m.n, m.nchains
        for _ in range(warmup):
            m.run(S, stepout, fetch_rows=False)
        t0 = time.perf_counter()
        kms = []
        for _ in range(steps):
            m.run(S, stepout, fetch_rows=False)
            kms.append(m.last_run_ms())
        dt = time.perf_counter() - t0
        value = R * S * steps / dt
        phi, th = m.get_state_all()
        phi_h, th_h = torch.from_numpy(phi).pin_memory(), torch.from_numpy(th).pin_memory()
        rows = S // stepout
        traj_h = torch.empty((R, rows, 8), dtype=torch.float64).pin_memory()
        roll_h = torch.empty((R, rows, 17), dtype=torch.float64).pin_memory()

        def step():
            m.set_state_all(phi_h.numpy(), th_h.numpy())
            m.run(S, stepout, traj=traj_h.numpy(), roll=roll_h.numpy())
            return m.gather()
        step()
        t0 = time.perf_counter()
        for _ in range(steps):
            tab = step()
        dte = time.perf_counter() - t0
        assert tab.shape == (R, 24) and np.all(tab[:, 17] > 0)
        return {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": G, "chains_total": R, "ms_per_step": 1e3 * dt / steps,
                "timing": "host wall clock around the synchronous pmc_multi_run (all devices)",
                "slowest_device_kernel_ms": sum(kms) / len(kms), "gather_backend": m.gather_backend(),
                "e2e": {"value": R * S * steps / dte, "unit": UNIT, "ms_per_step": 1e3 * dte / steps,
                        "h2d_bytes_per_step": int(2 * R * n * 8), "d2h_bytes_per_step": int(R * rows * 25 * 8 + R * 24 * 8),
                        "api": "pmc_multi_set_state_all + pmc_multi_run(host traj/roll) + pmc_multi_gather (one "
                               "ncclAllGather), single process, one host thread per device inside the library"},
                "gpu_launches": int(m.launch_count())}


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="graft", choices=["graft", "reference"])
    ap.add_argument("--workload", default="C2", choices=sorted(WORKLOADS))
    ap.add_argument("--chains-per-gpu", type=int, default=None)
    ap.add_argument("--trials-per-step", type=int, default=None)
    ap.add_argument("--cpu-baseline-seconds", type=float, default=10.0)
    ap.add_argument("--ref-step-seconds", type=float, default=8.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="headline only: skip workloads / strong / multi_abi")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the headline's outputs after its last timed step to DIR/<name>.npy (float64, < 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference_arm(args, rank, world)

    import torch
    import torch.distributed as dist
    import polymc as pm

    if not torch.cuda.is_available() or pm.device_count() < 1:
        emit({"error": "no CUDA device: libpolymc_b200 has no CPU fallback"})
        return 2
    torch.cuda.set_device(local_rank)
    cx = Ctx()
    cx.pm, cx.rank, cx.world, cx.local_rank = pm, rank, world, local_rank
    cx.dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=cx.dev)
        # a host-side barrier for the phase in which rank 0 alone drives every GPU: a rank parked in an NCCL barrier
        # keeps a spinning kernel on its GPU, and two contexts on one GPU time-slice
        cx.cpu_group = dist.new_group(backend="gloo")
    cx.stream = torch.cuda.current_stream(cx.dev)
    # L2 flush buffer (larger than the 126 MB L2), written between timed steps
    cx.flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=cx.dev)

    def barrier():
        torch.cuda.synchronize(cx.dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(cx.dev)

    def max_over_ranks(v):
        if world == 1:
            return int(v)
        t = torch.tensor([int(v)], dtype=torch.int64, device=cx.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return int(t.item())
    cx.barrier, cx.max_over_ranks = barrier, max_over_ranks
    # measured FP64 roofline denominator (DFMA microbenchmark, before the clocks heat up)
    cx.probe_tf = max(pm.fp64_peak_probe(local_rank, 1 << 16)[0] for _ in range(3))
    cx.derived_tf = 148 * 64 * 2 * 1.965e9 / 1e12
    cx.sampler = ClockSampler(local_rank)
    cx.sampler.start()
    atexit.register(cx.sampler.stop)   # no nvidia-smi left running when a measurement raises

    head = measure(cx, args.workload, args.steps, args.warmup, want_e2e=not args.no_e2e,
                   chains_override=args.chains_per_gpu, S_override=args.trials_per_step, dump_dir=args.dump_outputs)

    extras = args.workload == "C2" and not args.no_extras and not args.chains_per_gpu and not args.trials_per_step
    workloads, strong, multi_abi = {}, {}, None
    if extras:
        xs = max(2, min(args.steps, 3))
        for nm in ("C3", "C4", "C5", "K1", "K6", "C2f32"):
            workloads[nm] = measure(cx, nm, xs, 3, want_e2e=not args.no_e2e)
        workloads["C2f32"]["dtype"] = "f32 rectangle pair terms; f64 state, row terms, acceptance and accumulators (opt-in, not the headline)"
        workloads["C4"]["limiter"] = ("device-timed: one chain per warp, 32 speculative trials per window; issue slots 61 % busy, the "
                                      "transcendental core (2 sincos, log, exp, 2 Philox per trial) is a quarter of the samples; at 8 GPUs "
                                      "2048 chains per GPU are 0.86 of one wave (13.8 warps per SM); e2e through run_sweep adds ~1 ms of host "
                                      "work per call (contiguous case table, one all-gather)")
        workloads["K6"]["limiter"] = ("100 chains cannot fill 148 SMs with one warp each: eight teams per chain evaluate different trials of "
                                      "the window and commit in order; a batch lasts as long as its slowest trial and ends at its first "
                                      "accepted one (profiles/r02d_tune_spec.txt)")
        workloads["K1"]["limiter"] = ("one warp per chain, 12 chains per SM (registers and shared memory): 3450 FP64 of 5984 warp instructions per "
                                      "trial, FP64 pipe 53 % busy, dependent-issue latency at 3 warps per scheduler; DESIGN.md section 8")
        for nm in ("C2s", "C5s"):
            r = measure(cx, nm, xs, 3, want_e2e=not args.no_e2e)
            r["limiter"] = ("148 chains per GPU at 8 GPUs are one wave: two SMs per chain and the work-ordered queue keep the FP64 "
                            "pipe busy for 0.97 of what 1184 chains on one GPU reach" if nm == "C5s" else
                            "512 chains per GPU at 8 GPUs quantise badly over 592 CTA slots (80 SMs carry three chains, 68 four): the "
                            "library switches to two SMs per chain for such fills")
            strong[nm[:-1]] = r
        barrier()
        if world > 1:
            torch.cuda.synchronize(cx.dev)
            if rank == 0:
                try:
                    multi_abi = measure_multi_abi(cx, xs, 3)
                except Exception as e:  # the multi-device ABI is reported, never fatal for the headline
                    multi_abi = {"error": str(e)}
            dist.barrier(group=cx.cpu_group)   # the other ranks wait on the host, their GPUs idle
    cx.sampler.stop()

    # ---- CPU baseline (rank 0, N=1 only) -----------------------------------------------------------
    cpu_baseline = None
    kw = WORKLOADS[args.workload]["cases"][0]
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        trials = sized_cpu_sample(kw, threads, args.cpu_baseline_seconds)
        ups, secs = cpu_reference_run(kw, threads, trials, threads, algo=0)
        t1 = max(1, int(trials * 3.0 / max(secs, 1e-9)))        # ≈3 s of the exact-ΔU formulation beside it
        ups1, secs1 = cpu_reference_run(kw, threads, t1, threads, algo=1)
        cpu_baseline = {"value": ups, "unit": UNIT, "cores": threads, "kind": "port", "build": cpu_build_flags(),
                        "sample": f"{threads} chains x {trials} trials (one chain per thread, {secs:.1f} s), same "
                                  f"parameters; oracle algo 0 = the reference's full-recompute algorithm",
                        "delta_u_variant": {"value": ups1, "unit": UNIT,
                                            "sample": f"{threads} chains x {t1} trials ({secs1:.1f} s); oracle algo 1 = the "
                                                      "changed-pair formulation the GPU path uses, written as a checker "
                                                      "(it also accumulates the sum of |terms|), not tuned"}}

    if rank == 0:
        line = {
            "metric": head["metric"], "value": head["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True,
            "scaling": head["scaling"], "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": head["config"], "clocks": head["clocks"], "e2e": head["e2e"], "gpu_launches": head["gpu_launches"],
            "roofline": head["roofline"], "cpu_baseline": cpu_baseline,
            "wall_s_timed_region": head["wall_s_timed_region"],
        }
        if extras:
            line["workloads"] = workloads
            line["strong"] = strong
            if multi_abi is not None:
                line["multi_abi"] = multi_abi
        emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
