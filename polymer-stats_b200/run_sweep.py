#!/usr/bin/env python
"""A whole parameter study in one process (SURVEY.md §8f rank 3): replaces `julia -p N run/<study>.jl` +
`julia scripts/aggregate_mcmc.jl` (+ `scripts/reduce_tabular_data.jl`).

    python polymer-stats_b200/run_sweep.py --driver clustering --out study.csv [--pooled-out pooled.csv] \
        [--outdir outs/] --runs 5 --grid E0=0.1,1,10 --grid Fz=0,0.5,1 --kappaflag -- \
        --energy-type interacting --bend-mod 0.5 -n 100 --num-steps 200000 --burn-in 20000

Everything after `--` is the common command line of the driver (same options as mcmc_eap_chain.jl /
mcmc_clustering_eap_chain.jl); every `--grid NAME=v1,v2,…` multiplies the case list (NAME is the long option
name without dashes).  All chains of the study run concurrently on the GPU (sharded over ranks under torchrun);
the aggregated table is the one aggregate_mcmc.jl would build from the per-case `.out` files, which are only
written when --outdir is given."""
import argparse
import itertools
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from polymc import aggregate, mcmc, mcmc_clustering, mcmc_clustering_2d, sweep  # noqa: E402


def main(argv=None) -> int:
    argv = list(sys.argv[1:] if argv is None else argv)
    common = []
    if "--" in argv:
        k = argv.index("--")
        argv, common = argv[:k], argv[k + 1:]
    ap = argparse.ArgumentParser(prog="run_sweep")
    ap.add_argument("--driver", choices=["plain", "clustering", "clustering2d"], default="plain",
                    help="mcmc_eap_chain.jl, mcmc_clustering_eap_chain.jl or 2D/mcmc_clustering_eap_chain.jl")
    ap.add_argument("--grid", action="append", default=[], help="NAME=v1,v2,... (long option name of the driver)")
    ap.add_argument("--runs", type=int, default=1, help="independent runs per case (the launchers' run-NNN)")
    ap.add_argument("--out", required=True, help="aggregated CSV (aggregate_mcmc.jl format)")
    ap.add_argument("--pooled-out", default=None, help="pooled CSV (reduce_tabular_data.jl format)")
    ap.add_argument("--outdir", default=None, help="also write the per-case <prefix>.out files here")
    ap.add_argument("--by", default=None, metavar="PARAM",
                    help="also write one CSV per combination of the OTHER parameters (the sweep over PARAM; FxFz for "
                         "both force components), as scripts/aggregate_by.jl does, into --by-outdir")
    ap.add_argument("--by-outdir", default=None)
    ap.add_argument("--kappaflag", action="store_true", help="file names / table carry the kappa column")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--bit-identical", action="store_true",
                    help="choose the launch shapes from the whole study instead of this rank's share: results are then the same "
                         "bit for bit for any number of GPUs (a share runs up to ~15 %% slower than in its own shape)")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--temper", choices=["kT", "Fz", "Fx"], default=None,
                    help="replica exchange (parallel tempering): cases that differ only in this option form one ladder, "
                         "and neighbouring rungs swap configurations every --exchange-every trials")
    ap.add_argument("--exchange-every", type=int, default=100, help="trials between two exchange rounds")
    ap.add_argument("--exchange-out", default=None,
                    help="CSV of the exchange statistics: one row per adjacent rung pair (needs --temper)")
    a = ap.parse_args(argv)
    if a.exchange_out and not a.temper:
        ap.error("--exchange-out needs --temper")
    host = {"plain": mcmc, "clustering": mcmc_clustering, "clustering2d": mcmc_clustering_2d}[a.driver]
    axes = []
    for g in a.grid:
        name, vals = g.split("=", 1)
        axes.append((name, vals.split(",")))
    pargs_list = []
    for combo in itertools.product(*[v for _, v in axes]):
        extra = []
        for (name, _), v in zip(axes, combo):
            extra += [f"--{name}", v]
        pargs_list.append(host.parse_args(common + extra))
    # under torchrun: one rank per GPU, chains sharded by global chain id, one all_gather of the results (NCCL)
    rank, world, torch_device = 0, int(os.environ.get("WORLD_SIZE", "1")), None
    if a.temper and world > 1:
        ap.error("--temper needs a single rank: a ladder must live in one handle (run without torchrun)")
    if world > 1:
        import torch
        import torch.distributed as dist
        a.device = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(a.device)
        torch_device = torch.device("cuda", a.device)
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch_device)
        rank = dist.get_rank()
    if a.by and not a.by_outdir:
        ap.error("--by needs --by-outdir")
    exchange = {}
    header, rows, texts, entries = sweep.sweep_table(pargs_list, driver=a.driver, runs=a.runs, seed=a.seed,
                                                     device=a.device, torch_device=torch_device,
                                                     kappaflag=a.kappaflag, with_entries=True, bit_identical=a.bit_identical,
                                                     temper=a.temper, exchange_every=a.exchange_every, exchange=exchange)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()
    if rank != 0:
        return 0
    aggregate.write_table(a.out, header, rows)
    if a.pooled_out:
        ct = pargs_list[0]["chain-type"]
        h2, r2 = aggregate.reduce_table(header, rows, len(aggregate.input_headers(ct, a.kappaflag)))
        aggregate.write_table(a.pooled_out, h2, r2)
    if a.outdir:
        aggregate.write_out_files(a.outdir, texts)
    if a.exchange_out:
        fixed = [name for name, _ in axes if name != a.temper]
        sweep.write_exchange_csv(a.exchange_out, *sweep.exchange_rows(pargs_list, a.temper, exchange, fixed))
    if a.by:
        os.makedirs(a.by_outdir, exist_ok=True)
        ct = pargs_list[0]["chain-type"]
        for name, (h, r) in aggregate.aggregate_by(entries, a.by, ct, a.kappaflag, runflag=a.runs > 1,
                                                         dims=2 if a.driver == "clustering2d" else 3).items():
            aggregate.write_table(os.path.join(a.by_outdir, name), h, r)
    print(f"{len(pargs_list)} cases x {a.runs} runs -> {a.out}", file=sys.stderr)
    return 0


if __name__ == "__main__":
    sys.exit(main())
