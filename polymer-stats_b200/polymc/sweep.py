"""Sweeps across GPUs (north_star "Sweeps across GPUs"; SURVEY.md §8e).

The reference fans cases out with `pmap`, one fresh `julia` process per case
(run/interacting_dielectric_study.jl:37-47), and "gathers" through files on a shared filesystem.
Here the chains of a sweep (cases × replicas) are independent units: each rank (one process per
GPU, torch.distributed) takes a contiguous block of global chain ids, runs it with no data-path
collective, and only the final per-chain averages are gathered (NCCL all_gather over NVLink).
Philox streams are keyed by the GLOBAL chain id, so the result does not depend on the GPU count.
"""
from __future__ import annotations

from collections import OrderedDict

import numpy as np

from . import lib


def shard_range(total: int, rank: int, world: int):
    """Contiguous block [lo, hi) of `total` units owned by `rank` (SURVEY §8e partitioning)."""
    if world < 1 or not (0 <= rank < world):
        raise ValueError("bad rank/world")
    lo = total * rank // world
    hi = total * (rank + 1) // world
    return lo, hi


def bucket_cases(cases):
    """Group case indices by (n, energy_type): one handle/kernel per bucket (include/polymc.h)."""
    buckets = OrderedDict()
    if isinstance(cases, lib.CaseTable):   # vectorised: a phase-diagram grid has tens of thousands of cases
        ns, es = cases.column("n"), cases.column("energy_type")
        key = ns.astype(np.int64) * 8 + es.astype(np.int64)
        uniq, first = np.unique(key, return_index=True)
        for k in uniq[np.argsort(first)].tolist():   # buckets in order of first appearance, like the loop below
            buckets[(int(k // 8), int(k % 8))] = np.flatnonzero(key == k)
        return buckets
    for i, c in enumerate(cases):
        buckets.setdefault((int(c.n), int(c.energy_type)), []).append(i)
    return buckets


TEMPER_FIELDS = ("kT", "Fz", "Fx")


def tempering_ladders(cases, temper: str):
    """Replica-exchange ladders of a sweep: cases that agree on every field except `temper` ("kT", "Fz" or "Fx")
    form one ladder, ordered by increasing `temper`.  -> list of lists of case indices.  Refuses umbrella sampling
    (its weights depend on kT and F), a ladder of one rung and two rungs with the same value."""
    if temper not in TEMPER_FIELDS:
        raise lib.PolymcError(-1, f"temper must be one of {', '.join(TEMPER_FIELDS)} (got {temper!r})")
    rec = cases.rec if isinstance(cases, lib.CaseTable) else lib.CaseTable(cases).rec
    if np.any(rec["umbrella"] != 0):
        raise lib.PolymcError(-1, "umbrella sampling cannot be tempered: its weights depend on kT and F")
    rest = rec.copy()
    rest[temper] = 0.0           # every other field, byte for byte, is the key of the ladder
    groups = OrderedDict()
    for i in range(rest.shape[0]):
        groups.setdefault(rest[i].tobytes(), []).append(i)
    ladders = []
    for idx in groups.values():
        vals = rec[temper][idx]
        if len(idx) < 2:
            raise lib.PolymcError(-1, f"case {idx[0]} has no partner that differs only in {temper}: a ladder needs at "
                                      "least two rungs")
        if len(np.unique(vals)) != len(vals):
            raise lib.PolymcError(-1, f"cases {idx} repeat a value of {temper}: every rung of a ladder needs its own")
        ladders.append([idx[k] for k in np.argsort(vals, kind="stable")])
    return ladders


def _dist():
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            return dist
    except Exception:
        pass
    return None


def gather_rows(local: np.ndarray, total_rows: int, lo: int, device=None) -> np.ndarray:
    """Assemble [total_rows][k] from each rank's [hi-lo][k] block.  One all_gather of equal-sized
    padded blocks (NCCL when the process group is NCCL, gloo on CPU); identity without a group."""
    dist = _dist()
    local = np.ascontiguousarray(local, dtype=np.float64)
    if dist is None or dist.get_world_size() == 1:
        assert local.shape[0] == total_rows
        return local
    import torch
    world = dist.get_world_size()
    k = local.shape[1]
    maxrows = max(shard_range(total_rows, r, world)[1] - shard_range(total_rows, r, world)[0] for r in range(world))
    pad = np.zeros((maxrows, k))
    pad[: local.shape[0]] = local
    t = torch.from_numpy(pad)
    if device is not None:
        t = t.to(device)
    out = torch.empty((world * maxrows, k), dtype=t.dtype, device=t.device)
    dist.all_gather_into_tensor(out, t)        # one collective (concatenated form: NCCL and gloo), one copy back
    out = out.cpu().numpy()
    if total_rows == world * maxrows:          # equal shards: the gathered buffer is the result
        return out
    out = out.reshape(world, maxrows, k)
    full = np.empty((total_rows, k))
    for r in range(world):
        a, b = shard_range(total_rows, r, world)
        full[a:b] = out[r, : b - a]
    return full


NCOL = 37  # 16 averages, acceptance rate, normaliser, 17 raw sums, 2 raw sums of the clustering driver's extras


def _segments(mine: np.ndarray, replicas: int):
    """Split a rank's sorted global chain ids into runs that one handle can serve: a handle holds
    `ncases` consecutive cases × `replicas` chains with ids chain_id_base + local index
    (include/polymc.h), or a part of a single case.  Yields (pos, end, first_case, ncases, nrep)."""
    m = len(mine)
    if m == 0:
        return
    mine = np.asarray(mine, dtype=np.int64)
    # maximal runs of consecutive ids (vectorised: a phase-diagram sweep has tens of thousands of chains)
    breaks = np.flatnonzero(np.diff(mine) != 1) + 1
    starts = np.concatenate([[0], breaks])
    ends = np.concatenate([breaks, [m]])
    for pos, run_end in zip(starts.tolist(), ends.tolist()):
        while pos < run_end:
            g0 = int(mine[pos])
            case0, off = divmod(g0, replicas)
            run = run_end - pos
            if off != 0 or run < replicas:          # a partial case at a shard boundary
                take = min(run, replicas - off)
                yield pos, pos + take, case0, 1, take
                pos += take
            else:                                   # whole consecutive cases in one handle
                ncases = run // replicas
                yield pos, pos + ncases * replicas, case0, ncases, replicas
                pos += ncases * replicas


def _local_ladders(ladders, case0: int, ncases: int):
    """The ladders of a handle holding cases [case0, case0 + ncases), as its own case indices."""
    local = []
    for lad in ladders:
        inside = [case0 <= c < case0 + ncases for c in lad]
        if any(inside) and not all(inside):
            raise lib.PolymcError(-1, f"the ladder of cases {lad} spans two handles (cases of different num-monomers "
                                      "or energy-type interleave): list the tempered option's grid last")
        if all(inside):
            local.append([c - case0 for c in lad])
    return local


def _collect_exchange(exchange, st, ladders, case0: int, ncases: int, nrep: int):
    exchange["attempts"][case0:case0 + ncases] += st["attempts"]
    exchange["accepts"][case0:case0 + ncases] += st["accepts"]
    for k, lad in enumerate(ladders):
        if case0 <= lad[0] < case0 + ncases:    # walkers by their starting case: label − chain_id_base = chain index
            walkers = np.concatenate([np.arange((c - case0) * nrep, (c - case0 + 1) * nrep) for c in lad])
            exchange["round_trips"][k] += int(st["round_trips"][walkers].sum())


def run_shard(cases, replicas: int, nsteps: int, stepout: int = 0, seed: int = 0, device: int = 0,
              rank: int = 0, world: int = 1, protocol=None, bit_identical: bool = False, pair_precision: str = "fp64",
              temper=None, exchange_every: int = 100, exchange=None):
    """Run this rank's contiguous block of every (n, energy) bucket.  Returns a list of
    (global chain ids of the bucket, lo, block [hi-lo][NCOL]).  No communication.

    protocol None: `nsteps` trials of mcmc_eap_chain.jl's loop.  protocol = dict(burn_in=…, schedule=[…]):
    the clustering driver's ladder (mcmc_clustering_eap_chain.jl:365-386) — a burn-in stage per kT
    multiplier, then `nsteps` production trials at kT.

    temper "kT" / "Fz" / "Fx": replica exchange every `exchange_every` trials along the ladders of
    tempering_ladders() in every run of the protocol (each init, each burn-in stage).  A ladder lives in one
    handle, so this needs a single rank.  `exchange`, a dict, receives the ladders, the per-case attempts and
    accepts with the next rung and the round trips of every ladder."""
    if not isinstance(cases, lib.CaseTable):
        cases = list(cases)
    ladders = None
    if temper is not None:
        if world > 1:
            raise lib.PolymcError(-1, "replica exchange needs a single rank: a ladder must live in one handle")
        exchange_every = int(exchange_every)
        lengths = [nsteps] + ([int(protocol.get("burn_in", 0))] if protocol and not protocol.get("plain") else [])
        if exchange_every < 1 or any(k % exchange_every for k in lengths):
            raise lib.PolymcError(-1, f"--exchange-every ({exchange_every}) must divide --num-steps and --burn-in")
        ladders = tempering_ladders(cases, temper)
        if exchange is not None:
            exchange.update(ladders=ladders, attempts=np.zeros(len(cases), np.int64),
                            accepts=np.zeros(len(cases), np.int64), round_trips=np.zeros(len(ladders), np.int64))
    out = []
    for (_, _), idxs in bucket_cases(cases).items():
        # global chain ids of this bucket, case-major
        gids = (np.asarray(idxs, dtype=np.int64)[:, None] * replicas + np.arange(replicas, dtype=np.int64)).ravel()
        lo, hi = shard_range(len(gids), rank, world)
        mine = gids[lo:hi]
        block = np.zeros((hi - lo, NCOL))
        for pos, end, case0, ncases, nrep in _segments(mine, replicas):
            # The Markov chains (Philox streams keyed by global chain id) never depend on the sharding.  The launch shape —
            # block size, packing, one or two SMs per chain — is chosen for THIS shard's size (fastest: a 512-chain
            # share of a 4096-chain sweep runs 15 % faster in its own shape, profiles/r02b_tune_pair_small.txt), which
            # changes the order of some floating-point sums; bit_identical=True chooses it from the UNSHARDED bucket
            # size instead, and the results are then the same bit for bit for any rank count.
            with lib.Ensemble(cases[case0:case0 + ncases], replicas=nrep, seed=seed, device=device,
                              chain_id_base=int(mine[pos]), ensemble_chains=len(gids) if bit_identical else 0) as ens:
                if pair_precision != "fp64":   # opt-in FP32 rectangle where a kernel serves it (include/polymc.h)
                    ens.set_pair_precision(pair_precision)
                local = None
                if ladders is not None:
                    local = _local_ladders(ladders, case0, ncases)
                    ens.set_ladders(local)
                run, run_ex = ens.run, ens.run_ex
                if local:
                    def run(k, so, fetch_rows):
                        return ens.run_tempering(k, exchange_every, so, fetch_rows=fetch_rows)

                    def run_ex(k, so, fetch_rows):
                        return ens.run_tempering_ex(k, exchange_every, so, fetch_rows=fetch_rows)
                if protocol is None or protocol.get("plain"):
                    # mcmc_eap_chain.jl:276-361: num-inits passes of nsteps trials with the re-initialisation rule between
                    inits = int(protocol.get("num_inits", 1)) if protocol else 1
                    for init in range(inits):
                        run(nsteps, stepout, fetch_rows=False)
                        if init + 1 < inits:
                            ens.reinit()
                else:
                    if protocol.get("x0") is not None:      # inc/eap_chain.jl:63-78
                        ens.init_x0(protocol["x0"], protocol["dx0"])
                    for mult in protocol.get("schedule", []):
                        ens.begin_stage(float(mult))
                        run_ex(int(protocol.get("burn_in", 0)), 0, fetch_rows=False)
                    ens.begin_stage(1.0)
                    run_ex(nsteps, 0, fetch_rows=False)
                    block[pos:end, 35:37] = ens.extra_accumulators()
                if local and exchange is not None:
                    _collect_exchange(exchange, ens.exchange_stats(), ladders, case0, ncases, nrep)
                avg, ar, nrm = ens.averages()
                block[pos:end, :16] = avg
                block[pos:end, 16] = ar
                block[pos:end, 17] = nrm
                block[pos:end, 18:35] = ens.accumulators()
        out.append((gids, lo, block))
    return out


def assemble(total: int, parts):
    """dict of result arrays from [(gids, full [len(gids)][NCOL]), ...]."""
    if len(parts) == 1 and len(parts[0][0]) == total:
        gids, full = parts[0]
        if total == 0 or (gids[0] == 0 and gids[-1] == total - 1 and np.all(np.diff(gids) == 1)):
            # one bucket holding every chain in order (the usual sweep): columns of the gathered block, no scatter
            return {"avg": full[:, :16], "acc_rate": full[:, 16], "normalizer": full[:, 17], "sums": full[:, 18:35],
                    "extra_sums": full[:, 35:37]}
    res = {"avg": np.full((total, 16), np.nan), "acc_rate": np.full(total, np.nan),
           "normalizer": np.full(total, np.nan), "sums": np.full((total, 17), np.nan),
           "extra_sums": np.full((total, 2), np.nan)}
    for gids, full in parts:
        res["avg"][gids] = full[:, :16]
        res["acc_rate"][gids] = full[:, 16]
        res["normalizer"][gids] = full[:, 17]
        res["sums"][gids] = full[:, 18:35]
        res["extra_sums"][gids] = full[:, 35:37]
    return res


def run_sweep(cases, replicas: int, nsteps: int, stepout: int = 0, seed: int = 0, device: int = 0,
              torch_device=None, protocol=None, bit_identical: bool = False, pair_precision: str = "fp64",
              temper=None, exchange_every: int = 100):
    """Run every (case, replica) chain of a sweep for nsteps trials, sharded over the ranks of the
    current torch.distributed group (or a single process), then gather the final per-chain results on
    every rank.  Chain order = case-major: avg [ncases*replicas][16], acc_rate, normalizer, sums [..][17].
    With temper (run_shard), "exchange" holds the ladders and their exchange statistics."""
    dist = _dist()
    rank = dist.get_rank() if dist else 0
    world = dist.get_world_size() if dist else 1
    if not isinstance(cases, lib.CaseTable):
        cases = list(cases)
    parts, exchange = [], {}
    for gids, lo, block in run_shard(cases, replicas, nsteps, stepout, seed, device, rank, world, protocol, bit_identical,
                                     pair_precision, temper, exchange_every, exchange):
        parts.append((gids, gather_rows(block, len(gids), lo, device=torch_device)))
    res = assemble(len(cases) * replicas, parts)
    if temper is not None:
        res["exchange"] = exchange
    return res


def sweep_table(pargs_list, driver: str = "plain", runs: int = 1, seed: int = 0, device: int = 0, torch_device=None,
                kappaflag: bool = False, pooled: bool = False, with_entries: bool = False, bit_identical: bool = False,
                temper=None, exchange_every: int = 100, exchange=None):
    """A whole launcher + aggregate_mcmc.jl (+ reduce_tabular_data.jl) pipeline in one call (SURVEY §8f
    rank 3): every pargs dict of `pargs_list` is one case (one launcher command line), run `runs` times as
    independent replica chains (the launchers' `run-NNN` cases); the result is the aggregated table the
    reference's scripts would build from the `.out` files.  Returns (header, rows, entries) with entries =
    [(prefix, stdout text)] for optional `.out` emission.  temper / exchange_every: replica exchange along the
    ladders of the sweep (run_shard); the table keeps its format, a row per case being a row per rung.  `exchange`,
    a dict, receives the ladders and their statistics (see exchange_rows)."""
    from . import aggregate as agg
    from . import mcmc as plain_host
    from . import mcmc_clustering as cl_host
    from . import mcmc_clustering_2d as cl2d_host
    if not pargs_list:
        raise lib.PolymcError(-1, "empty sweep")
    if driver not in ("plain", "clustering", "clustering2d"):
        raise lib.PolymcError(-1, "driver must be plain, clustering or clustering2d")
    planar = driver == "clustering2d"   # the 2-D tree: 2D/mcmc_clustering_eap_chain.jl, aggregate_mcmc.jl … 2D
    host = cl2d_host if planar else cl_host if driver == "clustering" else plain_host
    chain_type = pargs_list[0]["chain-type"]
    for p in pargs_list:
        host.validate({**p, "replicas": 1})
        if p["chain-type"] != chain_type:
            raise lib.PolymcError(-1, "one aggregated table holds one chain type (aggregate_mcmc.jl:40-47)")
    cases = [host.case_from_pargs(p) for p in pargs_list]
    p0 = pargs_list[0]
    # Options that shape the PROTOCOL of a run (not the physics of a case) apply to the whole ensemble of one call:
    # they must agree across the sweep, otherwise a row would claim a command line that was not run.
    proto_keys = ["num-steps"] + (["num-inits", "force-init"] if driver == "plain" else ["burn-in", "burn-schedule"]) + \
        ([] if driver != "clustering" else ["x0", "dx0"])
    for p in pargs_list:
        for k in proto_keys:
            if p.get(k) != p0.get(k):
                raise lib.PolymcError(-1, f"--{k} must be the same for every case of one sweep ({p.get(k)!r} vs "
                                          f"{p0.get(k)!r}): run one sweep per value")
    if driver == "plain":
        protocol = dict(plain=True, num_inits=int(p0.get("num-inits", 1)))
    else:
        protocol = dict(burn_in=p0["burn-in"], schedule=cl_host.parse_julia_vector(p0["burn-schedule"], "burn-schedule"))
        if driver == "clustering" and p0.get("x0") is not None:
            x0 = cl_host.parse_julia_vector(p0["x0"], "x0")
            dx0 = cl_host.parse_julia_vector(p0["dx0"], "dx0")
            if len(x0) != 2 or len(dx0) < 2:   # a per-monomer x0 belongs to one chain length, i.e. one case
                raise lib.PolymcError(-1, f"a sweep takes --x0 as [phi, theta] (Invalid input for 'x0', {p0['x0']})")
            protocol.update(x0=x0, dx0=dx0[:2])
    # two cases with the same file-name prefix would overwrite each other's .out file and be indistinguishable rows
    seen = {}
    for i, p in enumerate(pargs_list):
        pre = agg.prefix_of(p, chain_type, kappaflag, run=None)
        if pre in seen:
            raise lib.PolymcError(-1, f"cases {seen[pre]} and {i} share the output prefix '{pre}': the swept option is not "
                                      "part of the file-name tokens (aggregate_mcmc.jl:40-57; use --kappaflag for bend-mod)")
        seen[pre] = i
    res = run_sweep(cases, runs, p0["num-steps"], 0, seed, device, torch_device, protocol, bit_identical,
                    p0.get("pair-precision", "fp64"), temper, exchange_every)
    if exchange is not None and temper is not None:
        exchange.update(res["exchange"])
    runflag = runs > 1
    entries, texts = [], []
    for i, p in enumerate(pargs_list):
        for r in range(runs):
            g = i * runs + r
            prefix = agg.prefix_of(p, chain_type, kappaflag, run=(r + 1) if runflag else None)
            avg = res["avg"][g]
            if planar:
                entries.append((prefix, agg.output_values_2d(avg, res["acc_rate"][g], p["mlen"], p["num-monomers"])))
                texts.append((prefix, agg.out_text_2d(avg, res["acc_rate"][g], p["mlen"], p["num-monomers"])))
                continue
            ex = (res["extra_sums"][g] / res["normalizer"][g]) if driver == "clustering" else None
            entries.append((prefix, agg.output_values(avg, res["acc_rate"][g], p["mlen"], p["num-monomers"], ex)))
            texts.append((prefix, agg.out_text(avg, res["acc_rate"][g], p["mlen"], p["num-monomers"], ex)))
    header, rows = agg.aggregate_table(entries, chain_type, kappaflag, runflag, dims=2 if planar else 3)
    if pooled:
        header, rows = agg.reduce_table(header, rows, len(agg.input_headers(chain_type, kappaflag)))
    if with_entries:  # [(prefix, output values)]: the input of agg.aggregate_by (scripts/aggregate_by.jl)
        return header, rows, texts, entries
    return header, rows, texts


def exchange_rows(pargs_list, temper: str, exchange: dict, fixed=()):
    """The replica-exchange table of a tempered sweep: one row per adjacent rung pair with the ladder's `fixed` options
    (e.g. the other grid axes), the two rung values, attempts, accepts, acceptance rate and the ladder's round trips
    (bottom → top → bottom, summed over its walkers).  -> (header, rows)."""
    header = list(fixed) + [f"{temper}_lo", f"{temper}_hi", "attempts", "accepts", "rate", "round_trips"]
    rows = []
    for k, lad in enumerate(exchange["ladders"]):
        p = pargs_list[lad[0]]
        for lo, hi in zip(lad[:-1], lad[1:]):
            att, acc = int(exchange["attempts"][lo]), int(exchange["accepts"][lo])
            rows.append([p[f] for f in fixed] + [pargs_list[lo][temper], pargs_list[hi][temper], att, acc,
                                                 acc / att if att else float("nan"), int(exchange["round_trips"][k])])
    return header, rows


def write_exchange_csv(path: str, header, rows):
    """exchange_rows() as CSV: counts as integers, other numbers as Julia prints Float64, anything else as text."""
    from .output import julia_float

    def cell(x):
        if isinstance(x, (bool, str)):
            return str(x)
        if isinstance(x, (int, np.integer)):
            return str(int(x))
        return julia_float(x)
    with open(path, "w") as f:
        f.write(",".join(header) + "\n")
        for row in rows:
            f.write(",".join(cell(x) for x in row) + "\n")
