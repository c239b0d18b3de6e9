"""Generates run_plan.json: which run kernel, block size and pair precision the library chooses for each handle of a grid
that crosses every threshold of the launch planner on both sides (chain length, ensemble size, precision, energy type,
driver, accumulator mode and the environment overrides).  Each entry is observed through the Python API only:
kernel_name(), block_threads() and pair_precision(), or the error code of the create.  The choices depend on the SM
count, so the file is recorded on a B200 (148 SMs); tests/test_gpu_run_plan.py replays the grid.

    PMC_LIB_PATH=<library> python tests/golden/make_run_plan.py [OUT]
"""
import json
import os
import sys

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "run_plan.json")
REPLICAS = 2

PLAIN_N = [2, 16, 64, 65, 100, 110, 111, 128, 129, 384, 385, 512, 768, 769, 1024, 1025, 1536, 1537, 2048, 3800, 4096]
PLAIN_HINTS = [0, 100, 148, 300, 326, 444, 533, 600, 888, 1184, 4096, 65536]
CLUSTER_N = [2, 16, 40, 41, 64, 100, 110, 111, 150, 160, 161, 256, 257, 400, 640, 800, 1000, 1500, 1600]
CLUSTER_HINTS = [0, 25, 100, 148, 200, 444, 500, 740, 1000, 4096]
PLANAR_N = [16, 100, 161, 400]
LANE_HINTS = [0, 2368, 2369, 65535, 65536, 119999, 120000]
LANE_CLUSTER_N = [16, 1024, 1025]
LANE_CLUSTER_HINTS = [0, 10999, 11000, 32767, 32768]


def grid():
    """Handles: (case keywords, ensemble hint (0: its own size), environment at create, queries).  A query is
    (pair precision, environment at the query)."""
    unset = None
    for n in PLAIN_N:
        for spec in ([unset, "0"] if n <= 110 else [unset]):
            for hint in PLAIN_HINTS:
                yield (dict(n=n, energy_type="interacting"), hint, {"PMC_RUN_SPEC": spec},
                       [(prec, {"PMC_RUN_PAIR": pair}) for prec in ("fp64", "fp32") for pair in (unset, "0", "2")])
    for et, extra, ns in (("interacting", dict(clustering=True), CLUSTER_N),
                          ("cutoff", dict(), CLUSTER_N),
                          ("interacting", dict(clustering=True, planar=True), PLANAR_N)):
        for n in ns:
            for spec in (unset, "0"):
                for hint in CLUSTER_HINTS:
                    yield (dict(n=n, energy_type=et, **extra), hint, {"PMC_CLUSTER_SPEC": spec},
                           [("fp64", {"PMC_CLUSTER_SPEC": spec})])
    for et in ("noninteracting", "Ising"):
        for n in (16, 100):
            for accum in (0, 1):
                for hint in LANE_HINTS:
                    yield (dict(n=n, energy_type=et, accum_mode=accum), hint, {},
                           [("fp64", {"PMC_LANE_MODE": mode}) for mode in (unset, "1", "2")])
        for n in LANE_CLUSTER_N:
            for accum in (0, 1):
                for hint in LANE_CLUSTER_HINTS:
                    yield (dict(n=n, energy_type=et, accum_mode=accum, clustering=True), hint, {},
                           [("fp64", {"PMC_LANE_CLUSTER_MODE": mode}) for mode in (unset, "1", "2")])


def set_env(env):
    for k, v in env.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = v


def observe(pm, case_kw, hint, create_env, queries):
    """What the library chooses for one handle of the grid: a dict that run_plan.json stores for it."""
    set_env(create_env)
    try:
        try:
            ens = pm.Ensemble(pm.make_case(**case_kw), replicas=REPLICAS, ensemble_chains=hint)
        except pm.PolymcError as e:
            return {"create": e.code}
        out = []
        with ens:
            for prec, env in queries:
                set_env(env)
                try:
                    ens.set_pair_precision(prec)
                    out.append([ens.kernel_name(), ens.block_threads(), ens.pair_precision()])
                except pm.PolymcError as e:
                    out.append([e.code])
                finally:
                    set_env({k: None for k in env})
        return {"create": 0, "queries": out}
    finally:
        set_env({k: None for k in create_env})


def record(pm):
    """One entry per handle of grid(); "seen" holds [kernel_name, block_threads, pair_precision] (or [error code]) per
    query of the handle, in grid order."""
    return [{"case": case_kw, "hint": hint, "create_env": create_env,
             "seen": observe(pm, case_kw, hint, create_env, queries)}
            for case_kw, hint, create_env, queries in grid()]


if __name__ == "__main__":
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))),
                                    "polymer-stats_b200"))
    import polymc as pm
    entries = record(pm)
    with open(sys.argv[1] if len(sys.argv) > 1 else OUT, "w") as f:
        json.dump(entries, f, indent=None, separators=(",", ":"))
        f.write("\n")
    print(len(entries), "handles,", sum(len(e["seen"].get("queries", [])) for e in entries), "queries")
