"""north_star: "It keeps … the output.jl tabular format, so run/* sweep scripts and scripts/aggregate_mcmc.jl work
unchanged."  Checked literally: the UNMODIFIED reference script scripts/aggregate_mcmc.jl, executed by tools/minijl, reads
`<prefix>.out` files written by this package (the stdout block of the CLI twins under the launchers' file names) and must
produce the table polymc.aggregate produces directly — byte for byte.

The files the reference scripts wrote for these inputs are stored in tests/golden/ref/script_tables.json, so the
comparison runs on any machine.  With POLYMC_REFERENCE_DIR set to a checkout of the reference, the scripts are also run
now and must write the same files.  CPU only."""
import io
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "polymer-stats_b200"))
REF = os.environ.get("POLYMC_REFERENCE_DIR")
SCRIPT = os.path.join(REF, "scripts", "aggregate_mcmc.jl") if REF else None
with open(os.path.join(ROOT, "tests", "golden", "ref", "script_tables.json")) as _f:
    STORED = json.load(_f)["tables"]


def assert_reference_agrees(key, ours, run_reference):
    """ours: {file name: text} as polymc.aggregate writes it.  The reference script wrote STORED[key] for the same
    inputs; with the reference tree at hand, run_reference() runs it now and returns its files."""
    if REF:
        assert run_reference() == ours
    assert STORED[key] == ours


def run_reference_aggregate(argv):
    from minijl.interp import Interp
    it = Interp(argv=list(argv))
    out = io.StringIO()
    it.stdout = out
    it.genv.vars["stdout"] = out
    it.run_main(SCRIPT)
    return out.getvalue()


def cases(rng, chain_type, count):
    out = []
    for k in range(count):
        p = {"E0": float(rng.choice([0.0, 0.5, 1.25, 2.0])) + 0.001 * k, "K1": 1.0, "K2": float(rng.choice([0.0, 0.25])), "mu": 0.5,
             "kT": float(rng.choice([0.5, 1.0])), "Fz": 0.25 * k, "Fx": 0.0, "num-monomers": int(rng.choice([50, 100])), "mlen": 1.0,
             "bend-mod": float(rng.choice([0.0, 0.5]))}
        out.append((p, rng.normal(size=16) * 10.0 ** rng.integers(-3, 4), rng.normal(size=2), float(rng.uniform(0.01, 0.6))))
    return out


@pytest.mark.parametrize("chain_type,kappaflag,runflag", [("dielectric", True, False), ("polar", False, True), ("dielectric", False, False)])
def test_reference_aggregate_script_reads_our_out_files(tmp_path, chain_type, kappaflag, runflag):
    from polymc import aggregate as ag
    rng = np.random.default_rng(7)
    text, entries = [], []
    for k, (p, avg, ex, ar) in enumerate(cases(rng, chain_type, 5)):
        prefix = ag.prefix_of(p, chain_type, kappaflag, run=k + 1 if runflag else None)
        text.append((prefix, ag.out_text(avg, ar, p["mlen"], p["num-monomers"], ex)))          # the clustering driver's 12 lines
        entries.append((prefix, ag.output_values(avg, ar, p["mlen"], p["num-monomers"], ex)))
    outdir = tmp_path / "study"
    ag.write_out_files(str(outdir), text)
    ours = tmp_path / "ours.csv"
    ag.write_table(str(ours), *ag.aggregate_table(entries, chain_type, kappaflag, runflag, 3))
    theirs = tmp_path / "theirs.csv"
    argv = [str(theirs), str(outdir), "*.out", chain_type, "3D", "true" if kappaflag else "false"] + (["true"] if runflag else [])

    def run_reference():
        log = run_reference_aggregate(argv)
        assert log.count("processing") == 5
        return {"table.csv": theirs.read_text()}
    assert_reference_agrees(f"aggregate_mcmc/{chain_type}-{kappaflag}-{runflag}", {"table.csv": ours.read_text()},
                            run_reference)


def test_reference_aggregate_script_reads_our_2d_out_files(tmp_path):
    from polymc import aggregate as ag
    rng = np.random.default_rng(8)
    text, entries = [], []
    for p, avg, ex, ar in cases(rng, "dielectric", 4):
        prefix = ag.prefix_of(p, "dielectric", False)
        text.append((prefix, ag.out_text_2d(avg, ar, p["mlen"], p["num-monomers"])))
        entries.append((prefix, ag.output_values_2d(avg, ar, p["mlen"], p["num-monomers"])))
    outdir = tmp_path / "study2d"
    ag.write_out_files(str(outdir), text)
    ours, theirs = tmp_path / "ours.csv", tmp_path / "theirs.csv"
    ag.write_table(str(ours), *ag.aggregate_table(entries, "dielectric", False, False, 2))

    def run_reference():
        run_reference_aggregate([str(theirs), str(outdir), "*.out", "dielectric", "2D"])
        return {"table.csv": theirs.read_text()}
    assert_reference_agrees("aggregate_mcmc/2D", {"table.csv": ours.read_text()}, run_reference)


def test_reference_aggregate_script_on_the_plain_drivers_ten_lines(tmp_path):
    """mcmc_eap_chain.jl prints 10 lines (no Ealign / psi): the script then writes 20 output columns under its 22 headers —
    upstream behaviour, reproduced by both sides."""
    from polymc import aggregate as ag
    rng = np.random.default_rng(9)
    text, entries = [], []
    for p, avg, ex, ar in cases(rng, "dielectric", 3):
        prefix = ag.prefix_of(p, "dielectric", False)
        text.append((prefix, ag.out_text(avg, ar, p["mlen"], p["num-monomers"])))
        entries.append((prefix, ag.output_values(avg, ar, p["mlen"], p["num-monomers"])))
    outdir = tmp_path / "plain"
    ag.write_out_files(str(outdir), text)
    ours, theirs = tmp_path / "ours.csv", tmp_path / "theirs.csv"
    ag.write_table(str(ours), *ag.aggregate_table(entries, "dielectric", False, False, 3))

    def run_reference():
        run_reference_aggregate([str(theirs), str(outdir), "*.out", "dielectric"])
        return {"table.csv": theirs.read_text()}
    assert_reference_agrees("aggregate_mcmc/ten_lines", {"table.csv": ours.read_text()}, run_reference)


@pytest.mark.parametrize("chain_type,kappaflag", [("dielectric", False), ("dielectric", True), ("polar", False)])
def test_reference_reduce_script_on_our_tables(tmp_path, chain_type, kappaflag):
    """scripts/reduce_tabular_data.jl (unmodified, run by minijl) pools the repeated runs of a table written by
    polymc.aggregate; polymc.aggregate.reduce_table — what run_sweep.py --pooled-out writes — gives the same file."""
    from minijl.interp import Interp
    from polymc import aggregate as ag
    rng = np.random.default_rng(11)
    entries = []
    for k, (p, _, _, _) in enumerate(cases(rng, chain_type, 4)):
        for run in range(1, 4 + (k % 2)):                       # 3 or 4 runs per case
            avg, ex, ar = rng.normal(size=16), rng.normal(size=2), float(rng.uniform(0.01, 0.6))
            entries.append((ag.prefix_of(p, chain_type, kappaflag, run=run), ag.output_values(avg, ar, p["mlen"], p["num-monomers"], ex)))
    header, rows = ag.aggregate_table(entries, chain_type, kappaflag, True, 3)
    indir, outdir = tmp_path / "tables", tmp_path / "reduced"
    indir.mkdir()
    ag.write_table(str(indir / "study.csv"), header, rows)
    nparams = len(ag.input_headers(chain_type, kappaflag))
    ours = tmp_path / "ours.csv"
    ag.write_table(str(ours), *ag.reduce_table(header, rows, nparams))

    def run_reference():
        it = Interp(argv=[str(indir), str(outdir), chain_type] + (["true"] if kappaflag else []))
        sink = io.StringIO()
        it.stdout = sink
        it.genv.vars["stdout"] = sink
        it.run_main(os.path.join(REF, "scripts", "reduce_tabular_data.jl"))
        return {"study.csv": (outdir / "study.csv").read_text()}
    assert_reference_agrees(f"reduce_tabular_data/{chain_type}-{kappaflag}", {"study.csv": ours.read_text()}, run_reference)


@pytest.mark.parametrize("param,runflag", [("E0", False), ("Fz", False), ("FxFz", False), ("E0", True)])
def test_reference_aggregate_by_script_on_our_out_files(tmp_path, monkeypatch, param, runflag):
    """scripts/aggregate_by.jl (unmodified, run by minijl — including the `julia scripts/aggregate_mcmc.jl …` command it
    spawns per group, which a nested interpreter runs) splits a study into one table per combination of the other
    parameters; polymc.aggregate.aggregate_by gives the same files, upstream quirks included (with the run flag the glob
    wildcards only the last digit of the run number)."""
    from minijl.interp import Interp
    from polymc import aggregate as ag
    rng = np.random.default_rng(13)
    text, entries = [], []
    for e0 in (0.0, 0.5, 1.0):
        for fz, fx in ((0.0, 0.0), (0.25, 0.0), (0.25, 0.1)):
            for run in ((1, 2, 11) if runflag else (None,)):
                p = {"E0": e0, "K1": 1.0, "K2": 0.25, "kT": 1.0, "Fz": fz, "Fx": fx, "num-monomers": 100, "mlen": 1.0}
                avg, ex, ar = rng.normal(size=16), rng.normal(size=2), float(rng.uniform(0.01, 0.6))
                prefix = ag.prefix_of(p, "dielectric", False, run=run)
                text.append((prefix, ag.out_text(avg, ar, 1.0, 100, ex)))
                entries.append((prefix, ag.output_values(avg, ar, 1.0, 100, ex)))
    indir, outdir = tmp_path / "study", tmp_path / "by"
    ag.write_out_files(str(indir), text)
    ours = {}
    for name, (header, rows) in ag.aggregate_by(entries, param, "dielectric", False, runflag, 3).items():
        mine = tmp_path / ("ours_" + name)
        ag.write_table(str(mine), header, rows)
        ours[name] = mine.read_text()
    assert len(ours) >= 3

    def run_reference():
        monkeypatch.chdir(REF)            # the script spawns `julia scripts/aggregate_mcmc.jl` relative to the tree
        it = Interp(argv=[str(outdir), str(indir), param, "dielectric", "3D", "false"] + (["true"] if runflag else []))
        sink = io.StringIO()
        it.stdout = sink
        it.genv.vars["stdout"] = sink
        it.run_main(os.path.join(REF, "scripts", "aggregate_by.jl"))
        return {name: (outdir / name).read_text() for name in os.listdir(outdir)}
    assert_reference_agrees(f"aggregate_by/{param}-{runflag}", ours, run_reference)


LAUNCHERS = sorted(__import__("glob").glob(os.path.join(REF, "run", "*.jl"))) if REF else []
# two launchers draw their cases from Distributions.jl (no scripted stream here); one is not valid Julia upstream
# (`zip(a, b; c; d)`: positional arguments after the semicolon)
NOT_RUN = {"phases-random_2023-05-15.jl", "phases-random_2023-07-11.jl", "phases_2023-05-15.jl"}


@pytest.mark.skipif(not LAUNCHERS, reason="needs the reference's run/ launchers: set POLYMC_REFERENCE_DIR")
def test_every_reference_launcher_command_is_accepted_by_the_cli_twins(tmp_path):
    """north_star: "It keeps the existing CLI options … so run/* sweep scripts … work unchanged."  Every launcher of the
    reference's run/ directory is executed UNMODIFIED by minijl with the `julia <driver>.jl …` commands it spawns
    intercepted: a sample of each launcher's cases (first, last, every k-th) is checked — the driver is one of the two the
    package twins, the twin's parser accepts the whole command line, the values arrive, and the `<prefix>.out` file the
    launcher writes is named the way polymc.aggregate.prefix_of names it (so aggregate_mcmc.jl finds the parameters)."""
    from minijl.interp import Interp
    from minijl import builtins as B
    from polymc import aggregate as ag, mcmc, mcmc_clustering
    twins = {"mcmc_eap_chain.jl": mcmc, "mcmc_clustering_eap_chain.jl": mcmc_clustering}
    ran = commands = 0
    for path in LAUNCHERS:
        name = os.path.basename(path)
        if name in NOT_RUN:
            continue
        work = tmp_path / name
        work.mkdir()                          # (a few launchers expect their work directory to exist)
        it = Interp(argv=[str(work)])
        sink = io.StringIO()
        it.stdout = it.stderr = sink
        it.genv.vars["stdout"] = sink
        cmds = []
        it.cmd_runner = lambda argv, cmds=cmds: (cmds.append(list(argv)) or "<r>    =   [0.0, 0.0, 0.0]\\n")

        def sampled_pmap(f, cases, it=it):     # the launchers fan out with pmap: run a sample of the cases
            cases = list(B.iterate(cases))
            step = max(1, len(cases) // 25)
            for c in cases[::step] + cases[-1:]:
                it.call(f, [c])
            return None
        it.genv.vars["pmap"] = sampled_pmap
        it.run_main(path)
        assert cmds, name
        ran += 1
        for argv in cmds:
            commands += 1
            assert os.path.basename(argv[0]) == "julia", (name, argv[:4])
            k = next(i for i, a in enumerate(argv) if a.endswith(".jl"))
            driver, args = argv[k], argv[k + 1:]
            assert driver in twins, (name, driver)
            assert all(a in ("-t", "-O", "-p") or a.isdigit() for a in argv[1:k]), (name, argv[:k])    # julia's own flags
            p = twins[driver].parse_args(args)            # argparse exits on an option it does not know
            assert p["num-monomers"] == int(args[args.index("-n") + 1]) if "-n" in args else True
            assert p["E0"] == float(args[args.index("--E0") + 1])
            # the file the launcher writes: <workdir>/<prefix>.out with the tokens aggregate_mcmc.jl parses back
            prefix = os.path.basename(p["prefix"])
            tokens = dict(t.split("-", 1) for t in prefix.split("_"))
            chain = p["chain-type"]
            want = ag.prefix_of(p, chain, "kappa" in tokens, run=int(tokens["run"]) if "run" in tokens else None)
            wtok = dict(t.split("-", 1) for t in want.split("_"))
            if set(tokens) == set(wtok):      # (the older launchers write the run number unpadded: compare it as a number)
                assert {k: v for k, v in tokens.items() if k != "run"} == {k: v for k, v in wtok.items() if k != "run"}, (name, prefix, want)
                assert "run" not in tokens or int(tokens["run"]) == int(wtok["run"])
            # (some launchers run several variants per case: <prefix>_umbrella.out, or standard/<prefix>.out, …)
            assert any(f.startswith(prefix) and f.endswith(".out") for _, _, fs in os.walk(work) for f in fs), (name, prefix)
    assert ran >= 35 and commands >= 500
