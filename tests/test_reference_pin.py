"""The oracle, pinned to the reference itself (SURVEY §8c, VERDICT r01 "what's missing" #1).

tests/golden/ref/*.json hold outputs of the UNMODIFIED reference sources — inc/eap_chain.jl, inc/energy.jl,
inc/acceptance.jl, inc/average.jl (fine seams) and the three driver scripts mcmc_eap_chain.jl,
mcmc_clustering_eap_chain.jl, 2D/mcmc_clustering_eap_chain.jl run end to end with `rand` scripted to pop a tape of
uniforms (tests/golden/make_ref_fixtures.py; executed with tools/minijl because the image has no Julia, and runnable
with a real `julia` as well).  Here the CPU oracle is checked against them:

  * energies, Ω, r, p, ψ, move!, cluster_flip! (segment, α) on the fixtures' chains — to 1e-12·Σ|terms|;
  * whole driver runs in the oracle's tape mode (same uniforms in the reference's rand() call order): the same number
    of uniforms consumed, the same acceptance rate (every decision), trajectory / rolling rows and printed averages —
    for the literal algorithm (algo 0) AND the changed-term formulation (algo 1) the CUDA path implements;
  * the product's host formatting (polymc.output) reproduces the reference's stdout lines and CSV text byte for byte
    from the same numbers, and its CLI twins parse the reference's option lines to the same case.

The GPU library is then tied to the same files in tests/test_gpu_reference_pin.py.
"""
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest

from ref_tape import splitmix_tape

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = os.path.join(ROOT, "tests", "golden", "ref")
TOL = 1e-12


@pytest.fixture(scope="module")
def fine():
    with open(os.path.join(REF_DIR, "fine_seams.json")) as f:
        return json.load(f)


@pytest.fixture(scope="module")
def runs():
    with open(os.path.join(REF_DIR, "driver_runs.json")) as f:
        return json.load(f)["runs"]


def num(x):
    return float(x) if not isinstance(x, str) else {"NaN": math.nan, "Inf": math.inf, "-Inf": -math.inf}[x]


def oracle_case(O, c, **over):
    kw = dict(n=c["n"], E0=c["E0"], K1=c["K1"], K2=c["K2"], mu=c["mu"], kT=c["kT"], Fz=c["Fz"], Fx=c["Fx"], b=c["b"],
              chain_type=c["chain_type"], energy_type=c["energy_type"], kappa=c["kappa"], psi0=c["psi0"],
              cutoff_radius=c["cutoff_radius"], clustering=True)
    kw.update(over)
    return O.make_case(**kw)


def test_fixture_provenance(fine, runs):
    assert "unmodified reference" in fine["generator"] and len(fine["cases"]) == 16
    assert {r["driver"] for r in runs} == {"mcmc_eap_chain.jl", "mcmc_clustering_eap_chain.jl", "2D/mcmc_clustering_eap_chain.jl"}
    assert len(runs) >= 14


def test_energies_match_the_reference_functions(O, fine):
    """U(chain), U_interaction, U_Ising, UCutoff, Ω, r, p, Σψ, Σcos²θ of inc/eap_chain.jl on 16 chains."""
    for c in fine["cases"]:
        phi, th = np.array(c["phi"]), np.array(c["theta"])
        ch = O.Chain(oracle_case(O, c), phi, th)
        e = ch.energy_ex()
        scale = 1.0 + ch.abs_pair_sum() + abs(c["U"]) + abs(c["sum_us"])
        assert abs(e["U"] - c["U"]) <= TOL * scale, (c["name"], e["U"], c["U"])
        assert abs(e["su"] - c["sum_us"]) <= TOL * scale
        assert e["Omega"] == pytest.approx(c["Omega"], rel=1e-13, abs=1e-13)
        assert e["psi"] * (c["n"] - 1) == pytest.approx(c["sum_psi"], rel=1e-12)
        assert e["cos2"] == pytest.approx(c["sum_cos2"], rel=1e-13)
        np.testing.assert_allclose(ch.r(), c["r"], rtol=1e-13, atol=1e-13 * c["n"])
        np.testing.assert_allclose(ch.p(), c["p"], rtol=1e-13, atol=1e-13 * c["n"])
        # the three pair sums, whatever the chain's own energy type is
        for et, key in (("interacting", "U_interaction"), ("Ising", "U_Ising"), ("cutoff", "U_cutoff")):
            other = O.Chain(oracle_case(O, c, energy_type=et), phi, th)
            assert abs(other.energy()["Udd"] - c[key]) <= TOL * (1.0 + other.abs_pair_sum()), (c["name"], key)


def test_moves_match_the_reference_move(O, fine):
    """move!(copy, idx, dϕ, dθ) (inc/eap_chain.jl:230-257): the full-recompute result of the reference against both
    the oracle's literal move and its changed-pair ΔU (the formulation the CUDA path uses)."""
    for c in fine["cases"]:
        oc = oracle_case(O, c)
        ch = O.Chain(oc, np.array(c["phi"]), np.array(c["theta"]))
        scale = 1.0 + ch.abs_pair_sum() + abs(c["U"])
        for m in c["moves"]:
            idx0 = m["idx"] - 1
            t = ch.copy()
            t.move(idx0, m["dphi"], m["dtheta"])
            e = t.energy_ex()
            Uref, Oref = num(m["U"]), num(m["Omega"])
            assert abs(e["U"] - Uref) <= TOL * (scale + t.abs_pair_sum()), (c["name"], m)
            assert t.state()[1][idx0] == pytest.approx(m["theta_new"], abs=1e-15)
            if math.isfinite(Oref):
                assert e["Omega"] == pytest.approx(Oref, rel=1e-12, abs=1e-12)
            np.testing.assert_allclose(t.r(), m["r"], rtol=1e-12, atol=1e-12 * c["n"])
            np.testing.assert_allclose(t.p(), m["p"], rtol=1e-12, atol=1e-12 * c["n"])
            d = ch.delta_segment(idx0, m["dphi"], m["dtheta"], 0, idx0, idx0)
            assert abs(d["dU"] - (Uref - c["U"])) <= 20 * TOL * (scale + t.abs_pair_sum()), (c["name"], m["idx"])
            if math.isfinite(Oref):
                assert d["dOmega"] == pytest.approx(Oref - c["Omega"], rel=1e-10, abs=1e-11)
            else:
                assert d["dOmega"] == -math.inf


def test_cluster_flips_match_the_reference(O, fine):
    """move! + cluster_flip! (inc/eap_chain.jl:269-333): the reference's α and the state it leaves, against the oracle's
    segment update with the reference's own cluster bounds."""
    nflip = 0
    for c in fine["cases"]:
        oc = oracle_case(O, c)
        ch = O.Chain(oc, np.array(c["phi"]), np.array(c["theta"]))
        scale = 1.0 + ch.abs_pair_sum() + abs(c["U"])
        for f in c["cluster_flips"]:
            idx0 = f["idx"] - 1
            reflect = f["lo"] > 0
            lo0, hi0 = (f["lo"] - 1, f["hi"] - 1) if reflect else (idx0, idx0)
            if not reflect:
                assert f["alpha"] == 1.0 and f["draws"] >= 1
            else:
                assert lo0 <= idx0 <= hi0
                nflip += 1
            d = ch.delta_segment(idx0, f["dphi"], f["dtheta"], int(reflect), lo0, hi0)
            t = ch.copy()
            t.move_segment(idx0, f["dphi"], f["dtheta"], int(reflect), lo0, hi0)
            np.testing.assert_allclose(t.state()[1], f["theta"], rtol=0, atol=1e-15)
            np.testing.assert_allclose(t.state()[0], f["phi"], rtol=0, atol=1e-15)
            sc = scale + t.abs_pair_sum()
            assert abs(t.energy_ex()["U"] - num(f["U"])) <= TOL * sc
            assert abs(d["dU"] - (num(f["U"]) - c["U"])) <= 20 * TOL * sc, (c["name"], f["idx"])
            if math.isfinite(num(f["Omega"])):
                assert d["dOmega"] == pytest.approx(num(f["Omega"]) - c["Omega"], rel=1e-10, abs=1e-11)
            if reflect:       # α of eap_chain.jl:317-330 from the link probabilities before / after the reflection
                m = ch.copy()
                m.move(idx0, f["dphi"], f["dtheta"])
                n = c["n"]
                up = m.link_prob(hi0) if hi0 < n - 1 else 0.0
                lp = m.link_prob(lo0 - 1) if lo0 > 0 else 0.0
                nup = t.link_prob(hi0) if hi0 < n - 1 else 0.0
                nlp = t.link_prob(lo0 - 1) if lo0 > 0 else 0.0
                assert ((1 - nup) * (1 - nlp)) / ((1 - up) * (1 - lp)) == pytest.approx(f["alpha"], rel=1e-12)
            np.testing.assert_allclose(t.r(), f["r"], rtol=1e-12, atol=1e-12 * c["n"])
            np.testing.assert_allclose(t.p(), f["p"], rtol=1e-12, atol=1e-12 * c["n"])
            assert t.energy_ex()["cos2"] == pytest.approx(f["sum_cos2"], rel=1e-12)
            assert t.energy_ex()["psi"] * (c["n"] - 1) == pytest.approx(f["sum_psi"], rel=1e-12)
    assert nflip >= 30


def test_metropolis_functor_and_reinit_rule(fine):
    """inc/acceptance.jl:1-3, 24-37 — restated here in four lines each and replayed on the reference's own sequence:
    accept iff logπ+log α ≥ logπ_prev or ϵ < exp(·); on accept logπ_prev ← logπ + log α (the α carry)."""
    for c in fine["cases"]:
        prev = None
        for s in c["metropolis"]:
            prev_in = num(s["logpi_prev_before"])
            if prev is not None:
                assert prev_in == prev
            cur = num(s["logpi_trial"]) + math.log(s["alpha"])
            acc = cur >= prev_in or (math.isfinite(cur) and s["eps"] < math.exp(cur - prev_in))
            assert acc == s["accepted"]
            prev = cur if acc else prev_in
            assert num(s["logpi_prev_after"]) == pytest.approx(prev, rel=1e-15)
        assert c["logpi_weightless"] == pytest.approx(-c["U"] / c["kT"] + c["Omega"] + 1.0, rel=1e-14)   # WeightlessFunction ≡ 1.0
        cF = 0.2 + 0.8 * math.exp(-(c["Fx"] ** 2 + c["Fz"] ** 2) / c["kT"])
        assert c["weight"] == pytest.approx(c["sum_us"] / c["kT"] * cF - c["log_gauge"], rel=1e-13)
        g0 = (-(c["K1"] + 2 * c["K2"]) * c["E0"] ** 2 if c["chain_type"] == "dielectric" else -c["mu"] * c["E0"]) * c["n"] / (3 * c["kT"])
        assert c["log_gauge"] == pytest.approx(g0 + c["Omega"], rel=1e-13)
    for m in fine["metropolis_acc"]:
        assert (m["eps"] <= math.exp(-m["dU"] / m["kT"]) * m["s_b"] / m["s_a"]) == m["accept"]


# ---- whole driver runs ----------------------------------------------------------------------------------------------
def host_of(driver):
    import polymc.mcmc as plain
    import polymc.mcmc_clustering as cl
    import polymc.mcmc_clustering_2d as cl2
    return {"mcmc_eap_chain.jl": plain, "mcmc_clustering_eap_chain.jl": cl, "2D/mcmc_clustering_eap_chain.jl": cl2}[driver]


def oracle_case_from_pmc(O, pc, pm):
    ct = {v: k for k, v in pm.CHAIN_TYPES.items()}[pc.chain_type]
    et = {v: k for k, v in pm.ENERGY_TYPES.items()}[pc.energy_type]
    return O.make_case(n=pc.n, E0=pc.E0, K1=pc.K1, K2=pc.K2, mu=pc.mu, kT=pc.kT, Fz=pc.Fz, Fx=pc.Fx, b=pc.b,
                       chain_type=ct, energy_type=et, phi_step=pc.phi_step, theta_step=pc.theta_step, adj_lb=pc.adj_lb,
                       adj_ub=pc.adj_ub, adj_scale=pc.adj_scale, steps_per_adjust=pc.steps_per_adjust,
                       do_flips=bool(pc.do_flips), umbrella=bool(pc.umbrella), kappa=pc.kappa, psi0=pc.psi0,
                       cutoff_radius=pc.cutoff_radius, cluster_prob=pc.cluster_prob, clustering=bool(pc.clustering),
                       alpha_carry=bool(pc.alpha_carry), cutoff_full=bool(pc.cutoff_full), planar=bool(pc.planar))


def parse_csv(text):
    lines = text.strip().split("\n")
    return lines[0].split(","), np.array([[float(x) for x in ln.split(",")] for ln in lines[1:]])


def parse_stdout(lines):
    out = {}
    for ln in lines:
        k, v = ln.split("=", 1)
        v = v.strip()
        out[k.strip()] = np.array([float(x) for x in v.strip("[]").split(",")]) if v.startswith("[") else float(v)
    return out


def replay(O, pm, run, algo):
    """The protocol of the driver script on the oracle in tape mode.  Returns (traj rows, rolling rows, state rows or
    None, averages16, extras or None, acceptance rate, uniforms consumed)."""
    host = host_of(run["driver"])
    pargs = host.parse_args(run["options"] + ["--prefix", "x", "-v", "0"])
    oc = oracle_case_from_pmc(O, host.case_from_pargs(pargs), pm)
    tape = splitmix_tape(run["tape_seed"], run["tape_len"])
    r = O.Run(oc, 0, 0, algo, tape=tape, reinit_stale=True)
    stepout = pargs["stepout"]
    if run["driver"] == "mcmc_eap_chain.jl":
        trajs, rolls = [], []
        for init in range(pargs["num-inits"]):
            t, rl = r.steps(pargs["num-steps"], stepout)
            trajs.append(t)
            rolls.append(rl)
            r.reinit(force=pargs["force-init"])          # mcmc_eap_chain.jl:352-361 runs after EVERY init, the last too
        avg, _, _ = r.averages()
        ar = r.diag()["nacc_total"] / (pargs["num-inits"] * pargs["num-steps"])
        return np.concatenate(trajs), np.concatenate(rolls), None, avg, None, ar, r.tape_pos()
    from polymc.mcmc_clustering import parse_julia_vector
    if pargs.get("x0") is not None:
        r.init_x0(parse_julia_vector(pargs["x0"], "x0"), parse_julia_vector(pargs["dx0"], "dx0")[:2])
    for mult in parse_julia_vector(pargs["burn-schedule"], "burn-schedule"):
        r.begin_stage(pargs["kT"] * mult)
        r.steps_ex(pargs["burn-in"], stepout)
    r.begin_stage(pargs["kT"])
    t, rl, st = r.steps_ex(pargs["num-steps"], stepout, True)
    avg, ar, _ = r.averages()
    return t, rl, st, avg, r.extra_averages(), ar, r.tape_pos()


def _run_ids():
    with open(os.path.join(REF_DIR, "driver_runs.json")) as f:
        return [r["name"] for r in json.load(f)["runs"]]


@pytest.mark.parametrize("algo", [0, 1])
@pytest.mark.parametrize("name", _run_ids())
def test_driver_runs_match_the_reference_scripts(O, pm, runs, name, algo):
    run = next(r for r in runs if r["name"] == name)
    if algo == 1 and name.startswith("plain_ising_three_inits"):
        pytest.skip("the stale acceptor after a re-init swap (mcmc_eap_chain.jl:360) exists only in the literal algorithm")
    traj, roll, state, avg, extras, ar, used = replay(O, pm, run, algo)
    out = parse_stdout(run["stdout"])
    planar = run["driver"].startswith("2D/")
    assert used == run["tape_used"], "the oracle consumed a different number of uniforms than the reference"
    assert ar == pytest.approx(out["AR"], rel=1e-15)                                   # every accept/reject decision
    th, tr = parse_csv(run["trajectory_csv"])
    rh, rr = parse_csv(run["rolling_csv"])
    cols3 = [0, 1, 3, 4, 6, 7] if planar else list(range(8))       # the planar chain lives in the x–z plane of the 3-D rows
    scale = max(1.0, np.abs(tr[:, :len(cols3)]).max())
    np.testing.assert_allclose(traj[:, cols3], tr[:, :len(cols3)], rtol=0, atol=1e-9 * scale)
    if planar:
        rc = [0, 1, 3, 4, 6, 7, 8, 10, 11, 13, 14, 15, 16]
        assert rh == ["step", "r1", "r3", "r1sq", "r3sq", "rsq", "p1", "p3", "p1sq", "p3sq", "psq", "U", "Usq"]
        assert th == ["step", "r1", "r3", "p1", "p3", "U"]
    else:
        rc = list(range(rr.shape[1]))
    np.testing.assert_allclose(roll[:, rc], rr, rtol=1e-9, atol=1e-9 * max(1.0, np.abs(rr).max()))
    if state is not None and not planar:                       # phi1,theta1,phi2,theta2,… (mcmc_clustering_eap_chain.jl:317)
        n = state.shape[1] // 2
        np.testing.assert_allclose(state, tr[:, 8:8 + 2 * n], rtol=0, atol=1e-10)
    # the printed averages
    v3 = (lambda a: a[[0, 2]]) if planar else (lambda a: a)
    sc = max(1.0, np.abs(avg).max())
    np.testing.assert_allclose(v3(avg[0:3]), out["<r>"], rtol=0, atol=1e-10 * sc)
    np.testing.assert_allclose(v3(avg[3:6]), out["<rj2>"], rtol=0, atol=1e-10 * sc)
    np.testing.assert_allclose(v3(avg[7:10]), out["<p>"], rtol=0, atol=1e-10 * sc)
    np.testing.assert_allclose(v3(avg[10:13]), out["<pj2>"], rtol=0, atol=1e-10 * sc)
    for k, key in ((6, "<r2>"), (13, "<p2>"), (14, "<U>"), (15, "<U2>")):
        assert avg[k] == pytest.approx(out[key], rel=1e-10, abs=1e-10 * sc)
    if extras is not None and not planar:
        assert extras[0] == pytest.approx(out["<cos2(θ)>"], rel=1e-10)
        assert extras[1] == pytest.approx(out["<ψ>"], rel=1e-10)


def test_stale_acceptor_after_reinit_is_reference_behaviour(O, pm, runs):
    """ADVICE r01: mcmc_eap_chain.jl:360 swaps the chain but leaves acceptor.logπ_prev at the OLD chain's value.  The
    reference run with --num-inits 3 is reproduced only by the oracle's literal switch (reinit_stale); the rebinding
    variant — what the CUDA path and the oracle's default do, documented in DESIGN.md / the CLI help — differs."""
    run = next(r for r in runs if r["name"] == "plain_ising_three_inits")
    host = host_of(run["driver"])
    pargs = host.parse_args(run["options"] + ["--prefix", "x", "-v", "0"])
    oc = oracle_case_from_pmc(O, host.case_from_pargs(pargs), pm)
    tape = splitmix_tape(run["tape_seed"], run["tape_len"])
    out = parse_stdout(run["stdout"])
    res = {}
    for stale in (True, False):
        r = O.Run(oc, 0, 0, 0, tape=tape, reinit_stale=stale)
        swaps = 0
        for init in range(pargs["num-inits"]):
            r.steps(pargs["num-steps"], 0)
            swaps += int(r.reinit(force=False))
        res[stale] = (r.diag()["nacc_total"] / (pargs["num-inits"] * pargs["num-steps"]), swaps)
    assert res[True][0] == pytest.approx(out["AR"], rel=1e-15)
    if res[True][1] > 0:
        assert res[False][0] != res[True][0]


def test_host_formatting_reproduces_the_reference_text(runs):
    """polymc.output prints the reference's numbers exactly as the reference does (Julia's shortest round-trip Float64
    text): the stdout lines and both CSV files of every run, byte for byte."""
    import io
    from polymc import output as po
    for run in runs:
        out = parse_stdout(run["stdout"])
        planar = run["driver"].startswith("2D/")
        if planar:
            avg = np.zeros(16)
            avg[[0, 2]], avg[[3, 5]], avg[6] = out["<r>"], out["<rj2>"], out["<r2>"]
            avg[[7, 9]], avg[[10, 12]], avg[13] = out["<p>"], out["<pj2>"], out["<p2>"]
            avg[14], avg[15] = out["<U>"], out["<U2>"]
            pargs = host_of(run["driver"]).parse_args(run["options"] + ["--prefix", "x"])
            lines = po.result_lines_2d(avg, out["AR"], pargs["mlen"], pargs["num-monomers"])
        else:
            avg = np.concatenate([out["<r>"], out["<rj2>"], [out["<r2>"]], out["<p>"], out["<pj2>"], [out["<p2>"], out["<U>"], out["<U2>"]]])
            pargs = host_of(run["driver"]).parse_args(run["options"] + ["--prefix", "x"])
            if "<ψ>" in out:
                lines = po.result_lines_clustering(avg, out["<cos2(θ)>"], out["<ψ>"], out["AR"], pargs["mlen"], pargs["num-monomers"])
            else:
                lines = po.result_lines(avg, out["AR"], pargs["mlen"], pargs["num-monomers"])
        # <r/nb> is a derived line: r / (mlen·n) is recomputed, everything else must be the identical text
        for mine, ref in zip(lines, run["stdout"]):
            if ref.startswith("<r/nb>"):
                np.testing.assert_allclose(parse_stdout([mine])["<r/nb>"], parse_stdout([ref])["<r/nb>"], rtol=1e-15)
            else:
                assert mine == ref
        for key in ("trajectory_csv", "rolling_csv"):
            head, rows = parse_csv(run[key])
            buf = io.StringIO()
            po.write_rows(buf, rows)
            assert buf.getvalue() == run[key].split("\n", 1)[1]
        if not planar:
            n = pargs["num-monomers"]
            want = po.TRAJ_HEADER if run["driver"] == "mcmc_eap_chain.jl" else po.traj_header_clustering(n)
            assert run["trajectory_csv"].split("\n", 1)[0] == want
            want = po.ROLL_HEADER if run["driver"] == "mcmc_eap_chain.jl" else po.ROLL_HEADER_CLUSTERING
            assert run["rolling_csv"].split("\n", 1)[0] == want


REFERENCE = os.environ.get("POLYMC_REFERENCE_DIR")


@pytest.mark.skipif(not REFERENCE or not os.path.isdir(os.path.join(REFERENCE, "inc")),
                    reason="needs the reference sources: set POLYMC_REFERENCE_DIR")
def test_fixtures_regenerate_from_the_reference_sources(runs):
    """Freshness: one driver run regenerated NOW from the reference sources equals the committed fixture."""
    name = "cluster_noninteracting_x0"
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "golden", "make_ref_fixtures.py"), "--only", name,
                        "--reference", REFERENCE],
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    fresh = json.load(open(p.stdout.strip().split("\n")[-1]))["runs"][0]
    want = next(r for r in runs if r["name"] == name)
    for k in ("stdout", "trajectory_csv", "rolling_csv", "tape_used"):
        assert fresh[k] == want[k]
