"""GPU parity tests added in round 2 (VERDICT r01 "next" #1-#3): the run kernel of the real n=4096 launch shape, the
polar n=512 configuration (C3), the 3σ ensemble test at C2's own parameters, packing by ensemble hint, pmc_kernel_name, checkpoints, and one ensemble over several devices behind the C ABI.

Everything goes through the C ABI (polymc.lib → libpolymc_b200.so); the oracle is the checker only.
"""
import math
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from conftest import both_cases

pytestmark = pytest.mark.gpu


def _compare_run(ens, run, chain, traj, roll, steps, stepout, scale_pairs=False):
    ot, orl = run.steps(steps, stepout)
    d, od = ens.diagnostics()[chain], run.diag()
    assert d[4] == od["nacc_total"] and d[5] == od["steps_total"], (chain, d[4], od["nacc_total"])
    assert d[0] == pytest.approx(od["phi_step"], rel=1e-14) and d[1] == pytest.approx(od["theta_step"], rel=1e-14)
    scale = max(1.0, np.abs(ot).max(), run.chain().abs_pair_sum() if scale_pairs else 0.0)
    np.testing.assert_allclose(traj[chain], ot, rtol=0, atol=1e-9 * scale)
    np.testing.assert_allclose(roll[chain], orl, rtol=1e-9, atol=1e-9 * max(1.0, np.abs(orl).max()))
    phi, th = ens.get_state(chain)
    ophi, oth = run.chain().state()
    np.testing.assert_allclose(phi, ophi, rtol=0, atol=1e-12)
    np.testing.assert_allclose(th, oth, rtol=0, atol=1e-12)


def test_c5_run_kernel_trajectory_n4096(pm, O, monkeypatch):
    """The kernel behind the C5 number — whatever the library picks for n=4096 at the C5 ensemble size, asked
    through pmc_kernel_name — against oracle algo 1: 2 chains × 120 trials, same decisions, rows to 1e-9·scale.
    The windowed one-CTA kernel does not fit this chain, so it runs on CTA pairs even with pairs switched off."""
    n, steps = 4096, 120
    pc, oc = both_cases(pm, O, n=n, E0=1.0, K1=1.0, K2=0.0, Fz=0.5, energy_type="interacting", steps_per_adjust=40)
    with pm.Ensemble(pc, replicas=2, seed=20260101, ensemble_chains=148) as ens:
        name = ens.kernel_name()
        assert name.startswith("k_run_cta_pair<512"), name
        monkeypatch.setenv("PMC_RUN_PAIR", "0")
        assert ens.kernel_name().startswith("k_run_cta_pair<512"), ens.kernel_name()
        monkeypatch.delenv("PMC_RUN_PAIR")
        traj, roll = ens.run(steps, 30)
        for c in (0, 1):
            _compare_run(ens, O.Run(oc, 20260101, c, 1), c, traj, roll, steps, 30, scale_pairs=True)


def test_polar_n512_trajectory(pm, O):
    """Config C3's chain: polar monomers with dipole-dipole coupling, n=512, several (mu, E0, Fz) sweep points in one
    handle; the headline kernel on the shared Philox stream takes the oracle's decisions."""
    pts = [dict(mu=0.1, E0=1.0, Fz=1.0), dict(mu=0.2, E0=10.0, Fz=-1.0), dict(mu=0.01, E0=0.1, Fz=5.0)]
    cases = [both_cases(pm, O, n=512, chain_type="polar", energy_type="interacting", steps_per_adjust=100, **p)
             for p in pts]
    with pm.Ensemble([c[0] for c in cases], replicas=2, seed=303) as ens:
        assert ens.kernel_name().startswith("k_run_cta_win<")
        traj, roll = ens.run(500, 100)
        for ci, (_, oc) in enumerate(cases):
            chain = 2 * ci + 1
            _compare_run(ens, O.Run(oc, 303, chain, 1), chain, traj, roll, 500, 100, scale_pairs=True)


_C2_CPU = {}   # the CPU arm of the C2 statistics test, computed once for both precisions


@pytest.mark.parametrize("precision", ["fp64", "fp32"])
def test_c2_parameters_three_sigma_vs_reference_algorithm(pm, O, precision):
    """north_star's statistical gate at the headline configuration itself: interacting dielectric n=512, E0=1, kT=1,
    Fz=0.5 (C2).  GPU: 4096 replicas; CPU: the oracle's algo 0 (= the reference's own algorithm: full recompute,
    stateful acceptor) on all host cores with a different seed.  Both sides follow the reference protocol (averages
    from step 1, θ~U(0,π) initial chains), so the per-replica averages after the same number of trials are i.i.d.
    draws from the same law: all 16 averages — including <U> and <U²> — and the acceptance rate must agree within
    3σ of the combined standard error of the replica means; the rolling rows give per-replica batch means, whose
    late-batch averages must agree as well."""
    kw = dict(n=512, E0=1.0, K1=1.0, K2=0.0, kT=1.0, b=1.0, Fz=0.5, Fx=0.0, energy_type="interacting")
    pc, oc = both_cases(pm, O, **kw)
    steps, stepout = 6000, 1000
    Rg = 4096
    Rc = max(32, 2 * (os.cpu_count() or 8))
    with pm.Ensemble(pc, replicas=Rg, seed=777) as ens:
        # fp32: the opt-in FP32 rectangle (pmc_set_pair_precision) must pass the same gate against the FP64 reference algorithm
        ens.set_pair_precision(precision)
        assert ens.pair_precision() == precision
        _, groll = ens.run(steps, stepout)
        g_avg, g_ar, _ = ens.averages()

    def one(c):
        run = O.Run(oc, 4242, c, 0)
        _, rl = run.steps(steps, stepout)
        a, ar, _ = run.averages()
        return a, ar, rl
    if "res" not in _C2_CPU:
        with ThreadPoolExecutor(max_workers=os.cpu_count() or 8) as ex:   # ctypes releases the GIL
            _C2_CPU["res"] = list(ex.map(one, range(Rc)))
    res = _C2_CPU["res"]
    c_avg = np.array([r[0] for r in res])
    c_ar = np.array([r[1] for r in res])
    croll = np.array([r[2] for r in res])
    for k in range(16):
        sg = g_avg[:, k].std(ddof=1) / math.sqrt(Rg)
        sc = c_avg[:, k].std(ddof=1) / math.sqrt(Rc)
        assert abs(g_avg[:, k].mean() - c_avg[:, k].mean()) <= 3.0 * math.hypot(sg, sc) + 1e-12, (pm.AVG_NAMES[k],
                                                                                                g_avg[:, k].mean(),
                                                                                                c_avg[:, k].mean(), sg, sc)
    sg, sc = g_ar.std(ddof=1) / math.sqrt(Rg), c_ar.std(ddof=1) / math.sqrt(Rc)
    assert abs(g_ar.mean() - c_ar.mean()) <= 3.0 * math.hypot(sg, sc)

    # batch means: the rolling average times its step count is the running sum; its increments are the batches
    def batches(roll, col):
        k = roll[:, :, 0]
        return np.diff(np.concatenate([np.zeros((roll.shape[0], 1)), roll[:, :, col] * k], axis=1), axis=1) / stepout
    for col in (3, 7, 10, 14, 15, 16):   # r3, rsq, p3, psq, U, Usq
        bg, bc = batches(groll, col)[:, 2:].mean(axis=1), batches(croll, col)[:, 2:].mean(axis=1)
        sg, sc = bg.std(ddof=1) / math.sqrt(Rg), bc.std(ddof=1) / math.sqrt(Rc)
        assert abs(bg.mean() - bc.mean()) <= 3.0 * math.hypot(sg, sc) + 1e-12, (col, bg.mean(), bc.mean(), sg, sc)


def test_packing_follows_the_ensemble_hint(pm):
    """ADVICE r01 / VERDICT weak #5: the chain-per-lane vs chain-per-warp choice follows pmc_set_ensemble_hint like the
    block size does, so a shard of a large sweep runs the kernel the whole ensemble would and its results are
    bit-identical to the unsharded run — across the lane/warp threshold."""
    c = pm.make_case(n=16, E0=1.0, Fz=0.5, energy_type="Ising")
    R = 81920                                  # above the chain-per-lane threshold (65 536 for Ising chains)
    with pm.Ensemble(c, replicas=R, seed=6) as whole:
        assert whole.kernel_name().startswith("k_run_lane<")
        whole.run(400, 0)
        want = whole.averages()[0]
    half = R // 2
    for base in (0, half):
        with pm.Ensemble(c, replicas=half, seed=6, chain_id_base=base) as part:
            assert part.kernel_name().startswith("k_run_warp<")       # its own size would pick the other packing
            part.set_ensemble_hint(R)
            assert part.kernel_name().startswith("k_run_lane<")
            part.run(400, 0)
            np.testing.assert_array_equal(part.averages()[0], want[base:base + half])
    k = pm.make_case(n=16, E0=1.0, Fz=0.5, energy_type="Ising", kappa=0.5, clustering=True, adj_ub=0.4)
    with pm.Ensemble(k, replicas=512, seed=6) as part:
        assert part.kernel_name().startswith("k_run_warp_cluster<")
        part.set_ensemble_hint(16384)
        assert part.kernel_name().startswith("k_run_lane_cluster<")


def test_kernel_name_is_the_librarys_own_decision(pm):
    c2 = pm.make_case(n=512, E0=1.0, Fz=0.5, energy_type="interacting")
    with pm.Ensemble(c2, replicas=8, seed=1, ensemble_chains=4096) as ens:
        assert ens.kernel_name() == "k_run_cta_win<128,4,2>"
    k1 = pm.make_case(n=100, E0=1.0, Fz=0.25, energy_type="interacting", kappa=0.5, clustering=True)
    with pm.Ensemble(k1, replicas=8, seed=1, ensemble_chains=4096) as ens:
        assert ens.kernel_name().startswith("k_run_cta_cluster<32,10")
    c4 = pm.make_case(n=100, E0=1.0, Fz=0.5)
    with pm.Ensemble(c4, replicas=64, seed=1) as ens:
        assert ens.kernel_name().startswith("k_run_warp<0,")


@pytest.mark.parametrize("kw", [dict(n=96, energy_type="interacting"), dict(n=50, energy_type="Ising"),
                                dict(n=64, energy_type="interacting", kappa=0.5, clustering=True, adj_ub=0.4)])
def test_checkpoint_resume_is_bit_identical(pm, kw):
    """pmc_checkpoint_save / _load: a run continued in a fresh handle (a later process) from the blob equals the
    uninterrupted run bit for bit — state, accumulators, step sizes, counters, rows."""
    c = pm.make_case(E0=1.0, K2=0.1, Fz=0.5, Fx=0.1, steps_per_adjust=100, **kw)
    clustering = bool(kw.get("clustering"))

    def go(ens, steps):
        return ens.run_ex(steps, 100)[:2] if clustering else ens.run(steps, 100)
    with pm.Ensemble(c, replicas=5, seed=99, chain_id_base=3) as a, pm.Ensemble(c, replicas=5, seed=99, chain_id_base=3) as b:
        if clustering:
            a.begin_stage(2.0)
            b.begin_stage(2.0)
        go(a, 700)
        blob = a.checkpoint()
        ta, ra = go(a, 500)
        with pm.Ensemble(c, replicas=5, seed=99, chain_id_base=3) as fresh:
            fresh.restore(blob)
            tf, rf = go(fresh, 500)
            np.testing.assert_array_equal(tf, ta)
            np.testing.assert_array_equal(rf, ra)
            np.testing.assert_array_equal(fresh.accumulators(), a.accumulators())
            np.testing.assert_array_equal(fresh.diagnostics()[:, :6], a.diagnostics()[:, :6])
            np.testing.assert_array_equal(fresh.get_state_all()[0], a.get_state_all()[0])
        tb, _ = go(b, 1200)
        np.testing.assert_allclose(tb[:, 7:], ta, rtol=0, atol=1e-9 * max(1.0, np.abs(ta).max()))
        with pm.Ensemble(c, replicas=4, seed=99, chain_id_base=3) as other:
            with pytest.raises(pm.PolymcError):
                other.restore(blob)


def test_accumulators_dd_are_the_sums(pm):
    c = pm.make_case(n=40, E0=1.0, Fz=0.5, energy_type="Ising", accum_mode=1)
    with pm.Ensemble(c, replicas=3, seed=5) as ens:
        ens.run(5000, 0)
        hi, lo = ens.accumulators_dd()
        s = ens.accumulators()
        np.testing.assert_allclose(hi[:, :17] + lo[:, :17], s, rtol=1e-15)
        assert np.all(np.abs(lo) <= np.spacing(np.abs(hi)))       # a normalised double-double
        assert np.all(hi[:, 16] == 5000.0)


def _check_multi_against_single(pm, devices, R, kw, steps, stepout, expect_backend=None):
    c = [pm.make_case(**kw), pm.make_case(**dict(kw, Fz=1.0, kT=0.8))]
    with pm.MultiEnsemble(c, replicas=R, seed=31, devices=devices) as m, pm.Ensemble(c, replicas=R, seed=31) as one:
        assert m.ndevices == len(devices) and m.nchains == 2 * R
        if expect_backend:
            assert m.gather_backend() == expect_backend
        one.set_ensemble_hint(0)
        # every shard picks its launch shape from the same ensemble size ⇒ bit-identical to the single handle
        m.set_ensemble_hint(2 * R)
        one.set_ensemble_hint(2 * R)
        np.testing.assert_array_equal(m.get_state_all()[0], one.get_state_all()[0])
        tm, rm = m.run(steps, stepout)
        t1, r1 = one.run(steps, stepout)
        np.testing.assert_array_equal(tm, t1)
        np.testing.assert_array_equal(rm, r1)
        tab = m.gather()
        avg, ar, nrm = one.averages()
        np.testing.assert_array_equal(tab[:, :16], avg)
        np.testing.assert_array_equal(tab[:, 16], ar)
        np.testing.assert_array_equal(tab[:, 17], nrm)
        d = one.diagnostics()
        np.testing.assert_array_equal(tab[:, 18:22], d[:, [0, 1, 5, 6]])
        # asynchronous run + set_state through the ensemble-wide seams
        phi, th = one.get_state_all()
        m.set_state_all(phi, th)
        tr, rl = m.run_async(steps, stepout)
        m.wait()
        t2, r2 = one.run(steps, stepout)
        np.testing.assert_array_equal(tr, t2)
        sh = m.shard(len(devices) - 1)
        assert sh.first + sh.nchains == 2 * R and sh.device == devices[-1]
        np.testing.assert_array_equal(sh.energy_all(), one.energy_all()[sh.first:])
        with pytest.raises(pm.PolymcError):
            m.run_async(10, 0)
            m.run(10, 0)            # a run is in flight
        m.wait()


@pytest.mark.parametrize("kw,steps", [(dict(n=96, E0=1.0, Fz=0.5, energy_type="interacting", steps_per_adjust=100), 600),
                                      (dict(n=60, E0=1.0, Fz=0.5, energy_type="Ising", steps_per_adjust=100), 3000)])
def test_multi_device_abi_on_one_gpu(pm, kw, steps):
    """pmc_multi_* with several shards on ONE device (device list [0,0,0]; NCCL needs distinct devices, so the rows
    travel by device-to-device copies): slices, host threads, gather and padding (odd shard sizes)."""
    _check_multi_against_single(pm, [0, 0, 0], 5, kw, steps, 100, expect_backend="peer")


def test_multi_device_ensemble_refuses_cases_that_would_pick_different_kernels(pm):
    """A shard validates its cases against its own first case only, and a handle runs the composite-trial kernels as soon
    as one of its cases bends: the ensemble-wide check keeps a case's kernel independent of the device split."""
    base = dict(E0=1.0, Fz=0.5, energy_type="interacting")
    for a, b in [(dict(base, n=48), dict(base, n=64)),
                 (dict(base, n=48), dict(base, n=48, energy_type="Ising")),
                 (dict(base, n=48), dict(base, n=48, kappa=0.5))]:
        with pytest.raises(pm.PolymcError, match="must share"):
            pm.MultiEnsemble([pm.make_case(**a), pm.make_case(**b)], replicas=2, seed=1, devices=[0, 0])


def test_multi_device_abi_over_all_gpus(pm):
    """≥ 2 GPUs: one process drives every device through pmc_multi_*, the result rows are gathered with ONE
    ncclAllGather over NVLink, and the results equal the single-device run bit for bit."""
    G = pm.device_count()
    if G < 2:
        pytest.skip("needs >= 2 GPUs")
    kw = dict(n=128, E0=1.0, Fz=0.5, energy_type="interacting", steps_per_adjust=100)
    _check_multi_against_single(pm, list(range(G)), 37, kw, 500, 100, expect_backend="nccl")


def test_umbrella_replicas_pooled_as_ratios_match_closed_form(pm):
    """ADVICE r01 (medium): --umbrella-sampling with --replicas R.  Per-replica gauges differ by exp(Ω0_r), so the
    hosts pool the per-replica ratios; the pooled estimate agrees with the closed form within 3σ of the replica
    spread, every replica carries the same weight, and the naive Σ values / Σ normalisers is dominated by few."""
    import closed_form as CF
    from polymc.mcmc import pool_replicas
    kw = dict(E0=2.0, K1=1.0, K2=0.0, Fz=1.5)
    n, R = 30, 16
    cf = CF.chain_averages(n, **kw)
    with pm.Ensemble(pm.make_case(n=n, energy_type="noninteracting", umbrella=True, **kw), replicas=R, seed=12) as ens:
        ens.run(60000, 0)
        sums = ens.accumulators()
    pooled, norm = pool_replicas(sums, umbrella=True)
    ratios = sums[:, :16] / sums[:, 16:17]
    sem = ratios.std(axis=0, ddof=1) / math.sqrt(R)
    for k in (2, 5, 6, 9, 14):            # r3, r3sq, rsq, p3, U
        assert abs(pooled[k] / norm - cf[k]) <= 3.0 * sem[k] + 1e-9 * max(1.0, abs(cf[k])), (pm.AVG_NAMES[k], pooled[k], cf[k])
    w = sums[:, 16] / sums[:, 16].sum()
    assert w.max() > 2.0 / R              # the raw normalisers ARE unequal (why the sums are not pooled)


@pytest.mark.parametrize("n,R,steps", [(96, 3, 2000), (512, 5, 600), (700, 150, 300)])
def test_pair_kernel_trajectory(pm, O, monkeypatch, n, R, steps):
    """k_run_cta_pair (two SMs per chain: a 2-CTA cluster splits the changed-pair set, partial sums exchanged through
    distributed shared memory, chains taken from a work-ordered queue), forced for short chains with PMC_RUN_PAIR=2:
    same decisions, rows, step sizes and final state as the oracle; launches chunk like the one-CTA kernels; more chains
    than resident clusters (150 > 74) exercise the queue."""
    monkeypatch.setenv("PMC_RUN_PAIR", "2")
    pc, oc = both_cases(pm, O, n=n, E0=1.0, K2=0.1, Fz=0.5, Fx=0.2, energy_type="interacting", steps_per_adjust=100)
    with pm.Ensemble(pc, replicas=R, seed=23, chain_id_base=7) as ens, pm.Ensemble(pc, replicas=R, seed=23, chain_id_base=7) as two:
        assert ens.kernel_name().startswith("k_run_cta_pair<")
        traj, roll = ens.run(steps, steps // 4)
        for c in sorted({0, R // 2, R - 1}):
            _compare_run(ens, O.Run(oc, 23, 7 + c, 1), c, traj, roll, steps, steps // 4, scale_pairs=True)
        t1, _ = two.run(steps // 2, steps // 4)
        t2, _ = two.run(steps // 2, steps // 4)
        np.testing.assert_array_equal(np.concatenate([t1, t2], axis=1)[:, :, 0], traj[:, :, 0])
        np.testing.assert_array_equal(two.diagnostics()[:, 4:6], ens.diagnostics()[:, 4:6])
        np.testing.assert_allclose(np.concatenate([t1, t2], axis=1), traj, rtol=0, atol=1e-9 * max(1.0, np.abs(traj).max()))
        counts = ens.diagnostics()[:, 4:6]
    monkeypatch.setenv("PMC_RUN_PAIR", "0")
    with pm.Ensemble(pc, replicas=R, seed=23, chain_id_base=7) as one:
        assert not one.kernel_name().startswith("k_run_cta_pair<")
        t0, _ = one.run(steps, steps // 4)
        np.testing.assert_allclose(t0, traj, rtol=0, atol=1e-9 * max(1.0, np.abs(traj).max()))
        np.testing.assert_array_equal(one.diagnostics()[:, 4:6], counts)


def test_cli_numeric_type_float128_prints_double_double_averages(pm, tmp_path):
    """--numeric-type float128: the device sums are double-double (pmc_accumulators_dd) and the CLI twin prints their
    exact quotients with 36 significant digits; to double precision they equal the float64 run (same seed)."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    outs = {}
    for nt in ("float64", "float128"):
        argv = [sys.executable, os.path.join(root, "polymer-stats_b200", "mcmc_eap_chain.py"), "--energy-type", "Ising",
                "--E0", "1.0", "--Fz", "0.5", "-n", "30", "--num-steps", "20000", "--stepout", "5000", "-v", "0",
                "--prefix", str(tmp_path / nt), "--seed", "11", "--replicas", "3", "--numeric-type", nt]
        p = subprocess.run(argv, capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stderr
        outs[nt] = p.stdout.strip().split("\n")
    assert len(outs["float128"]) == 10
    for a, b in zip(outs["float64"], outs["float128"]):
        ka, va = a.split("=", 1)
        kb, vb = b.split("=", 1)
        assert ka == kb
        xa = [float(x) for x in va.strip().strip("[]").split(",")]
        xb = [float(x) for x in vb.strip().strip("[]").split(",")]
        np.testing.assert_allclose(xa, xb, rtol=1e-13, atol=1e-13)
    assert len(outs["float128"][3].split("=")[1].strip()) >= 40          # 36 significant digits + exponent


@pytest.mark.parametrize("kw", [
    dict(n=64, E0=1.0, K1=1.0, K2=0.1, Fz=0.5, Fx=0.1, steps_per_adjust=100),
    dict(n=48, E0=0.4, Fz=0.3, kT=4.0, chain_type="polar", mu=0.5, do_flips=True, steps_per_adjust=333),   # acceptance ≈ 0.5
    dict(n=24, E0=2.0, Fz=0.0, kT=0.5, umbrella=True),
    dict(n=100, E0=1.0, Fz=0.5),                                                                            # eight teams only
])
def test_speculative_teams_of_the_plain_driver_are_the_sequential_chain(pm, kw):
    """k_run_cta_win_spec: small ensembles of short interacting chains run 2, 4 or 8 one-warp teams per chain on different
    trials of the window and commit them in order.  Acceptance counts and final chains are identical to the one-trial
    kernel (k_run_cta_win), rows agree to the rounding of the pair-sum order."""
    case = pm.make_case(energy_type="interacting", **kw)
    R, steps = 10, 4000
    ref = None
    for hint, teams in ((10 ** 6, 0), (800, 2), (300, 4), (0, 8)):
        if kw["n"] > 64 and teams in (2, 4):
            continue                      # longer chains: speculation only when every chain can have a whole SM
        with pm.Ensemble(case, replicas=R, seed=515, ensemble_chains=hint) as ens:
            name = ens.kernel_name()
            assert name.startswith(f"k_run_cta_win_spec<{teams}," if teams else "k_run_cta_win<"), name
            traj, roll = ens.run(steps, 500)
            ens.run(777, 0)
            got = dict(acc=ens.diagnostics()[:, 4].copy(), final=ens.get_state_all(), traj=traj, roll=roll, avg=ens.averages()[0])
        if ref is None:
            ref = got
            assert 0 < ref["acc"].sum() < R * (steps + 777)
            continue
        np.testing.assert_array_equal(got["acc"], ref["acc"])
        for a, b in zip(got["final"], ref["final"]):
            np.testing.assert_array_equal(a, b)
        for key in ("traj", "roll", "avg"):   # the initial r, p, U come from a reduction whose order follows the block size
            np.testing.assert_allclose(got[key], ref[key], rtol=1e-9, atol=1e-9)
