"""Replica exchange across kT and force ladders on the GPU (pmc_set_ladders, pmc_exchange, pmc_run_tempering*,
pmc_exchange_stats): the exchange kernel against the rule restated on the host, whole tempered runs against the
oracle on the shared Philox stream, the fused driver against the explicit loop, checkpoints, the closed-form
ensembles at 4096 chains, walker labels, and the refusals of the C ABI.

Everything goes through the C ABI (polymc.lib → libpolymc_b200.so); the oracle and tests/tempering_ref.py check.
"""
import math

import numpy as np
import pytest

import closed_form as CF
import tempering_ref as TR
from conftest import both_cases

pytestmark = pytest.mark.gpu

# pmc_checkpoint_save layout (polymc.cu CkptHeader, chain_math.cuh MonoRec / ChainDyn / ChainDynX)
_HDR = 72
_MONO = np.dtype([("phi", "f8"), ("theta", "f8"), ("nx", "f8"), ("ny", "f8"), ("nz", "f8"), ("sth", "f8")])
_DYN = np.dtype([("U", "f8"), ("Omega", "f8"), ("su", "f8"), ("r", "f8", 3), ("p", "f8", 3), ("phi_step", "f8"),
                 ("theta_step", "f8"), ("log_gauge", "f8"), ("drift_max", "f8"), ("acc", "f8", 17),
                 ("comp", "f8", 17), ("nacc", "i8"), ("natt", "i8"), ("nacc_total", "i8"), ("steps_total", "i8"),
                 ("step", "i8"), ("init", "i4"), ("valid", "i4")])
_DYNX = np.dtype([("spsi", "f8"), ("scos2", "f8"), ("carry", "f8"), ("acc", "f8", 2), ("comp", "f8", 2),
                  ("ncluster", "f8"), ("cluster_sum", "f8"), ("cluster_max", "f8")])
_MOVES = ("Omega", "su", "r", "p")                      # ChainDyn fields that travel with the configuration
_STAYS = ("phi_step", "theta_step", "log_gauge", "drift_max", "acc", "comp", "nacc", "natt", "nacc_total",
          "steps_total", "step", "init", "valid")


def _snapshot(ens):
    """The device state of every chain, read from a checkpoint: records [chains][n], ChainDyn, ChainDynX."""
    blob = ens.checkpoint()
    c, n = ens.nchains, ens.n
    assert len(blob) >= _HDR + c * n * _MONO.itemsize + c * (_DYN.itemsize + _DYNX.itemsize)
    off = _HDR
    mono = np.frombuffer(blob, _MONO, c * n, off).reshape(c, n)
    off += c * n * _MONO.itemsize
    dyn = np.frombuffer(blob, _DYN, c, off)
    dynx = np.frombuffer(blob, _DYNX, c, off + c * _DYN.itemsize)
    return mono, dyn, dynx


def _same(x, y):
    x, y = np.ascontiguousarray(x).reshape(-1), np.ascontiguousarray(y).reshape(-1)
    return x.dtype == y.dtype and np.array_equal(x.view(np.uint8), y.view(np.uint8))


def _check_round(ens, cases, book, seed, kT_scale, pre, post, acc):
    """One pmc_exchange against the host restatement: the decisions (same Δ from the same inputs, same ε), and what
    moved and what stayed, bit for bit."""
    mono0, dyn0, dynx0 = pre
    mono1, dyn1, dynx1 = post
    want = np.zeros(ens.nchains, np.int32)
    swapped = set()
    R = ens.replicas
    for a, b, stat, flags in book.round_pairs():
        ca, cb = cases[a // R], cases[b // R]
        delta, Uab, Uba = TR.exchange_delta(ca.kT * kT_scale, cb.kT * kT_scale, dyn0["U"][a], dyn0["U"][b],
                                            dyn0["r"][a], dyn0["r"][b], ca.Fx, ca.Fz, cb.Fx, cb.Fz)
        take = delta >= 0.0 or TR.draw_exchange_eps(seed, a, int(dyn0["init"][a]), book.round) < math.exp(delta)
        book.record(a, b, stat, flags, take)
        if not take:
            continue
        want[a] = 1
        swapped |= {a, b}
        assert _same(mono1[a], mono0[b]) and _same(mono1[b], mono0[a])
        assert dyn1["U"][a] == Uab and dyn1["U"][b] == Uba
        for f in _MOVES:
            assert _same(dyn1[f][a], dyn0[f][b]) and _same(dyn1[f][b], dyn0[f][a]), f
        for f in ("spsi", "scos2"):
            assert _same(dynx1[f][a], dynx0[f][b]) and _same(dynx1[f][b], dynx0[f][a]), f
        assert dynx1["carry"][a] == 0.0 and dynx1["carry"][b] == 0.0
    book.round += 1
    np.testing.assert_array_equal(acc, want)
    for f in _STAYS:
        assert _same(dyn1[f], dyn0[f]), f
    for f in ("acc", "comp", "ncluster", "cluster_sum", "cluster_max"):
        assert _same(dynx1[f], dynx0[f]), f
    still = np.array([c not in swapped for c in range(ens.nchains)])
    assert _same(mono1[still], mono0[still]) and _same(dyn1[still], dyn0[still]) and _same(dynx1[still], dynx0[still])
    return int(want.sum())


KERNEL_CASES = {
    # plain driver, interacting n = 64: a kT ladder with --do-flips, and a force ladder
    "plain_kT_flips": (dict(n=64, E0=1.0, K2=0.1, Fz=0.5, energy_type="interacting", do_flips=True, steps_per_adjust=100),
                       "kT", [0.6, 0.9, 1.4, 2.0], 3, 0),
    "plain_Fz": (dict(n=64, E0=1.0, K2=0.1, kT=1.0, Fx=0.2, energy_type="interacting", steps_per_adjust=100),
                 "Fz", [0.0, 0.4, 0.9, 1.6], 3, 0),
    # the headline kernel: n = 512 in a 4096-chain launch shape
    "plain_n512": (dict(n=512, E0=1.0, K2=0.1, Fz=0.5, energy_type="interacting", steps_per_adjust=100),
                   "kT", [0.8, 1.0, 1.3], 2, 4096),
    # the clustering driver, all pairs + bending, α carry off and on
    "cluster_carry0": (dict(n=100, E0=1.0, K2=0.1, Fz=0.5, energy_type="interacting", kappa=0.5, clustering=True,
                            alpha_carry=False, adj_ub=0.4, steps_per_adjust=100), "kT", [0.7, 1.0, 1.5], 3, 0),
    "cluster_carry1": (dict(n=100, E0=1.0, K2=0.1, Fz=0.5, energy_type="interacting", kappa=0.5, clustering=True,
                            alpha_carry=True, adj_ub=0.4, steps_per_adjust=100), "Fz", [0.2, 0.6, 1.2], 3, 0),
    # Ising through the lane / warp kernels
    "ising_lane": (dict(n=40, E0=1.0, Fz=0.3, energy_type="Ising", steps_per_adjust=100), "kT", [0.5, 0.8, 1.2, 2.0], 8, 0),
    # the 2-D tree
    "planar": (dict(n=40, E0=1.0, K2=0.2, Fz=0.5, energy_type="interacting", clustering=True, planar=True,
                    adj_ub=0.4, steps_per_adjust=100), "kT", [0.5, 0.9, 1.5], 3, 0),
}


def _ladder_cases(pm, O, base, kind, values):
    pcs, ocs = zip(*[both_cases(pm, O, **{**base, kind: v}) for v in values])
    return list(pcs), list(ocs)


@pytest.mark.parametrize("name", list(KERNEL_CASES))
def test_exchange_kernel_matches_the_restated_rule(pm, O, name):
    """10 rounds of run(200) + exchange(): every decision equals the host restatement's on the same inputs with ε from
    the shared Philox stream; accepted pairs swap records, Ω, Σu, r, p, Σψ, Σcos²θ and the re-expressed U, reset the
    carry; accumulators, step sizes, counters, cluster statistics and everything of rejected pairs stay bit for bit;
    exchange_stats equals the host's bookkeeping."""
    base, kind, values, R, hint = KERNEL_CASES[name]
    pcs, _ = _ladder_cases(pm, O, base, kind, values)
    clustering = bool(base.get("clustering"))
    seed = 4242
    with pm.Ensemble(pcs, replicas=R, seed=seed, ensemble_chains=hint) as ens:
        name_before = ens.kernel_name()
        if hint:
            assert name_before.startswith("k_run_cta_win"), name_before
        ladder = list(range(len(values)))
        ens.set_ladders([ladder])
        assert ens.kernel_name() == name_before
        book = TR.Exchange(len(values), R)
        book.set_ladders([ladder])
        if clustering:
            ens.begin_stage(1.0)
        taken = 0
        for _ in range(10):
            (ens.run_ex if clustering else ens.run)(200)
            pre = _snapshot(ens)
            acc = ens.exchange()
            taken += _check_round(ens, pcs, book, seed, 1.0, pre, _snapshot(ens), acc)
        assert taken > 0
        st = ens.exchange_stats()
        np.testing.assert_array_equal(st["attempts"], book.stats[:, 0])
        np.testing.assert_array_equal(st["accepts"], book.stats[:, 1])
        np.testing.assert_array_equal(st["walker"], book.walker)
        np.testing.assert_array_equal(st["round_trips"], book.trips)


@pytest.mark.parametrize("name", ["plain_kT_flips", "plain_Fz", "plain_n512", "ising_lane"])
def test_tempered_run_matches_the_oracle(pm, O, name):
    """The plain driver: run(200) + exchange() for 10 rounds against oracle Runs fed the library's Philox draws
    (tempering_ref.philox_tape) and exchanged by the restated rule: the same accepted flags every round, and at the
    end the same states, averages, acceptance counts, step sizes and exchange statistics (tolerances of
    test_gpu_round2._compare_run)."""
    base, kind, values, R, hint = KERNEL_CASES[name]
    pcs, ocs = _ladder_cases(pm, O, base, kind, values)
    seed, rounds, every = 97, 10, 200
    ladder = list(range(len(values)))
    ref = TR.Ladders(ocs, R, seed, chain_id_base=0, tape_steps=rounds * every)
    ref.set_ladders([ladder])
    with pm.Ensemble(pcs, replicas=R, seed=seed, ensemble_chains=hint) as ens:
        ens.set_ladders([ladder])
        for k in range(rounds):
            ens.run(every)
            for run in ref.runs:
                run.steps(every)
            np.testing.assert_array_equal(ens.exchange(), ref.exchange(), err_msg=f"round {k}")
        avg, ar, nrm = ens.averages()
        diag = ens.diagnostics()
        phi, th = ens.get_state_all()
        for c, run in enumerate(ref.runs):
            oavg, oar, onrm = run.averages()
            od = run.diag()
            assert diag[c, 4] == od["nacc_total"] and diag[c, 5] == od["steps_total"], c
            assert diag[c, 0] == pytest.approx(od["phi_step"], rel=1e-14)
            np.testing.assert_allclose(avg[c], oavg, rtol=1e-9, atol=1e-9 * max(1.0, np.abs(oavg).max()))
            assert nrm[c] == onrm and ar[c] == pytest.approx(oar, rel=1e-14)
            ophi, oth = run.chain().state()
            np.testing.assert_allclose(phi[c], ophi, rtol=0, atol=1e-12)
            np.testing.assert_allclose(th[c], oth, rtol=0, atol=1e-12)
        st = ens.exchange_stats()
        np.testing.assert_array_equal(st["attempts"], ref.stats[:, 0])
        np.testing.assert_array_equal(st["accepts"], ref.stats[:, 1])
        np.testing.assert_array_equal(st["walker"], ref.walker)
        np.testing.assert_array_equal(st["round_trips"], ref.trips)
        assert ref.stats[:, 1].sum() > 0


@pytest.mark.parametrize("name", ["plain_kT_flips", "cluster_carry1", "ising_lane"])
def test_run_tempering_is_the_explicit_loop(pm, O, name):
    """pmc_run_tempering / _ex (chunks on the device, rows placed there, one copy per output) equal
    run(E, stepout) + exchange() repeated, bit for bit: rows, averages, states, diagnostics, exchange statistics."""
    base, kind, values, R, hint = KERNEL_CASES[name]
    pcs, _ = _ladder_cases(pm, O, base, kind, values)
    clustering = bool(base.get("clustering"))
    ladder = [list(range(len(values)))]
    out = []
    for fused in (False, True):
        with pm.Ensemble(pcs, replicas=R, seed=11) as ens:
            ens.set_ladders(ladder)
            if clustering:
                ens.begin_stage(2.0)
                ens.run_tempering_ex(400, 200)                       # a burn-in stage, no rows
                ens.begin_stage(1.0)
            ens.run(100) if not clustering else ens.run_ex(100)      # step counter not at a chunk boundary
            if fused:
                rows = (ens.run_tempering_ex(1000, 200, 50, want_state=True) if clustering
                        else ens.run_tempering(1000, 200, 50))
            else:
                parts = []
                for _ in range(5):
                    parts.append(ens.run_ex(200, 50, want_state=True) if clustering else ens.run(200, 50))
                    ens.exchange()
                rows = tuple(np.concatenate([p[j] for p in parts], axis=1) for j in range(len(parts[0])))
            st = ens.exchange_stats()
            out.append((rows, ens.averages(), ens.get_state_all(), ens.diagnostics(), st,
                        ens.extra_averages() if clustering else None))
    (ra, aa, sa, da, xa, ea), (rb, ab, sb, db, xb, eb) = out
    assert rb[0].shape == (R * len(values), 1000 // 50, 8)
    for x, y in zip(ra, rb):
        assert _same(x, y)
    for x, y in zip(aa + sa + (da,), ab + sb + (db,)):
        assert _same(x, y)
    for k in xa:
        np.testing.assert_array_equal(xa[k], xb[k])
    if clustering:
        assert _same(ea, eb)
    assert xa["accepts"].sum() > 0


def test_ladders_without_exchange_change_nothing(pm, O):
    """A handle with ladders set but never exchanged runs bit-identically to one without, on the same kernel."""
    base, kind, values, R, _ = KERNEL_CASES["plain_kT_flips"]
    pcs, _ = _ladder_cases(pm, O, base, kind, values)
    out = []
    for ladders in (None, [[0, 1, 2, 3]]):
        with pm.Ensemble(pcs, replicas=R, seed=3) as ens:
            if ladders:
                ens.set_ladders(ladders)
            traj, roll = ens.run(600, 100)
            out.append((ens.kernel_name(), traj, roll, ens.averages(), ens.get_state_all(), ens.checkpoint()))
    a, b = out
    assert a[0] == b[0]
    for x, y in zip(a[1:3] + a[3] + a[4], b[1:3] + b[3] + b[4]):
        assert _same(x, y)
    assert b[5][:len(a[5])] == a[5]           # the same bytes, then the ladder block


def test_checkpoint_mid_tempering_resumes_bit_identically(pm, O):
    """Save during a tempered run, load into a fresh handle with the same ladders, continue: the same as the
    uninterrupted run; a ladder-less checkpoint keeps its size, and checkpoints and ladders must match."""
    base, kind, values, R, _ = KERNEL_CASES["cluster_carry1"]
    pcs, _ = _ladder_cases(pm, O, base, kind, values)
    ladder = [[0, 1, 2]]
    c, n = len(values) * R, int(base["n"])
    with pm.Ensemble(pcs, replicas=R, seed=21) as ens:
        plain_bytes = len(ens.checkpoint())
        assert plain_bytes == _HDR + c * n * _MONO.itemsize + c * (_DYN.itemsize + _DYNX.itemsize)
        ens.set_ladders(ladder)
        ens.begin_stage(1.0)
        ens.run_tempering_ex(600, 200)
        blob = ens.checkpoint()
        rows = ens.run_tempering_ex(600, 200, 100)
        want = (rows, ens.averages(), ens.get_state_all(), ens.exchange_stats())
    with pm.Ensemble(pcs, replicas=R, seed=21) as fresh:
        with pytest.raises(pm.PolymcError, match="ladders"):
            fresh.restore(blob)                                       # no ladders set
        fresh.set_ladders([[0, 2, 1]])
        with pytest.raises(pm.PolymcError, match="ladders differ"):
            fresh.restore(blob)
        fresh.set_ladders(ladder)
        fresh.restore(blob)
        rows = fresh.run_tempering_ex(600, 200, 100)
        got = (rows, fresh.averages(), fresh.get_state_all(), fresh.exchange_stats())
    assert want[0][2] is None and got[0][2] is None
    for x, y in zip(want[0][:2] + want[1] + want[2], got[0][:2] + got[1] + got[2]):
        assert _same(x, y)
    for k in want[3]:
        np.testing.assert_array_equal(want[3][k], got[3][k])


GPU_N, GPU_R = 8, 1024
GPU_BASE = dict(n=GPU_N, E0=1.0, K1=1.0, K2=0.0, Fz=0.5, energy_type="noninteracting", steps_per_adjust=100)
GPU_LADDERS = {"kT": [0.5, 0.8, 1.3, 2.0], "Fz": [0.0, 0.5, 1.2, 2.5]}


@pytest.mark.parametrize("kind", list(GPU_LADDERS))
def test_every_rung_samples_its_closed_form_ensemble_at_4096_chains(pm, kind):
    """The CPU tier's closed-form test on the GPU: 4 rungs × 1024 replicas of non-interacting n = 8 chains exchanging
    every 10 trials; the 16 averages of every rung within 3σ of the replica spread of the quadrature."""
    pcs = [pm.make_case(**{**GPU_BASE, kind: v}) for v in GPU_LADDERS[kind]]
    with pm.Ensemble(pcs, replicas=GPU_R, seed=808) as ens:
        assert ens.nchains == 4096
        ens.set_ladders([[0, 1, 2, 3]])
        ens.run_tempering(2000, 10)
        ens.begin_stage(1.0)
        ens.run_tempering(40000, 10)
        avg = ens.averages()[0]
        st = ens.exchange_stats()
    for k, v in enumerate(GPU_LADDERS[kind]):
        kw = {key: GPU_BASE[key] for key in ("E0", "K1", "K2", "Fz")}
        kw[kind] = v
        cf = CF.chain_averages(GPU_N, **kw)
        rung = avg[k * GPU_R:(k + 1) * GPU_R]
        z = np.abs(rung.mean(0) - cf) / (rung.std(0, ddof=1) / math.sqrt(GPU_R))
        assert np.all(z <= 3.0), (kind, v, np.round(z, 2))
    rate = st["accepts"][:3] / st["attempts"][:3]
    assert np.all((rate > 0.05) & (rate < 0.99)), rate


def test_walker_labels_are_a_permutation_and_round_trips_follow_them(pm, O):
    """After every round the labels of each ladder column are a permutation of its initial ids, and the round trips
    recomputed from the label history recorded on the host equal the library's."""
    base, kind, values, R, _ = KERNEL_CASES["ising_lane"]
    pcs, _ = _ladder_cases(pm, O, base, kind, values)
    m = len(values)
    with pm.Ensemble(pcs, replicas=R, seed=31, chain_id_base=500) as ens:
        ens.set_ladders([list(range(m))])
        hist = []
        for _ in range(200):
            ens.run(20)
            ens.exchange()
            w = ens.exchange_stats()["walker"]
            hist.append(w)
            for r in range(R):
                assert sorted(w[[k * R + r for k in range(m)]]) == [500 + k * R + r for k in range(m)]
        trips = ens.exchange_stats()["round_trips"]
    state = np.where(np.arange(m * R) < R, 1, 0)
    want = np.zeros(m * R, np.int64)
    for w in hist:
        for slot, lab in enumerate(w):
            i = lab - 500
            if slot < R:
                want[i] += state[i] == 2
                state[i] = 1
            elif slot >= (m - 1) * R and state[i] == 1:
                state[i] = 2
    np.testing.assert_array_equal(trips, want)
    assert want.sum() > 0


def test_refusals_through_the_c_abi(pm, O):
    """What cannot be tempered is refused with PMC_ERR_INVALID and a message in pmc_last_error."""
    base = dict(n=32, E0=1.0, K2=0.1, energy_type="interacting")
    cases = [pm.make_case(**base, kT=1.0), pm.make_case(**base, kT=2.0), pm.make_case(**{**base, "E0": 2.0}, kT=3.0),
             pm.make_case(**base, kT=4.0, umbrella=True)]
    with pm.Ensemble(cases, replicas=2, seed=1) as ens:
        for ladders, msg in (([[0, 5]], "not a case index"), ([[0, 1], [1, 3]], "more than once"),
                             ([[0]], "at least two rungs"), ([[0, 2]], "must agree on E0"),
                             ([[0, 3]], "umbrella"), ([[0, 1, 0]], "more than once")):
            with pytest.raises(pm.PolymcError, match=msg) as ei:
                ens.set_ladders(ladders)
            assert ei.value.code == -1
            assert msg in pm.load().pmc_last_error().decode()
        with pytest.raises(pm.PolymcError, match="no ladders"):
            ens.exchange()
        with pytest.raises(pm.PolymcError, match="no ladders"):
            ens.run_tempering(200, 100)
        ens.set_ladders([[0, 1]])
        with pytest.raises(pm.PolymcError, match="exchange_every must divide"):
            ens.run_tempering(250, 100)
        with pytest.raises(pm.PolymcError, match="stepout must divide"):
            ens.run_tempering(200, 100, 30)
        with pytest.raises(pm.PolymcError, match="clustering-driver"):
            ens.run_tempering_ex(200, 100)
        ens.set_ladders([])                                   # cleared: a plain handle again
        with pytest.raises(pm.PolymcError, match="no ladders"):
            ens.exchange()
    cut = dict(n=32, E0=1.0, energy_type="cutoff", cutoff_radius=3.0, clustering=True)
    with pm.Ensemble([pm.make_case(**cut, Fz=0.0), pm.make_case(**cut, Fz=1.0)], replicas=2, seed=1) as ens:
        with pytest.raises(pm.PolymcError, match="force ladder needs F in the energy"):
            ens.set_ladders([[0, 1]])
    with pm.Ensemble([pm.make_case(**cut, Fz=0.0, cutoff_full=True), pm.make_case(**cut, Fz=1.0, cutoff_full=True)],
                     replicas=2, seed=1) as ens:
        ens.set_ladders([[0, 1]])
        ens.begin_stage(1.0)
        ens.run_tempering_ex(200, 100)


def test_tempered_sweep_runs_every_stage_tempered(pm, tmp_path):
    """polymc.sweep with temper: the ladders of the grid, every burn-in stage and the production run tempered — the
    same numbers as driving one handle by hand — and run_sweep.py --temper writes the usual table (a row per rung)
    and the exchange table."""
    import os
    import subprocess
    import sys
    from polymc import mcmc_clustering, sweep
    common = ["--energy-type", "Ising", "--bend-mod", "0.5", "-n", "30", "--num-steps", "3000", "--burn-in", "300",
              "--burn-schedule", "[10; 1]", "-v", "0"]
    pl = [mcmc_clustering.parse_args(common + ["--kT", k, "--E0", e]) for e in ("0.5", "1") for k in ("2", "0.5", "1")]
    cases = [mcmc_clustering.case_from_pargs(p) for p in pl]
    proto = dict(burn_in=300, schedule=[10.0, 1.0])
    res = sweep.run_sweep(cases, 2, 3000, seed=11, protocol=proto, temper="kT", exchange_every=100)
    assert res["exchange"]["ladders"] == [[1, 2, 0], [4, 5, 3]]
    with pm.Ensemble(cases, replicas=2, seed=11) as ens:
        ens.set_ladders([[1, 2, 0], [4, 5, 3]])
        for mult in (10.0, 1.0):
            ens.begin_stage(mult)
            ens.run_tempering_ex(300, 100)
        ens.begin_stage(1.0)
        ens.run_tempering_ex(3000, 100)
        np.testing.assert_array_equal(res["avg"], ens.averages()[0])
        st = ens.exchange_stats()
    np.testing.assert_array_equal(res["exchange"]["attempts"], st["attempts"])
    np.testing.assert_array_equal(res["exchange"]["accepts"], st["accepts"])
    assert st["accepts"].sum() > 0
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out, xout = tmp_path / "study.csv", tmp_path / "exchange.csv"
    argv = [sys.executable, os.path.join(root, "polymer-stats_b200", "run_sweep.py"), "--driver", "clustering",
            "--out", str(out), "--exchange-out", str(xout), "--runs", "2", "--seed", "11", "--temper", "kT",
            "--grid", "E0=0.5,1", "--grid", "kT=2,0.5,1", "--"] + common
    r = subprocess.run(argv, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    assert len(open(out).read().strip().split("\n")) == 1 + 12
    lines = open(xout).read().strip().split("\n")
    assert lines[0] == "E0,kT_lo,kT_hi,attempts,accepts,rate,round_trips"
    assert [ln.split(",")[:3] for ln in lines[1:]] == [["0.5", "0.5", "1.0"], ["0.5", "1.0", "2.0"],
                                                       ["1.0", "0.5", "1.0"], ["1.0", "1.0", "2.0"]]
    assert all(int(ln.split(",")[3]) > 0 for ln in lines[1:])
