"""Replica exchange across kT and force ladders, CPU tier: the exchange rule restated on the oracle's runs
(tests/tempering_ref.py) samples every rung's closed-form ensemble, its swap rates match E[min(1, e^Δ)] estimated
from runs without exchange, and the sweep layer builds ladders, refuses what cannot be tempered and writes the
exchange table."""
import math

import numpy as np
import pytest

import closed_form as CF
import tempering_ref as TR

N, R = 8, 64
BASE = dict(n=N, E0=1.0, K1=1.0, K2=0.0, Fz=0.5, energy_type="noninteracting", steps_per_adjust=100)
LADDERS = {"kT": [0.5, 0.8, 1.3, 2.0], "Fz": [0.0, 0.5, 1.2, 2.5]}
# Exchange rounds come every 10 trials, about one update per monomer, so that a wrong exchange rule would leave its
# mark on the rungs' ensembles before the trials in between relax it away.
BURN, ROUNDS, EVERY = 100, 1000, 10


def _cases(O, kind):
    return [O.make_case(**{**BASE, kind: v}) for v in LADDERS[kind]]


@pytest.fixture(scope="module")
def tempered(O):
    """Per ladder kind: the averages of every chain and the per-round accepted flags of a tempered run."""
    out = {}
    for kind in LADDERS:
        T = TR.Ladders(_cases(O, kind), R, seed=2026, tape_steps=(BURN + ROUNDS) * EVERY,
                       rng=np.random.default_rng(2026))
        T.set_ladders([list(range(len(LADDERS[kind])))])
        for _ in range(BURN):
            for run in T.runs:
                run.steps(EVERY)
            T.exchange()
        T.begin_stage(1.0)           # forget the burn-in: fresh averagers, step sizes and stream tag
        flags = []
        for _ in range(ROUNDS):
            for run in T.runs:
                run.steps(EVERY)
            flags.append(T.exchange())
        avg = np.array([run.averages()[0] for run in T.runs])
        out[kind] = (T, avg, np.array(flags))
    return out


@pytest.mark.parametrize("kind", list(LADDERS))
def test_every_rung_samples_its_closed_form_ensemble(tempered, kind):
    """Non-interacting chains: the 16 averages of every rung agree with the single-monomer quadrature within 3σ of
    the spread over the 64 replicas, on a kT ladder and on a force ladder."""
    T, avg, flags = tempered[kind]
    assert flags.sum() > 0
    for k, v in enumerate(LADDERS[kind]):
        kw = {key: BASE[key] for key in ("E0", "K1", "K2", "Fz")}
        kw[kind] = v
        cf = CF.chain_averages(N, **kw)
        rung = avg[k * R:(k + 1) * R]
        mean, sem = rung.mean(axis=0), rung.std(axis=0, ddof=1) / math.sqrt(R)
        z = np.abs(mean - cf) / np.maximum(sem, 1e-12)
        assert np.all(z <= 3.0), (kind, v, np.round(z, 2))


def _log_ratio(ca, cb, Ua, ra, Ub, rb):
    """log π_a(x_b) + log π_b(x_a) − log π_a(x_a) − log π_b(x_b) for π_s(x) ∝ exp(−(U₀(x) − r(x)·F_s)/kT_s)·Ω(x),
    from the energies U_s each configuration has at its own rung (U₀ = U_s + r·F_s): the definition, written
    independently of the library's form of Δ."""
    U0a, U0b = Ua + ra[0] * ca.Fx + ra[2] * ca.Fz, Ub + rb[0] * cb.Fx + rb[2] * cb.Fz

    def U(c, U0, r):
        return U0 - (r[0] * c.Fx + r[2] * c.Fz)
    return (-U(ca, U0b, rb) / ca.kT - U(cb, U0a, ra) / cb.kT) - (-U(ca, U0a, ra) / ca.kT - U(cb, U0b, rb) / cb.kT)


def _pair_rate_expectation(O, kind, k):
    """E[min(1, e^Δ)] for rungs k, k+1 from configurations sampled at each rung by runs WITHOUT exchange, per
    replica column (mean and its standard error over columns)."""
    cases = _cases(O, kind)
    cols = []
    for r in range(R):
        # one steps() call per run (each call restarts the oracle's stream); a trajectory row (step, r, p, U) every
        # 100 trials, the first BURN·EVERY trials discarded
        total = (BURN + ROUNDS) * EVERY
        lo, _ = O.Run(cases[k], 99, 10_000 + r, 1).steps(total, 100)
        hi, _ = O.Run(cases[k + 1], 99, 20_000 + r, 1).steps(total, 100)
        keep = slice(BURN * EVERY // 100, None)
        d = [_log_ratio(cases[k], cases[k + 1], a[7], a[1:4], b[7], b[1:4]) for a, b in zip(lo[keep], hi[keep])]
        cols.append(np.mean(np.exp(np.minimum(d, 0.0))))
    cols = np.array(cols)
    return cols.mean(), cols.std(ddof=1) / math.sqrt(R)


@pytest.mark.parametrize("kind", list(LADDERS))
def test_swap_rate_matches_the_exchange_acceptance(O, tempered, kind):
    """The measured swap rate of every rung pair agrees within 3σ with E[min(1, e^Δ)] over independent samples of
    the two rungs; the counters of the diagnostics are the attempts and accepts the rounds made."""
    T, _, flags = tempered[kind]
    for k in range(len(LADDERS[kind]) - 1):
        rounds = flags[(np.arange(ROUNDS) + BURN) % 2 == k % 2]           # the rounds that attempt this pair
        per_col = rounds[:, k * R:(k + 1) * R].mean(axis=0)
        meas, meas_se = per_col.mean(), per_col.std(ddof=1) / math.sqrt(R)
        want, want_se = _pair_rate_expectation(O, kind, k)
        assert abs(meas - want) <= 3 * math.hypot(meas_se, want_se), (kind, k, meas, want, meas_se, want_se)
        assert 0.02 < want < 0.98, (kind, k, want)   # the ladder is neither trivial nor frozen
    assert T.stats[:, 0].sum() == sum(len(T.pairs[r & 1]) for r in range(T.round))


def test_walker_labels_stay_a_permutation_and_round_trips_follow_them(O):
    """Labels within one replica column are a permutation of the column's initial ids after every round; round
    trips recomputed from the recorded label history equal the counters."""
    cases = [O.make_case(**{**BASE, "kT": v}) for v in (0.6, 0.9, 1.4)]
    T = TR.Ladders(cases, 4, seed=5, chain_id_base=100, tape_steps=120 * 20, rng=np.random.default_rng(5))
    T.set_ladders([[0, 1, 2]])
    hist = [T.walker.copy()]
    for _ in range(120):
        for run in T.runs:
            run.steps(20)
        T.exchange()
        hist.append(T.walker.copy())
        for r in range(4):
            col = T.walker[[r, 4 + r, 8 + r]]
            assert sorted(col) == [100 + r, 104 + r, 108 + r]
    hist = np.array(hist)
    trips = np.zeros(12, dtype=np.int64)
    for w in range(12):
        state = 1 if w < 4 else 0
        for row in hist[1:]:
            slot = int(np.flatnonzero(row == 100 + w)[0])
            if slot < 4:
                trips[w] += state == 2
                state = 1
            elif slot >= 8 and state == 1:
                state = 2
    np.testing.assert_array_equal(trips, T.trips)
    assert trips.sum() > 0


@pytest.mark.parametrize("kw", [
    dict(n=64, energy_type="interacting", do_flips=True, E0=1.0, K2=0.1, Fz=0.5, Fx=0.2),
    dict(n=40, energy_type="Ising", E0=1.0, Fz=0.3),
])
def test_philox_tape_continues_the_librarys_stream(O, kw):
    """The oracle restarts the Philox stream at trial 1 on every steps() call; a run fed from philox_tape continues
    it across calls, as the library does: three chunks of 200 trials make the decisions of one 600-trial run."""
    c = O.make_case(steps_per_adjust=100, **kw)
    ref = O.Run(c, 77, 5, 1)
    ref.steps(600)
    run = O.Run(c, 77, 5, 1, tape=TR.philox_tape(c, 77, 5, 0, 0, 600))
    run.set_state(*O.draw_init(77, 5, 0, int(c.n)))
    for _ in range(3):
        run.steps(200)
    assert run.diag() == ref.diag()
    np.testing.assert_array_equal(run.averages()[0], ref.averages()[0])
    np.testing.assert_array_equal(run.chain().state()[0], ref.chain().state()[0])


# ---- host logic of the sweep layer (no device needed) --------------------------------------------------------------

def _pargs(argv):
    from polymc import mcmc
    return mcmc.parse_args(argv)


def test_ladders_from_a_sweep_grid(pm):
    from polymc import mcmc, sweep
    pl = [_pargs(["-n", "8", "--E0", e, "--kT", k, "--Fz", f]) for e in ("0.1", "1") for k in ("2", "0.5", "1")
          for f in ("0", "1")]
    cases = [mcmc.case_from_pargs(p) for p in pl]
    lad = sweep.tempering_ladders(cases, "kT")
    assert len(lad) == 4 and all(len(x) == 3 for x in lad)
    for x in lad:
        kts = [pl[c]["kT"] for c in x]
        assert kts == sorted(kts)
        assert len({(pl[c]["E0"], pl[c]["Fz"]) for c in x}) == 1
    assert sorted(c for x in lad for c in x) == list(range(len(pl)))
    assert sweep.tempering_ladders(pm.CaseTable(cases), "kT") == lad
    fz = sweep.tempering_ladders(cases, "Fz")
    assert len(fz) == 6 and all([pl[c]["Fz"] for c in x] == [0.0, 1.0] for x in fz)


@pytest.mark.parametrize("grid,temper,msg", [
    ([["--kT", "1"], ["--kT", "2"], ["--kT", "3", "--E0", "2"]], "kT", "at least two rungs"),   # a field differs
    ([["--kT", "1"]], "kT", "at least two rungs"),                                              # one rung
    ([["--kT", "1"], ["--kT", "1"]], "kT", "repeat a value"),                                   # repeated case
    ([["--kT", "1", "-B"], ["--kT", "2", "-B"]], "kT", "umbrella"),
    ([["--kT", "1"], ["--kT", "2"]], "E0", "temper must be one of"),
])
def test_sweep_refuses_what_cannot_be_tempered(pm, grid, temper, msg):
    from polymc import mcmc, sweep
    cases = [mcmc.case_from_pargs(_pargs(["-n", "8"] + g)) for g in grid]
    with pytest.raises(pm.PolymcError, match=msg):
        sweep.tempering_ladders(cases, temper)


def test_temper_needs_one_rank(pm):
    from polymc import mcmc, sweep
    cases = [mcmc.case_from_pargs(_pargs(["-n", "8", "--kT", k])) for k in ("1", "2")]
    with pytest.raises(pm.PolymcError, match="single rank"):
        sweep.run_shard(cases, 2, 100, rank=0, world=2, temper="kT")
    with pytest.raises(pm.PolymcError, match="must divide"):
        sweep.run_shard(cases, 2, 150, temper="kT", exchange_every=100)


def test_run_sweep_cli_refuses_temper_under_several_ranks(monkeypatch, tmp_path):
    import run_sweep
    monkeypatch.setenv("WORLD_SIZE", "2")
    with pytest.raises(SystemExit):
        run_sweep.main(["--out", str(tmp_path / "t.csv"), "--temper", "kT", "--grid", "kT=1,2", "--", "-n", "8"])
    monkeypatch.setenv("WORLD_SIZE", "1")
    with pytest.raises(SystemExit):   # --exchange-out without --temper
        run_sweep.main(["--out", str(tmp_path / "t.csv"), "--exchange-out", str(tmp_path / "x.csv"), "--", "-n", "8"])


def test_exchange_csv_format(tmp_path):
    from polymc import sweep
    pl = [_pargs(["-n", "8", "--E0", e, "--kT", k]) for e in ("0.1", "1") for k in ("0.5", "1", "2")]
    ex = {"ladders": [[0, 1, 2], [3, 4, 5]], "attempts": np.array([10, 8, 0, 6, 4, 0]),
          "accepts": np.array([5, 2, 0, 3, 1, 0]), "round_trips": np.array([3, 0])}
    header, rows = sweep.exchange_rows(pl, "kT", ex, fixed=["E0"])
    assert header == ["E0", "kT_lo", "kT_hi", "attempts", "accepts", "rate", "round_trips"]
    path = tmp_path / "x.csv"
    sweep.write_exchange_csv(str(path), header, rows)
    assert path.read_text().splitlines() == [
        "E0,kT_lo,kT_hi,attempts,accepts,rate,round_trips",
        "0.1,0.5,1.0,10,5,0.5,3",
        "0.1,1.0,2.0,8,2,0.25,3",
        "1.0,0.5,1.0,6,3,0.5,0",
        "1.0,1.0,2.0,4,1,0.25,0",
    ]
