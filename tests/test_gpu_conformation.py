"""Conformation sampling on the GPU (pmc_set_conformation, pmc_sample_conformation, pmc_run_sampled*,
pmc_conformation_sums): the kernel against the numpy restatement (tests/conformation_ref.py) on every kind of handle,
the fused driver against the explicit loop, the run kernels left alone, the closed forms of non-interacting chains at
4096 chains, the life cycle, checkpoints, refusals and the sweep's CSVs.
"""
import csv
import os

import numpy as np
import pytest

import closed_form as CF
import conformation_ref as CR

pytestmark = pytest.mark.gpu

_HDR = 72   # pmc_checkpoint_save: CkptHeader, then the records (chain_math.cuh MonoRec)
_MONO = np.dtype([("phi", "f8"), ("theta", "f8"), ("nx", "f8"), ("ny", "f8"), ("nz", "f8"), ("sth", "f8")])


def _records(ens):
    """n̂ [chains][n][3] exactly as the device holds it."""
    blob = ens.checkpoint()
    m = np.frombuffer(blob, _MONO, ens.nchains * ens.n, _HDR).reshape(ens.nchains, ens.n)
    return np.stack([m["nx"], m["ny"], m["nz"]], axis=-1)


def _bits(x):
    return np.ascontiguousarray(x, dtype=np.float64).view(np.uint64)


def _random_state(ens, rng, planar=False):
    phi = rng.uniform(0, 2 * np.pi, (ens.nchains, ens.n))
    theta = np.full((ens.nchains, ens.n), np.pi / 2) if planar else np.arccos(rng.uniform(-1, 1, (ens.nchains, ens.n)))
    ens.set_state_all(phi, theta)


def _max_n(pm):
    lo, hi = 4000, 4200
    while hi - lo > 1:
        mid = (lo + hi) // 2
        try:
            pm.Ensemble(pm.make_case(n=mid), replicas=1).close()
            lo = mid
        except pm.PolymcError:
            hi = mid
    return lo


HANDLES = {
    "plain_n2": dict(n=2),
    "plain_n8": dict(n=8, E0=1.0, Fz=0.5),
    "interacting_n100": dict(n=100, E0=1.0, energy_type="interacting"),
    "headline_n512": dict(n=512, E0=1.0, K1=1.0, Fz=0.5, energy_type="interacting"),
    "clustering_n100": dict(n=100, E0=1.0, energy_type="interacting", kappa=0.5, clustering=True),
    "ising_n100": dict(n=100, E0=1.0, energy_type="Ising"),
    "cutoff_n100": dict(n=100, E0=1.0, energy_type="cutoff", cutoff_radius=3.0),
    "planar_n100": dict(n=100, E0=1.0, clustering=True, planar=True),
    "max_n": None,
}


@pytest.mark.parametrize("name", list(HANDLES))
def test_kernel_matches_restatement(pm, name):
    kw = HANDLES[name] if HANDLES[name] is not None else dict(n=_max_n(pm), b=0.7)
    planar = bool(kw.get("planar"))
    reps = 2 if name == "max_n" else 6
    hint = 4096 if name == "headline_n512" else 0
    B = 37
    rng = np.random.default_rng(7)
    sums = []
    for trial in range(2):            # two identical handles: identical bits
        with pm.Ensemble(pm.make_case(**kw), replicas=reps, seed=11, ensemble_chains=hint) as ens:
            ens.set_conformation(B)
            assert ens.conformation_cols() == 8 + 3 * ens.n + B
            ref = [CR.Sums(ens.n, B) for _ in range(ens.nchains)]
            rng = np.random.default_rng(7)
            for k in range(3):
                if k != 2:            # the third sample repeats the second configuration
                    _random_state(ens, rng, planar)
                nh = _records(ens)
                b = kw.get("b", 1.0)
                for c in range(ens.nchains):
                    ref[c].add(nh[c], b, rz=ens.observables(c)[0][2])
                ens.sample_conformation()
            got = ens.conformation_sums()
            n = ens.n
            for c in range(ens.nchains):
                want, mag = ref[c].row, ref[c].mag
                assert got[c, 0] == 3.0
                np.testing.assert_array_equal(_bits(got[c, 8 + n:]), _bits(want[8 + n:]))   # profile + histogram
                err = np.abs(got[c, 1:8 + n] - want[1:8 + n])
                assert np.all(err <= 1e-12 * np.maximum(mag[1:8 + n], 1e-300)), (name, c, np.argmax(err / mag[1:8 + n]))
            sums.append(got)
    np.testing.assert_array_equal(_bits(sums[0]), _bits(sums[1]))


def _same_run(pm, kw, fused, explicit, reps=8, ladder=None, hint=0):
    outs = []
    for drive in (fused, explicit):
        with pm.Ensemble([pm.make_case(**k) for k in kw], replicas=reps, seed=5, ensemble_chains=hint) as ens:
            if ladder:
                ens.set_ladders(ladder)
            ens.set_conformation(16)
            rows = drive(ens)
            o = [ens.conformation_sums(), *ens.averages(), ens.diagnostics(), ens.accumulators(), *ens.get_state_all()]
            outs.append((o, rows))
    (a, ra), (b, rb) = outs
    for x, y in zip(a, b):
        np.testing.assert_array_equal(_bits(x), _bits(y))
    for x, y in zip(ra, rb):
        np.testing.assert_array_equal(_bits(x), _bits(y))


def _loop(ens, N, K, so, run, extra=()):
    rows = []
    for _ in range(N // K):
        rows.append(run(ens, K, so))
        for f in extra:
            f(ens)
        ens.sample_conformation()
    return [np.concatenate([r[j] for r in rows], axis=1) for j in range(len(rows[0]))]


@pytest.mark.parametrize("kind", ["plain", "headline", "clustering"])
def test_run_sampled_equals_explicit_loop(pm, kind):
    N, K, so = 600, 100, 50
    if kind == "clustering":
        kw = [dict(n=64, E0=1.0, energy_type="interacting", kappa=0.5, clustering=True, adj_ub=0.4)]
        _same_run(pm, kw, lambda e: e.run_sampled_ex(N, K, so, want_state=True),
                  lambda e: _loop(e, N, K, so, lambda e, k, s: e.run_ex(k, s, want_state=True)))
        return
    kw = [dict(n=512, E0=1.0, Fz=0.5, energy_type="interacting")] if kind == "headline" else [dict(n=40, E0=1.0, Fz=0.5)]
    _same_run(pm, kw, lambda e: e.run_sampled(N, K, so), lambda e: _loop(e, N, K, so, lambda e, k, s: e.run(k, s)),
              hint=4096 if kind == "headline" else 0)


def test_tempering_with_sampling_equals_explicit_loop(pm):
    N, K, so = 600, 100, 100
    kw = [dict(n=40, E0=1.0, Fz=0.5, kT=t) for t in (1.0, 1.3, 1.7)]
    _same_run(pm, kw, lambda e: e.run_tempering(N, K, so),
              lambda e: _loop(e, N, K, so, lambda e, k, s: e.run(k, s), extra=[lambda e: e.exchange()]),
              ladder=[[0, 1, 2]])


def test_run_kernels_untouched_and_checkpoint_format(pm):
    kw = dict(n=100, E0=1.0, Fz=0.5, energy_type="interacting")
    outs, blobs = [], []
    for on in (False, True):
        with pm.Ensemble(pm.make_case(**kw), replicas=8, seed=3) as ens:
            if on:
                ens.set_conformation(8)
            t, r = ens.run(500, 100)
            if on:
                ens.set_conformation(enable=False)
            assert ens.conformation_cols() == 0
            blobs.append(ens.checkpoint())
            outs.append([t, r, *ens.averages(), ens.diagnostics(), *ens.get_state_all()])
    for x, y in zip(*outs):
        np.testing.assert_array_equal(_bits(x), _bits(y))
    assert blobs[0] == blobs[1]


def _sampled_avgs(pm, case_kw, chains, nsteps, every, burn, bins):
    with pm.Ensemble(pm.make_case(**case_kw), replicas=chains, seed=20261022) as ens:
        ens.run(burn, 0, fetch_rows=False)
        ens.set_conformation(bins)
        ens.run_sampled(nsteps, every, 0, fetch_rows=False)
        return ens.conformation()


def _z(per_chain, want):
    per_chain = np.asarray(per_chain)
    return (per_chain.mean(axis=0) - want) / (per_chain.std(axis=0, ddof=1) / np.sqrt(per_chain.shape[0]))


CLOSED = {"field_force": dict(E0=1.0, K1=1.0, K2=0.0, Fz=0.6), "free": dict(E0=0.0, Fz=0.0)}


@pytest.mark.parametrize("which", list(CLOSED))
def test_closed_forms_at_scale(pm, which):
    """4096 non-interacting dielectric chains of n = 100 from the library's own random start, 20 000 trials of burn-in,
    then 20 000 trials sampled every 100: every closed form within 3σ of the spread across chains (the profile, 100
    numbers per column, within 4.5σ per monomer and 3σ on its mean).  ⟨n̂z²⟩ and the second moment of ζ see the
    single-bond density itself.  After only 2 000 trials of burn-in the field-and-force chains are still relaxing
    towards the field (⟨n̂z⟩ 10σ low, measured), hence the longer burn-in."""
    n, bins = 100, 200
    kw = dict(n=n, energy_type="noninteracting", chain_type="dielectric", **CLOSED[which])
    mom = CF.single_monomer_moments(**{k: v for k, v in kw.items() if k not in ("n", "energy_type")})
    m, mzz = mom["n"], mom["n2"][2]
    m2 = float(m @ m)
    k = np.arange(1, n)
    rg2 = float(((n - k) * ((k - 0.5) + (k * k - k + 0.5) * m2)).sum()) / n ** 2
    a = _sampled_avgs(pm, kw, 4096, 20000, 100, 20000, bins)
    assert np.all(a["samples"] == 200)
    zs = {"Rg2": float(_z(a["Rg2"], rg2))}
    for s in (1, 2, 10, 50):
        zs[f"C{s}"] = float(_z(a["bondcorr"][:, s], m2))
    zs["C0"] = float(np.max(np.abs(a["bondcorr"][:, 0] - 1.0)) / 1e-14)
    zn, zn2 = _z(a["nz"], m[2]), _z(a["nz2"], mzz)
    zs["nz_mean"] = float(_z(a["nz"].mean(axis=1), m[2]))
    zs["nz2_mean"] = float(_z(a["nz2"].mean(axis=1), mzz))
    centre = -1 + (np.arange(bins) + 0.5) * (2.0 / bins)
    mean = a["hist"] @ centre
    var = a["hist"] @ centre ** 2 - (2.0 / bins) ** 2 / 12   # Sheppard's correction of binned second moments
    zs["zeta_mean"] = float(_z(mean, m[2]))
    zs["zeta_msq"] = float(_z(var, (mzz - m[2] ** 2) / n + m[2] ** 2))
    print(which, {k: round(v, 2) for k, v in zs.items()}, "max |z| of the profile:", np.max(np.abs(zn)), np.max(np.abs(zn2)))
    assert all(abs(v) < 3 for v in zs.values()), zs
    assert np.max(np.abs(zn)) < 4.5 and np.max(np.abs(zn2)) < 4.5, (np.max(np.abs(zn)), np.max(np.abs(zn2)))


def test_life_cycle(pm):
    kw = [dict(n=30, E0=1.0, Fz=0.5, kT=t, energy_type="interacting") for t in (1.0, 1.5)]
    with pm.Ensemble([pm.make_case(**k) for k in kw], replicas=4, seed=9) as ens:
        ens.set_ladders([[0, 1]])
        ens.set_conformation(10)
        ens.run_sampled(300, 100)
        s0 = ens.conformation_sums()
        assert np.all(s0[:, 0] == 3)
        ens.reinit()
        np.testing.assert_array_equal(_bits(ens.conformation_sums()), _bits(s0))
        for _ in range(4):
            ens.exchange()
            np.testing.assert_array_equal(_bits(ens.conformation_sums()), _bits(s0))
        ens.begin_stage(1.0)
        assert np.all(ens.conformation_sums() == 0)
        ens.run_tempering(200, 100)
        # checkpoint / resume mid-run continues bit-identically
        blob = ens.checkpoint()
        ens.run_tempering(300, 100)
        want = ens.conformation_sums()
    with pm.Ensemble([pm.make_case(**k) for k in kw], replicas=4, seed=9) as ens2:
        ens2.set_ladders([[0, 1]])
        with pytest.raises(pm.PolymcError, match="conformation"):
            ens2.restore(blob)                      # no sampling here
        ens2.set_conformation(11)
        with pytest.raises(pm.PolymcError, match="conformation setting differs"):
            ens2.restore(blob)
        ens2.set_conformation(10)
        ens2.restore(blob)
        ens2.run_tempering(300, 100)
        np.testing.assert_array_equal(_bits(ens2.conformation_sums()), _bits(want))
    with pm.Ensemble([pm.make_case(**k) for k in kw], replicas=4, seed=9) as ens3:
        ens3.set_ladders([[0, 1]])
        ens3.run_tempering(200, 100)
        plain = ens3.checkpoint()
        ens3.set_conformation(10)
        with pytest.raises(pm.PolymcError, match="no conformation sums"):
            ens3.restore(plain)


def test_refusals(pm):
    with pm.Ensemble(pm.make_case(n=20, E0=1.0), replicas=2) as ens:
        for call in (ens.sample_conformation, ens.conformation_sums, lambda: ens.run_sampled(100, 10)):
            with pytest.raises(pm.PolymcError, match="not enabled"):
                call()
        L = pm.lib.load()
        for bins in (-1, 65537):
            with pytest.raises(pm.PolymcError, match="hist_bins"):
                ens.set_conformation(bins)
        ens.set_conformation(65536)
        assert ens.conformation_cols() == 8 + 60 + 65536
        ens.set_conformation(0)
        assert ens.conformation_cols() == 8 + 60
        with pytest.raises(pm.PolymcError, match="sample_every must divide nsteps"):
            pm.lib._check(L.pmc_run_sampled(ens._h, 100, 30, 0, None, None))
        with pytest.raises(pm.PolymcError, match="stepout must divide sample_every"):
            pm.lib._check(L.pmc_run_sampled(ens._h, 100, 50, 30, None, None))
        with pytest.raises(pm.PolymcError, match="clustering-driver"):
            ens.run_sampled_ex(100, 50)
        with pytest.raises(pm.PolymcError, match="no ladders"):
            ens.run_tempering(100, 50)
    with pm.Ensemble([pm.make_case(n=20), pm.make_case(n=20, umbrella=True)], replicas=2) as ens:
        with pytest.raises(pm.PolymcError, match="umbrella"):
            ens.set_conformation(4)
        assert ens.conformation_cols() == 0


def _read_csv(path):
    with open(path) as f:
        r = list(csv.reader(f))
    return r[0], r[1:]


def test_sweep_writes_pooled_conformation(pm, tmp_path):
    """run_sweep.py --conformation-* writes the four CSVs, and their values equal the pooled Ensemble.conformation()
    averages of the same chains.  The study table keeps its format and its chains, but by choice it is not bit-identical
    to the unsampled sweep's: run_sampled(N, K) is bit-identical to run(K); sample_conformation() repeated, and every
    run(K) starts with the re-synchronisation of the running U, r and p that run(N) does once, which moves the last bits
    of the r, p and U averages.  The table is held to 1e-9 of the unsampled one instead."""
    import run_sweep
    from polymc import sweep as SW
    common = ["--", "-n", "12", "--num-steps", "1000", "--E0", "1.0", "--energy-type", "interacting"]
    grid = ["--grid", "Fz=0,0.5", "--grid", "kT=1,2"]
    base = [*grid, "--runs", "3", "--seed", "4"]
    out0, out1 = str(tmp_path / "plain.csv"), str(tmp_path / "sampled.csv")
    assert run_sweep.main(["--out", out0, *base, *common]) == 0
    pre = str(tmp_path / "conf")
    assert run_sweep.main(["--out", out1, *base, "--conformation-every", "100", "--conformation-bins", "8",
                           "--conformation-out", pre, *common]) == 0
    h0, r0 = _read_csv(out0)
    h1, r1 = _read_csv(out1)
    assert h0 == h1 and len(r0) == len(r1)
    for x, y in zip(r0, r1):   # same chains; the per-chunk re-synchronisation moves the running scalars' last bits only
        for a, b in zip(x, y):
            try:
                assert abs(float(a) - float(b)) <= 1e-9 * max(1.0, abs(float(a)))
            except ValueError:
                assert a == b
    # the pooled averages of the same chains, from the Python API
    from polymc import mcmc
    pargs = [mcmc.parse_args(common[1:] + ["--Fz", fz, "--kT", kt]) for fz in ("0", "0.5") for kt in ("1", "2")]
    cases = [mcmc.case_from_pargs(p) for p in pargs]
    with pm.Ensemble(cases, replicas=3, seed=4) as ens:
        ens.set_conformation(8)
        ens.run_sampled(1000, 100, 0, fetch_rows=False)
        s = ens.conformation_sums().reshape(4, 3, -1).sum(axis=1)
    avg = pm.lib.conformation_averages(s, 12, 8)
    h, rows = _read_csv(pre + "_summary.csv")
    assert h == ["Fz", "kT", "samples", "S_xx", "S_yy", "S_zz", "S_xy", "S_xz", "S_yz", "Rg2", "Rg4"]
    got = np.array([[float(v) for v in row[2:]] for row in rows])
    np.testing.assert_array_equal(got[:, 0], avg["samples"])
    np.testing.assert_array_equal(got[:, 1:7], avg["S"])
    np.testing.assert_array_equal(got[:, 7], avg["Rg2"])
    np.testing.assert_array_equal(got[:, 8], avg["Rg4"])
    h, rows = _read_csv(pre + "_bondcorr.csv")
    assert h == ["Fz", "kT", "s", "C"] and len(rows) == 4 * 12
    np.testing.assert_array_equal(np.array([float(r[3]) for r in rows]).reshape(4, 12), avg["bondcorr"])
    h, rows = _read_csv(pre + "_profile.csv")
    assert h == ["Fz", "kT", "i", "nz", "nz2"] and [r[2] for r in rows[:2]] == ["1", "2"]
    np.testing.assert_array_equal(np.array([float(r[3]) for r in rows]).reshape(4, 12), avg["nz"])
    np.testing.assert_array_equal(np.array([float(r[4]) for r in rows]).reshape(4, 12), avg["nz2"])
    h, rows = _read_csv(pre + "_extension.csv")
    assert h == ["Fz", "kT", "zeta_lo", "zeta_hi", "count", "density"] and len(rows) == 4 * 8
    cnt = np.array([float(r[4]) for r in rows]).reshape(4, 8)
    np.testing.assert_array_equal(cnt, s[:, 8 + 36:])
    np.testing.assert_array_equal(np.array([float(r[5]) for r in rows]).reshape(4, 8),
                                  cnt / (s[:, :1] * 0.25))
    assert os.path.exists(out1)
