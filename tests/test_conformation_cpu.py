"""Conformation sampling, CPU tier: the numpy restatement (tests/conformation_ref.py) on hand-built chains, the closed
forms of non-interacting chains validated on the oracle's runs (so that a wrong formula is never blamed on the kernel),
and the host plumbing: the CSV tables, the run_sweep.py options and the refusals made before any device is touched."""
import ctypes as C

import numpy as np
import pytest

import closed_form as CF
import conformation_ref as CR


@pytest.mark.parametrize("name,nhat,b,want", CR.hand_chains(), ids=[c[0] for c in CR.hand_chains()])
def test_restatement_on_hand_built_chains(name, nhat, b, want):
    n, B = nhat.shape[0], 10
    acc = CR.Sums(n, B)
    acc.add(nhat, b)
    acc.add(nhat, b)
    row = acc.row
    assert row[0] == 2.0
    np.testing.assert_allclose(row[8:8 + n] / 2, want["C"], rtol=1e-14, atol=1e-14)
    np.testing.assert_array_equal(row[8 + n:8 + 2 * n], 2 * nhat[:, 2])
    np.testing.assert_array_equal(row[8 + 2 * n:8 + 3 * n], 2 * nhat[:, 2] ** 2)
    S = row[1:7] / 2
    x = CR.centres(nhat, b)
    assert abs(S[:3].sum() - ((x - x.mean(0)) ** 2).sum(1).mean()) < 1e-13
    if "Szz" in want:
        assert abs(S[2] - want["Szz"]) < 1e-13 and abs(S[0]) < 1e-30
    if "Syy" in want:
        assert S[1] == 0.0 and S[3] == 0.0 and S[5] == 0.0
    np.testing.assert_allclose(row[7] / 2, S[:3].sum() ** 2, rtol=1e-14)
    k = CR.bin_of(b * nhat[:, 2].sum(), n, b, B)
    assert row[8 + 3 * n + k] == 2.0 and row[8 + 3 * n:].sum() == 2.0
    assert k == min(B - 1, max(0, int(np.floor((want["zeta"] + 1) * B / 2))))


def test_bin_edges():
    assert CR.bin_of(-5.0, 5, 1.0, 4) == 0 and CR.bin_of(5.0, 5, 1.0, 4) == 3
    assert CR.bin_of(0.0, 5, 1.0, 4) == 2 and CR.bin_of(-1e-3, 5, 1.0, 4) == 1
    assert CR.bin_of(-2.5, 5, 1.0, 4) == 1       # ζ = −½ is the lower edge of bin 1


def _rg2(n, m2, b=1.0):
    k = np.arange(1, n)
    return b * b * float(((n - k) * ((k - 0.5) + (k * k - k + 0.5) * m2)).sum()) / n ** 2


def _z(x, want):
    x = np.asarray(x)
    return (x.mean(axis=0) - want) / (x.std(axis=0, ddof=1) / np.sqrt(x.shape[0]))


KINDS = {"field_force": dict(E0=1.0, K1=1.0, K2=0.0, Fz=0.6), "free": dict(E0=0.0, Fz=0.0)}


@pytest.mark.parametrize("kind", list(KINDS))
def test_closed_forms_hold_on_the_oracle(O, kind):
    """Non-interacting oracle chains (Philox mode) from the oracle's own random start, one run of 40 000 trials per
    chain with a state row every 100 trials, the first 10 000 trials discarded: the restatement's averages agree with the
    closed forms within 3σ of the spread across chains.  ⟨n̂z²⟩ and ⟨ζ²⟩ see the single-bond density itself (for the free
    chain ⟨R_g²⟩, C_s and ⟨n̂z⟩ depend on m = 0 alone).

    The samples come from one call: the oracle keys its draws by the trial index within a call, so a sequence of short
    calls would replay the same draws and sample another distribution."""
    n, chains, nsteps, every, burn_rows = 8, 256, 40000, 100, 100
    kw = dict(n=n, energy_type="noninteracting", chain_type="dielectric", **KINDS[kind])
    case = O.make_case(**kw)
    mom = CF.single_monomer_moments(**{k: v for k, v in kw.items() if k not in ("n", "energy_type")})
    m, mzz = mom["n"], mom["n2"][2]
    m2 = float(m @ m)
    per, zeta = [], []
    for c in range(chains):
        run = O.Run(case, 77, c, 1)
        _, _, st = run.steps_ex(nsteps, every, want_state=True)
        phi, theta = st[:, 0::2], st[:, 1::2]
        nh = np.stack([np.sin(theta) * np.cos(phi), np.sin(theta) * np.sin(phi), np.cos(theta)], axis=-1)
        if c == 0:     # the restatement's monomer centres are the oracle's x_i (load_chain's convention)
            np.testing.assert_allclose(CR.centres(nh[-1], 1.0), run.chain().xs(), rtol=0, atol=1e-12)
        acc = CR.Sums(n, 0)
        for x in nh[burn_rows:]:
            acc.add(x, 1.0)
        per.append(acc.row / acc.row[0])
        z = nh[burn_rows:, :, 2].sum(axis=1) / n        # ζ = r_z / (n b), r = b Σ n̂
        zeta.append([z.mean(), (z * z).mean()])
    per, zeta = np.array(per), np.array(zeta)
    zs = {"Rg2": _z(per[:, 1] + per[:, 2] + per[:, 3], _rg2(n, m2))}
    bc = per[:, 8:8 + n] / np.arange(n, 0, -1)
    np.testing.assert_allclose(bc[:, 0], 1.0, rtol=1e-14)
    for s in (1, 2, 5):
        zs[f"C{s}"] = _z(bc[:, s], m2)
    zs["nz"] = _z(per[:, 8 + n:8 + 2 * n].mean(1), m[2])
    zs["nz2"] = _z(per[:, 8 + 2 * n:8 + 3 * n].mean(1), mzz)
    zs["zeta"] = _z(zeta[:, 0], m[2])
    zs["zeta2"] = _z(zeta[:, 1], (mzz - m[2] ** 2) / n + m[2] ** 2)
    assert all(abs(v) < 3 for v in zs.values()), zs


def test_rg2_closed_form_on_exact_moments():
    """The formula against a brute-force expectation over i.i.d. bonds: for n = 3 with n̂ ∈ {±ẑ, ±x̂} each with
    probability ¼ (m = 0) and with n̂ = ẑ always (a rod, |m|² = 1)."""
    assert abs(_rg2(7, 1.0) - (7 * 7 - 1) / 12.0) < 1e-13        # the rod: (n² − 1)/12 for b = 1
    dirs = [np.array(v, float) for v in ([0, 0, 1], [0, 0, -1], [1, 0, 0], [-1, 0, 0])]
    tot = 0.0
    for a in dirs:
        for b_ in dirs:
            for c in dirs:
                x = CR.centres(np.array([a, b_, c]), 1.0)
                tot += ((x - x.mean(0)) ** 2).sum(1).mean()
    assert abs(tot / 64 - _rg2(3, 0.0)) < 1e-14


def test_conformation_tables_and_csv(tmp_path):
    import polymc as pm
    from polymc import sweep
    n, B = 3, 4
    sums = np.zeros((2, 8 + 3 * n + B))
    sums[:, 0] = [4, 8]
    sums[:, 1:7] = np.arange(12).reshape(2, 6)
    sums[:, 7] = [2, 4]
    sums[:, 8:8 + n] = [[12, 8, 4], [24, 16, 8]]
    sums[:, 8 + n:8 + 2 * n] = 1.0
    sums[:, 8 + 2 * n:8 + 3 * n] = 2.0
    sums[:, 8 + 3 * n:] = [[1, 2, 1, 0], [0, 0, 4, 4]]
    pargs = [{"Fz": 0.0, "kT": 1.0}, {"Fz": 0.5, "kT": 1.0}]
    conf = {"buckets": [dict(n=n, bins=B, cases=np.array([0, 1]), sums=sums)]}
    t = sweep.conformation_tables(pargs, conf, ["Fz"])
    assert t["summary"][0] == ["Fz", "samples", "S_xx", "S_yy", "S_zz", "S_xy", "S_xz", "S_yz", "Rg2", "Rg4"]
    assert t["summary"][1][0] == [0.0, 4, 0.0, 0.25, 0.5, 0.75, 1.0, 1.25, 0.75, 0.5]
    assert t["bondcorr"][1][:3] == [[0.0, 0, 1.0], [0.0, 1, 1.0], [0.0, 2, 1.0]]
    assert t["profile"][1][0] == [0.0, 1, 0.25, 0.5] and t["profile"][1][3] == [0.5, 1, 0.125, 0.25]
    assert t["extension"][1][1] == [0.0, -0.5, 0.0, 2, 1.0]
    assert t["extension"][1][6] == [0.5, 0.0, 0.5, 4, 1.0]
    avg = pm.lib.conformation_averages(sums, n, B)
    np.testing.assert_array_equal(avg["hist"][1], [0, 0, 0.5, 0.5])
    path = tmp_path / "x_extension.csv"
    sweep.write_exchange_csv(str(path), *t["extension"])
    lines = path.read_text().splitlines()
    assert lines[0] == "Fz,zeta_lo,zeta_hi,count,density"
    assert lines[2] == "0.0,-0.5,0.0,2,1.0"


def _main(argv):
    import run_sweep
    return run_sweep.main(argv)


def test_run_sweep_refusals_before_any_device(tmp_path):
    out = str(tmp_path / "t.csv")
    common = ["--", "-n", "4", "--num-steps", "100"]
    with pytest.raises(SystemExit):
        _main(["--out", out, "--conformation-out", str(tmp_path / "c"), *common])
    with pytest.raises(SystemExit):
        _main(["--out", out, "--grid", "kT=1,2", "--temper", "kT", "--exchange-every", "50",
               "--conformation-every", "25", *common])
    with pytest.raises(SystemExit):
        _main(["--out", out, "--conformation-every", "-1", *common])
    import polymc as pm
    with pytest.raises(pm.PolymcError, match="umbrella"):
        _main(["--out", out, "--conformation-every", "50", *common, "--umbrella-sampling"])
    with pytest.raises(pm.PolymcError, match="must divide --num-steps"):
        _main(["--out", out, "--conformation-every", "30", *common])
    from polymc import sweep
    with pytest.raises(pm.PolymcError, match="must equal --exchange-every"):
        sweep.run_shard([pm.make_case(n=4, kT=1.0), pm.make_case(n=4, kT=2.0)], 2, 100, temper="kT", exchange_every=50,
                        conformation_every=25)


def test_c_abi_without_a_device():
    """The new entry points refuse a null handle; without a device no handle exists (pmc_create: PMC_ERR_NO_DEVICE)."""
    import polymc as pm
    L = pm.lib.load()
    assert "pmc_run_sampled" in pm.lib.EXPORTS and "pmc_conformation_sums" in pm.lib.EXPORTS
    assert L.pmc_set_conformation(None, 1, 4) == -1
    assert L.pmc_sample_conformation(None) == -1
    assert L.pmc_conformation_cols(None) == 0
    assert L.pmc_run_sampled(None, 100, 10, 0, None, None) == -1
    assert L.pmc_conformation_sums(None, None) == -1
    if pm.device_count() == 0:
        h = C.c_void_p()
        rc = L.pmc_create(pm.make_case(n=4), 1, 1, 0, 0, 0, C.byref(h))
        assert rc == -2, pm.lib.load().pmc_last_error()
