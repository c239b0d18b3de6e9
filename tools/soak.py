"""Developer soak test (run on the GPU box): long runs of every kernel family; checks that every average stays finite,
that the trial counters add up, and reports the drift of the running energy against a full recompute (diag[7])."""
import sys, time
sys.path.insert(0, "polymer-stats_b200")
import numpy as np
import polymc as pm
CASES = [
    ("plain interacting n=512", dict(n=512, E0=1.0, Fz=0.5, energy_type="interacting"), 1024, 40000, False),
    ("plain interacting n=100 (small ensemble)", dict(n=100, E0=1.0, Fz=0.5, energy_type="interacting"), 100, 400000, False),
    ("plain Ising n=100 (warp)", dict(n=100, E0=1.0, Fz=0.5, energy_type="Ising"), 2048, 2000000, False),
    ("plain non-interacting n=100 (lane)", dict(n=100, E0=1.0, Fz=0.5), 65536, 200000, False),
    ("clustering interacting n=100", dict(n=100, E0=1.0, Fz=0.25, energy_type="interacting", kappa=0.5, clustering=True, adj_ub=0.4), 1184, 200000, True),
    ("clustering cut-off n=400", dict(n=400, E0=1.0, Fz=0.25, energy_type="cutoff", cutoff_radius=7.5, kappa=0.5, clustering=True, adj_ub=0.4), 592, 20000, True),
    ("clustering Ising n=100 (warp)", dict(n=100, E0=1.0, Fz=0.25, energy_type="Ising", kappa=0.5, clustering=True, adj_ub=0.4), 500, 2000000, True),
    ("clustering Ising n=100 (lane)", dict(n=100, E0=1.0, Fz=0.25, energy_type="Ising", kappa=0.5, clustering=True, adj_ub=0.4), 32768, 100000, True),
    ("plain interacting n=1024 (two SMs per chain)", dict(n=1024, E0=1.0, Fz=0.5, energy_type="interacting"), 592, 6000, False),
    ("plain interacting n=4096 (two SMs per chain, C5 shape)", dict(n=4096, E0=1.0, Fz=0.5, energy_type="interacting"), 148, 600, False),
    ("planar Ising n=100 (warp)", dict(n=100, E0=0.3, Fz=0.25, energy_type="Ising", clustering=True, planar=True, adj_ub=0.4), 500, 300000, True),
]
bad = 0
for name, kw, R, steps, cl in CASES:
    ens = pm.Ensemble(pm.make_case(**kw), replicas=R, seed=99)
    if cl:
        ens.begin_stage(1.0)
    run = (lambda s: ens.run_ex(s, 0, fetch_rows=False)) if cl else (lambda s: ens.run(s, 0, fetch_rows=False))
    t0 = time.time()
    run(steps // 2)
    run(steps - steps // 2)      # the second call re-synchronises: diag[7] = drift accumulated over the first
    dt = time.time() - t0
    avg, ar, nrm = ens.averages()
    d = ens.diagnostics()
    ok = bool(np.isfinite(avg).all() and np.all(nrm == steps) and np.all(d[:, 5] == steps) and np.all((ar > 0) & (ar < 1)))
    scale = np.maximum(1.0, np.abs(d[:, 6]))
    print("%-45s %s  %d chains x %d trials in %.1f s (%.1f M updates/s); acceptance %.3f; max drift |U_run - U_recomputed| "
          "= %.2e (relative %.1e)" % (name, "ok " if ok else "BAD", R, steps, dt, R * steps / dt / 1e6, ar.mean(),
                                      d[:, 7].max(), (d[:, 7] / scale).max()), flush=True)
    bad += not ok
    ens.close()

# Cross-kernel decision equality over long runs (compute-sanitizer is closed on this pool: a race in a barrier protocol
# would show up as a different accept/reject sequence): the same ensemble through the windowed one-CTA kernel and the
# CTA-pair kernel (cluster barrier + distributed shared memory) must count the same acceptances per chain — the reduction orders differ, so only a decision within rounding of its threshold could legitimately differ.
import os
for n, R, steps in ((512, 444, 20000), (1024, 300, 6000), (200, 1000, 40000)):
    counts = {}
    for tag, env in (("windowed", dict(PMC_RUN_PAIR="0")), ("pair", dict(PMC_RUN_PAIR="2"))):
        os.environ.update(env)
        with pm.Ensemble(pm.make_case(n=n, E0=1.0, Fz=0.5, energy_type="interacting"), replicas=R, seed=4242) as ens:
            name = ens.kernel_name()
            t0 = time.time()
            ens.run(steps, 0, fetch_rows=False)
            counts[tag] = (ens.diagnostics()[:, 4].copy(), name, time.time() - t0)
    same = np.array_equal(counts["windowed"][0], counts["pair"][0])
    diff = int((counts["windowed"][0] != counts["pair"][0]).sum())
    print("decision equality n=%d, %d chains x %d trials: %s (%s %.1f s, %s %.1f s); chains with a different acceptance "
          "count: %d" % (n, R, steps, "ok " if same else "DIFF", counts["windowed"][1], counts["windowed"][2], counts["pair"][1],
                         counts["pair"][2], diff), flush=True)
    bad += not same
os.environ.pop("PMC_RUN_PAIR", None)

# Chain per lane against chain per warp (32 speculative trials per window, resolved in order): both are the reference's
# sequential Markov chain on the same Philox stream, so the final STATES must be equal bit for bit and the acceptance
# counts equal — over long runs, with flips, with step adaptation on, for equal-idx (non-interacting) and neighbour
# (Ising) conflicts.
for kw, R, steps in ((dict(n=100, E0=1.0, Fz=0.5), 4096, 300000), (dict(n=100, E0=1.0, Fz=0.5, energy_type="Ising"), 4096, 300000),
                     (dict(n=12, E0=2.0, Fz=0.2, kT=0.5, energy_type="Ising", chain_type="polar", mu=0.7, do_flips=True), 2048, 400000),
                     (dict(n=7, E0=0.5, Fz=1.0, steps_per_adjust=333), 2048, 400000)):
    res = {}
    for tag, mode in (("lane", "1"), ("warp", "2")):
        os.environ["PMC_LANE_MODE"] = mode
        with pm.Ensemble(pm.make_case(**kw), replicas=R, seed=777) as ens:
            name = ens.kernel_name()
            t0 = time.time()
            ens.run(steps // 3, 0, fetch_rows=False)
            ens.run(steps - steps // 3, 1000, fetch_rows=False)
            res[tag] = (ens.diagnostics()[:, 4].copy(), ens.get_state_all(), name, time.time() - t0)
    os.environ.pop("PMC_LANE_MODE", None)
    same = np.array_equal(res["lane"][0], res["warp"][0]) and all(np.array_equal(a, b) for a, b in zip(res["lane"][1], res["warp"][1]))
    print("lane vs warp %s, %d chains x %d trials: %s (%s %.1f s, %s %.1f s)" % (
        {k: v for k, v in kw.items() if k in ("n", "energy_type", "do_flips")}, R, steps, "ok  states and acceptance counts identical"
        if same else "DIFF", res["lane"][2], res["lane"][3], res["warp"][2], res["warp"][3]), flush=True)
    bad += not same

# Composite trials: 8 / 4 / 2 one-warp teams on different trials of the window, committed in order (k_run_cta_cluster_spec),
# against one team per chain: identical acceptance counts, cluster statistics and final chains over long runs.
for kw, R, steps in ((dict(n=100, E0=1.0, Fz=0.25, energy_type="interacting", kappa=0.5), 96, 150000),
                     (dict(n=64, E0=0.5, Fz=0.3, kT=3.0, energy_type="interacting", kappa=0.2, cluster_prob=0.4), 96, 200000),
                     (dict(n=120, E0=1.0, Fz=0.25, energy_type="cutoff", cutoff_radius=5.0, kappa=0.5), 64, 100000)):
    res = {}
    for hint in (10 ** 6, 600, 300, 0):
        with pm.Ensemble(pm.make_case(clustering=True, adj_ub=0.4, **kw), replicas=R, seed=31337, ensemble_chains=hint) as ens:
            ens.begin_stage(1.0)
            t0 = time.time()
            ens.run_ex(steps // 2, 0, fetch_rows=False)
            ens.run_ex(steps - steps // 2, 5000, fetch_rows=False)
            res[hint] = (ens.diagnostics()[:, 4].copy(), ens.cluster_stats().copy(), ens.get_state_all(), ens.kernel_name(), time.time() - t0,
                         ens.diagnostics()[:, 6].copy())
    ref = res[10 ** 6]
    # per chain: identical acceptance count, cluster statistics and final chain in every variant
    eq = np.ones(R, dtype=bool)
    for r in res.values():
        eq &= (ref[0] == r[0]) & np.all(ref[1] == r[1], axis=1) & np.all(ref[2][0] == r[2][0], axis=1) & np.all(ref[2][1] == r[2][1], axis=1)
    # A chain of point dipoles without excluded volume can collapse until two monomers sit on top of each other
    # (|U| ~ 1e9 kT and more): there a trial's ΔU is a difference of sums that contain such a term, its rounding error
    # (1e-16 |U|) reaches the scale of kT·|log ε − logπ ratio| and the variants — whose staged positions differ in the
    # last bit — may legitimately part ways.  tests/devtools/debug_spec2.py: the first differing trial of such a chain has the same
    # ΔU through the seam in both shapes, and the speculative teams stay on the CPU oracle's trajectory.
    collapsed = np.abs(res[10 ** 6][5]) > 1e8
    same = bool(np.all(eq | collapsed))
    print("speculative teams %s, %d chains x %d trials (acceptance %.3f): %s  %s" % (
        {k: v for k, v in kw.items() if k in ("n", "energy_type")}, R, steps, ref[0].sum() / (R * steps),
        ("ok  identical acceptance counts, cluster statistics and final chains" if same else "DIFF") +
        ("" if eq.all() else " (%d chain(s) differ, all collapsed: |U| = %s)" % ((~eq).sum(), ", ".join("%.1e" % abs(u) for u in res[10 ** 6][5][~eq]))),
        ", ".join("%s %.1f s" % (r[3], r[4]) for r in res.values())), flush=True)
    bad += not same

# The same for the plain driver's single-monomer trials (k_run_cta_win_spec) against the one-trial kernel
for kw, R, steps, hints in ((dict(n=48, E0=1.0, Fz=0.5), 96, 300000, (10 ** 6, 800, 300, 0)),
                            (dict(n=64, E0=0.5, Fz=0.2, kT=3.0, chain_type="polar", mu=0.6, do_flips=True), 96, 300000, (10 ** 6, 800, 300, 0)),
                            (dict(n=100, E0=1.0, Fz=0.5), 96, 150000, (10 ** 6, 0))):
    res = {}
    for hint in hints:
        with pm.Ensemble(pm.make_case(energy_type="interacting", **kw), replicas=R, seed=271828, ensemble_chains=hint) as ens:
            t0 = time.time()
            ens.run(steps // 2, 0, fetch_rows=False)
            ens.run(steps - steps // 2, 5000, fetch_rows=False)
            d = ens.diagnostics()
            res[hint] = (d[:, 4].copy(), ens.get_state_all(), ens.kernel_name(), time.time() - t0, d[:, 6].copy())
    ref = res[10 ** 6]
    eq = np.ones(R, dtype=bool)
    for r in res.values():
        eq &= (ref[0] == r[0]) & np.all(ref[1][0] == r[1][0], axis=1) & np.all(ref[1][1] == r[1][1], axis=1)
    collapsed = np.abs(ref[4]) > 1e8     # see above: rounding at the scale of kT once two monomers sit on top of each other
    same = bool(np.all(eq | collapsed))
    print("speculative teams, plain driver %s, %d chains x %d trials (acceptance %.3f): %s  %s" % (
        {k: v for k, v in kw.items() if k in ("n", "chain_type")}, R, steps, ref[0].sum() / (R * steps),
        ("ok  identical acceptance counts and final chains" if same else "DIFF") +
        ("" if eq.all() else " (%d chain(s) differ, all collapsed: |U| = %s)" % ((~eq).sum(), ", ".join("%.1e" % abs(u) for u in ref[4][~eq]))),
        ", ".join("%s %.1f s" % (r[2], r[3]) for r in res.values())), flush=True)
    bad += not same

# The opt-in FP32 rectangle on a chain that stays extended (weak coupling): drift of the running energy per launch
with pm.Ensemble(pm.make_case(n=512, E0=0.3, Fz=1.0, energy_type="interacting"), replicas=1024, seed=5) as ens:
    ens.set_pair_precision("fp32")
    t0 = time.time()
    for _ in range(4):
        ens.run(5000, 0, fetch_rows=False)
    d = ens.diagnostics()
    ok = bool(np.isfinite(d).all() and np.all(d[:, 5] == 20000))
    print("fp32 rectangle n=512 E0=0.3: %s  %s, 1024 chains x 20000 trials in %.1f s (%.1f M updates/s); acceptance %.3f; |U| up to %.2e; "
          "max drift within 5000 trials %.2e" % ("ok " if ok else "BAD", ens.kernel_name(), time.time() - t0, 1024 * 20000 / (time.time() - t0) / 1e6,
                                                 d[:, 4].sum() / d[:, 5].sum(), np.abs(d[:, 6]).max(), d[:, 7].max()), flush=True)
    bad += not ok
sys.exit(1 if bad else 0)
