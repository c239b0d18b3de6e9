"""Tiny workload for compute-sanitizer (racecheck / memcheck): every kernel family of the library once."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "polymer-stats_b200"))
import polymc as pm

which = sys.argv[1] if len(sys.argv) > 1 else "all"
if which in ("all", "plain"):
    for et, n in (("interacting", 70), ("interacting", 200), ("Ising", 30), ("noninteracting", 30)):
        c = pm.make_case(n=n, E0=1.0, Fz=0.5, energy_type=et, steps_per_adjust=10, do_flips=True)
        with pm.Ensemble(c, replicas=3, seed=2) as ens:
            ens.run(40, 10)
            ens.delta_u(1, n // 2, 0.1, 0.2)
            ens.energy(2)
            ens.reinit()
            ens.run(20, 10)
            print(et, n, ens.kernel_name(), ens.averages()[1])
    os.environ["PMC_LANE_MODE"] = "1"                       # chain per lane, with row stores through shared memory
    with pm.Ensemble(pm.make_case(n=20, E0=1.0, Fz=0.5, energy_type="Ising"), replicas=70, seed=2) as ens:
        ens.run(40, 10)
        print(ens.kernel_name(), ens.averages()[1][:2])
    del os.environ["PMC_LANE_MODE"]
if which in ("all", "pair"):
    os.environ["PMC_RUN_PAIR"] = "2"                        # two SMs per chain: cluster barrier + distributed shared memory
    for n, R in ((70, 3), (300, 5)):
        with pm.Ensemble(pm.make_case(n=n, E0=1.0, Fz=0.5, energy_type="interacting", steps_per_adjust=10), replicas=R, seed=2) as ens:
            ens.run(30, 10)
            print(ens.kernel_name(), ens.averages()[1])
    del os.environ["PMC_RUN_PAIR"]
if which in ("all", "cluster"):
    for et, n in (("interacting", 40), ("interacting", 200), ("cutoff", 60), ("Ising", 30), ("noninteracting", 30)):
        c = pm.make_case(n=n, E0=1.0, Fz=0.5, energy_type=et, kappa=0.5, clustering=True, adj_ub=0.4, steps_per_adjust=10, cutoff_radius=3.0)
        with pm.Ensemble(c, replicas=3, seed=2) as ens:
            ens.begin_stage(2.0)
            ens.run_ex(40, 10)
            ens.delta_segment(1, n // 2, 0.1, 0.2, True, n // 2 - 1, n // 2 + 2)
            print(et, n, ens.kernel_name(), ens.averages()[1])
if which in ("all", "multi"):
    with pm.MultiEnsemble(pm.make_case(n=40, E0=1.0, Fz=0.5, energy_type="interacting"), replicas=5, seed=2, devices=[0, 0]) as m:
        m.run(30, 10)
        print("multi", m.gather_backend(), m.gather()[:, 16])
print("done")
