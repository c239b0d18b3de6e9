"""Chain per lane vs chain per warp on large O(1)-ΔU ensembles (product build; PMC_LANE_MODE forces the kernel)."""
import os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
child = r'''
import os, sys
sys.path.insert(0, os.path.join(%r, "polymer-stats_b200"))
import polymc as pm
et, n, R, steps = sys.argv[1], int(sys.argv[2]), int(sys.argv[3]), int(sys.argv[4])
c = pm.make_case(n=n, E0=1.0, Fz=0.5, energy_type=et)
ens = pm.Ensemble(c, replicas=R, seed=20260101)
ens.run(max(10, steps // 5), 0, fetch_rows=False)
best = 1e30
for _ in range(3):
    ens.run(steps, 500, fetch_rows=False)
    best = min(best, ens.last_run_ms())
print("%%s n=%%d R=%%d: %%.3f ms  %%.3f G updates/s" %% (et, n, R, best, R*steps/best/1e6))
''' % ROOT
for et in ("noninteracting", "Ising"):
    for R, steps in ((16384, 20000), (65536, 5000), (262144, 2000), (1048576, 500)):
        for mode in (1, 2):
            env = dict(os.environ, PMC_LANE_MODE=str(mode))
            out = subprocess.run([sys.executable, "-c", child, et, "100", str(R), str(steps)], env=env, capture_output=True, text=True)
            print({1: "lane", 2: "warp"}[mode], "->", out.stdout.strip() or out.stderr.strip()[-300:], flush=True)
