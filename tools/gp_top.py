"""Longest GP problems of the north sweep per wave / launch (cycles from the kernel's own clock64 counters)."""
import sys, os; sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import bench
from seaiceextentforecasting_b200.config import NORTH_INITS
from seaiceextentforecasting_b200.forecast import RetrospectiveSweep
w = bench.make_workload(0)
sw = RetrospectiveSweep(NORTH_INITS, w['sic'], w['sie'], bench.FMIN, bench.FMAX, w['psar'], w['sst'], w['lat'])
sw.run(); sw.run()
raw = sw.raw
for launch in sorted(sw._plan.launches, key=lambda l: l.p0):
    wi, a, b, name = launch.wave, launch.p0, launch.p1, "sst" if launch.sst else "sic-only"
    idx = np.arange(a, b); c = raw["cycles_total"][idx] / 1e6
    order = idx[np.argsort(-c)]
    print(f"wave {wi} {name}: {b - a} problems, sum {c.sum():.1f} Mcyc, mean {c.mean():.3f}, max {c.max():.3f}")
    for i in order[:8]:
        print("   ", sw.plan.prob_meta[i], "n", sw.plan.prob[i]["n"], "Np", raw[i]["n_pred"], "m", raw[i]["expm_m"], "s", raw[i]["expm_s"],
              "total Mcyc", round(raw[i]["cycles_total"] / 1e6, 3), "expm", round(raw[i]["cycles_expm"] / 1e6, 3))
