"""Per-stage timeline of one sweep step in two-wave mode (event times relative to the step start, ms)."""
import sys, os; sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import bench
from seaiceextentforecasting_b200.config import NORTH_INITS
from seaiceextentforecasting_b200.forecast import RetrospectiveSweep
wave_T = tuple(int(x) for x in sys.argv[1].split(',')) if len(sys.argv) > 1 else (12, 24)
w = bench.make_workload(0)
sw = RetrospectiveSweep(NORTH_INITS, w['sic'], w['sie'], bench.FMIN, bench.FMAX, w['psar'], w['sst'], w['lat'], wave_T=wave_T)
sw.upload()
for _ in range(3): sw.compute()
torch.cuda.synchronize()
for waves in (None, 1):
    for _ in range(3): sw.compute(waves=waves)       # steady state: the marked step is queued behind others
    e0 = torch.cuda.Event(enable_timing=True); e0.record()
    marks = []; sw.compute(marks, waves=waves)
    e1 = torch.cuda.Event(enable_timing=True); e1.record(); torch.cuda.synchronize()
    print("waves", waves, "wave_T", wave_T, "total ms", round(e0.elapsed_time(e1), 2), "ranges", sw.waves)
    for name, ev in marks: print("   %-22s %7.2f" % (name, e0.elapsed_time(ev)))
