"""The launch schedule of RetrospectiveSweep.compute(): every libsie_b200 call one step enqueues, in enqueue order, with
its integer arguments and its stream, pinned against tests/golden/sweep_schedule.json for the plain, tuned ("argmin")
and marginal sweeps.  The default multi-wave schedule is what bench.py times, so its order, ranges and streams must not
drift; the one-wave (waves=1) and serial (waves=0) schedules must issue the same calls, the serial one on one stream.

    python tests/test_sweep_schedule_gpu.py      # rewrites the golden file from the current tree (needs the GPU)
"""
import collections
import ctypes as C
import json
import os
import sys

import pytest

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sweep_schedule.json")
MODES = {"plain": {}, "argmin": {"hyper_mode": "argmin"},
         "marginal": {"hyper_mode": "marginal", "quantiles": (0.05, 0.5, 0.95)}}
SCHEDULES = {"default": None, "one_wave": 1, "serial": 0}
GP_LAUNCHES = ("sie_gp_forecast", "sie_gp_hyper_grid")


class Recorder:
    """Wraps every entry point of the loaded library that enqueues work (its last argument is the stream) and logs
    (name, integer arguments, stream ordinal numbered by first appearance).  Pointers are not recorded.  A GP launch's
    scratch capacity is recorded as whether it holds the launch's full CTA grid (sie_gp_scratch_bytes of its problem
    count): that, not the buffer's size, decides how the kernel runs."""

    def __init__(self, lib):
        from seaiceextentforecasting_b200 import _lib
        self.lib, self.calls, self._streams, self._orig = lib, [], {}, {}
        self._enqueue = {n: a for n, (_, a) in _lib._SIGS.items() if a and a[-1] is C.c_void_p}

    def __enter__(self):
        for name, argtypes in self._enqueue.items():
            self._orig[name] = getattr(self.lib, name)
            setattr(self.lib, name, self._wrap(name, argtypes, self._orig[name]))
        return self

    def __exit__(self, *exc):
        for name, fn in self._orig.items():
            setattr(self.lib, name, fn)

    def _wrap(self, name, argtypes, fn):
        def call(*args):
            ints = []
            for t, v in zip(argtypes[:-1], args[:-1]):
                if t is C.c_void_p:
                    continue
                if t is C.c_size_t and name in GP_LAUNCHES:     # ints[0] = problem count, ints[-1] = max_pred
                    v = v >= self.lib.sie_gp_scratch_bytes(ints[0], ints[-1], 64)
                ints.append(int(v))
            stream = args[-1].value if isinstance(args[-1], C.c_void_p) else args[-1]
            self.calls.append([name, ints, self._streams.setdefault(stream, len(self._streams))])
            return fn(*args)
        return call


def record(mode):
    """{schedule: [[name, ints, stream ordinal], ...]} of one compute() of the small 4-init + SST sweep per schedule."""
    import torch

    from seaiceextentforecasting_b200 import _lib
    from seaiceextentforecasting_b200.config import LS, NORTH_INITS, SS
    from seaiceextentforecasting_b200.forecast import RetrospectiveSweep
    from test_tuned_sweep_gpu import FMAX, FMIN, small_inputs
    w = small_inputs()
    kw = dict(MODES[mode], hyper_grid=(LS, SS)) if MODES[mode] else {}
    sw = RetrospectiveSweep(NORTH_INITS, w["sic"], w["sie"], FMIN, FMAX, w["psar"], w["sst"], w["lat"], wave_T=(16,),
                            **kw)
    assert sw.multi_wave and sw.gp_sst
    sw.upload()
    sw.compute()
    torch.cuda.synchronize()
    out = {}
    for name, waves in SCHEDULES.items():
        with Recorder(_lib.load()) as rec:
            sw.compute(waves=waves)
            torch.cuda.synchronize()
        out[name] = rec.calls
    return out


def multiset(calls):
    return collections.Counter((name, tuple(ints)) for name, ints, _ in calls)


@pytest.mark.parametrize("mode", list(MODES))
def test_schedule_is_pinned(lib_built, mode):
    with open(GOLDEN) as f:
        golden = json.load(f)[mode]
    got = record(mode)
    assert got["default"] == golden["default"]
    assert multiset(got["serial"]) == multiset(got["one_wave"]) == multiset(golden["serial"])
    assert {s for _, _, s in got["serial"]} == {0}


if __name__ == "__main__":
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import __graft_entry__
    __graft_entry__.build()
    result = {mode: record(mode) for mode in MODES}
    with open(GOLDEN, "w") as f:
        json.dump(result, f, indent=None, separators=(",", ":"))
        f.write("\n")
    print({m: {s: len(c) for s, c in r.items()} for m, r in result.items()})
