"""Host side of tuned retrospective sweeps (no GPU): the device-side problem expansion (run here on CPU tensors), the
tuned GPR dict, the multi-rank gather of the selection (world_size 2 over gloo) and the C ABI's argument checks."""
import ctypes
import os
import socket

import numpy as np

from seaiceextentforecasting_b200.config import CONFIGS, LS, NORTH_INITS
from seaiceextentforecasting_b200.forecast import (GP_PROBLEM_DTYPE, GP_RESULT_DTYPE, SELECTION_DTYPE, SweepPlan,
                                                   expand_problems)


def _sie():
    rng = np.random.default_rng(0)
    return {r: 10 + rng.standard_normal(42) for r in CONFIGS["north_june"].regions}


def _fake(plan):
    """Records / selections whose values name their problem: fmean = id, ell = id + 0.5, sig = id + 0.25, best = id % 7 - 1."""
    raw = np.zeros(plan.P, dtype=GP_RESULT_DTYPE)
    sel = np.zeros(plan.P, dtype=SELECTION_DTYPE)
    for i, ((ci, k, year), m) in enumerate(zip(plan.prob_meta, plan.prob_member)):
        pid = m * 10000 + ci * 1000 + k * 100 + (year - 2000)
        raw["fmean"][i], sel["ell"][i], sel["sig"][i], sel["best"][i] = pid, pid + 0.5, pid + 0.25, pid % 7 - 1
    return raw, sel


def test_expand_problems_is_np_repeat_with_the_ell_grid():
    import torch
    plan = SweepPlan(NORTH_INITS, _sie(), 2015, 2020)
    prob = torch.from_numpy(plan.prob.view(np.uint8).copy())
    out = torch.empty(plan.P * len(LS) * GP_PROBLEM_DTYPE.itemsize, dtype=torch.uint8)
    expand_problems(prob, torch.from_numpy(LS.copy()), out)
    ref = np.repeat(plan.prob, len(LS))
    ref["ell"] = np.tile(LS, plan.P)
    assert out.numpy().tobytes() == ref.tobytes()


def test_assemble_with_selection_adds_the_used_hyperparameters():
    for members in (1, 2):
        plan = SweepPlan(NORTH_INITS, _sie(), 2015, 2020, members=members)
        raw, sel = _fake(plan)
        plain, tuned = plan.assemble(raw), plan.assemble(raw, selection=sel)
        plains, tuneds = (plain, tuned) if members > 1 else ([plain], [tuned])
        for m, (p, t) in enumerate(zip(plains, tuneds)):
            for ci, cfg in enumerate(plan.cfgs):
                for k, reg in enumerate(cfg.regions):
                    for key, v in p[cfg.name].items():               # the plain keys are untouched
                        assert np.array_equal(t[cfg.name][key], v, equal_nan=True)
                    pid = np.array([m * 10000 + ci * 1000 + k * 100 + (y - 2000) for y in plan.years], dtype=float)
                    assert np.array_equal(t[cfg.name][reg + "_ell"], pid + 0.5)
                    assert np.array_equal(t[cfg.name][reg + "_sig"], pid + 0.25)
                    assert np.array_equal(t[cfg.name][reg + "_grid_index"], pid % 7 - 1)
                assert set(t[cfg.name]) - set(p[cfg.name]) == {reg + s for reg in cfg.regions
                                                               for s in ("_ell", "_sig", "_grid_index")}


def _worker(rank, world, port, q):
    import torch.distributed as dist
    from seaiceextentforecasting_b200 import parallel
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    ok = True
    for members in (1, 3):                                           # 3 members: ranks own unequal problem counts
        plan = SweepPlan(NORTH_INITS, _sie(), 2015, 2020, rank=rank, world=world, members=members)
        full = SweepPlan(NORTH_INITS, _sie(), 2015, 2020, members=members)
        raw, sel = _fake(plan)
        out = parallel.gather_results(plan, raw, selection=sel)
        full_raw, full_sel = _fake(full)
        ref = full.assemble(full_raw, selection=full_sel)
        outs, refs = (out, ref) if members > 1 else ([out], [ref])
        for o, r in zip(outs, refs):
            for c in r:
                ok &= o[c].keys() == r[c].keys()
                ok &= all(np.array_equal(o[c][k], r[c][k], equal_nan=True) for k in r[c])
    if rank == 0:
        q.put(bool(ok))
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_gather_assembles_the_tuned_sweep():
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    ok = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
    assert ok


def test_grid_select_rejects_bad_arguments(lib_built):
    """Checked before anything is enqueued, so no device is needed."""
    from seaiceextentforecasting_b200 import _lib
    lib = _lib.load()
    buf = (ctypes.c_double * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    null = ctypes.c_void_p(0)
    args = [p, p, 4, p, 20, p, 20, p, p, null]
    for i in (0, 1, 3, 5, 7, 8):                                     # each device pointer NULL in turn
        bad = list(args)
        bad[i] = null
        assert lib.sie_gp_grid_select(*bad) == -1
    for i, v in ((2, 0), (4, 0), (6, 0), (4, -3)):                   # P, n_ell, n_sig < 1
        bad = list(args)
        bad[i] = v
        assert lib.sie_gp_grid_select(*bad) == -1
    assert b"sie_gp_grid_select" in lib.sie_last_error()
