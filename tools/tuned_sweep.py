"""Tuned retrospective sweep on the bench's 8-member north step (bench.make_workload): every forecast at the minimum of
MLII's nlML over the reference's 20 x 20 (l, sigma_n~) grid (RetrospectiveSweep(hyper_grid=(LS, SS))).

    python tools/tuned_sweep.py [--steps K] [--reps R] [--members-total N] [--out FILE]
    torchrun --nproc-per-node G tools/tuned_sweep.py --members-total 1024 [--out FILE]

In one process: the plain and the tuned step device-resident (inputs in HBM, CUDA events after warm-up, the two
alternated R times, K steps each), the tuned step's split into network chain / grid / select + forecast (every stage
alone on one stream, minimum over passes), the card's name and power limit (read-only query), and the ensemble
stream: --members-total members (split over the ranks, weak scaling) run in batches of 8 through ONE sweep's device
buffers (RetrospectiveSweep.load_inputs), each batch with its H2D, tuned step and D2H + assemble, the next batch's
inputs generated on the host while the device computes.  Prints one JSON line (rank 0) and writes it to --out."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import bench  # noqa: E402
from seaiceextentforecasting_b200.config import LS, NORTH_INITS, SS  # noqa: E402
from seaiceextentforecasting_b200.forecast import RetrospectiveSweep  # noqa: E402

M = 8   # members per step (bench.MEMBERS)


def member_inputs(base, m):
    """bench.make_workload(m) from make_workload(0) without regenerating the base fields (the same perturbation:
    checked against make_workload for the first batch)."""
    if m == 0:
        return base
    rng = np.random.default_rng(5000 + m)
    sic = {}
    for name in NORTH_INITS:
        f = base["sic"][name]
        inside = (f > 0.0) & (f < 1.0)
        sic[name] = np.where(inside, np.clip(f + 0.05 * rng.standard_normal(f.shape), 0.0, 1.0), f)
    return dict(base, sic=sic, sst=base["sst"] + 0.05 * rng.standard_normal(base["sst"].shape))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q}


def sweep(ws, tuned):
    return RetrospectiveSweep(NORTH_INITS, [w["sic"] for w in ws], ws[0]["sie"], bench.FMIN, bench.FMAX, ws[0]["psar"],
                              [w["sst"] for w in ws], ws[0]["lat"], hyper_grid=(LS, SS) if tuned else None)


def device_ms(sw, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        sw.compute()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def split_ms(sw, passes=3):
    """Minimum over passes of: network chains (SST + SIC, serial), grid, select + forecast (waves=0: one stream)."""
    best = {}
    for _ in range(passes):
        marks = []
        sw.compute(marks, waves=0)
        torch.cuda.synchronize()
        t = dict(marks)
        first = marks[0][1]
        parts = {"network_chain": first.elapsed_time(t["gp.start"])}
        if "gp.grid" in t:
            parts.update(grid=t["gp.start"].elapsed_time(t["gp.grid"]), select_forecast=t["gp.grid"].elapsed_time(t["gp"]))
        else:
            parts["gp"] = t["gp.start"].elapsed_time(t["gp"])
        for k, v in parts.items():
            best[k] = min(best.get(k, v), v)
    return best


def resident(ws, args):
    """Plain and tuned step device-resident, alternated (the two sweeps live only inside this call)."""
    plain, tuned = sweep(ws, False), sweep(ws, True)
    for sw in (plain, tuned):
        sw.upload()
        for _ in range(args.warmup):
            sw.compute()
    torch.cuda.synchronize()
    ms = {"plain": [], "tuned": []}
    for r in range(args.reps):
        order = (("plain", plain), ("tuned", tuned)) if r % 2 == 0 else (("tuned", tuned), ("plain", plain))
        for name, sw in order:
            ms[name].append(device_ms(sw, args.steps))
    P = tuned.P
    evals = P * len(LS) * len(SS)
    split = split_ms(tuned)
    split_plain = split_ms(plain)
    med = {k: statistics.median(v) for k, v in ms.items()}
    tuned.download()
    plain.download()
    return {"timing": f"CUDA events around {args.steps} back-to-back compute() calls, {args.reps} repetitions "
                      "alternating plain / tuned, after warm-up; median reported",
            "plain_ms_per_step": ms["plain"], "tuned_ms_per_step": ms["tuned"],
            "plain_forecasts_per_s": P / (med["plain"] * 1e-3), "tuned_forecasts_per_s": P / (med["tuned"] * 1e-3),
            "grid_evaluations_per_step": evals,
            "grid_evaluations_per_s_step": evals / (med["tuned"] * 1e-3),
            "grid_evaluations_per_s_grid_kernel": evals / (split["grid"] * 1e-3),
            "split_ms_tuned_serial": split, "split_ms_plain_serial": split_plain,
            "tuned_problems_at_a_grid_point": int((tuned.best_index() >= 0).sum()),
            "problems": P, "info_minus1": int((tuned.raw["info"] == -1).sum())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--reps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--members-total", type=int, default=1024)
    ap.add_argument("--out")
    args = ap.parse_args()
    rank, local, world = (int(os.environ.get(k, d)) for k, d in (("RANK", 0), ("LOCAL_RANK", 0), ("WORLD_SIZE", 1)))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import __graft_entry__ as entry
    if rank == 0:
        entry.build()
    if world > 1:
        dist.barrier()
    base = bench.make_workload(0)
    ws = [member_inputs(base, rank * M + m) for m in range(M)]
    for m, w in enumerate(ws):                   # the cheap generator is bench's
        ref = bench.make_workload(rank * M + m)
        assert all(np.array_equal(w["sic"][n], ref["sic"][n], equal_nan=True) for n in NORTH_INITS)
        assert np.array_equal(w["sst"], ref["sst"], equal_nan=True)
    result = {"tool": "tools/tuned_sweep.py", "card": card(), "world": world,
              "workload": f"bench.make_workload members 0..{M - 1}: {M} x 432 north forecasts per step, grid "
                          f"{len(LS)} l x {len(SS)} sigma_n~ (north/June1st.py:210-211)"}

    if rank == 0:
        result["device_resident"] = resident(ws, args)
        torch.cuda.empty_cache()

    # ---------------- ensemble stream through load_inputs (weak scaling over ranks)
    per_rank = args.members_total // world
    first = rank * per_rank
    nb = per_rank // M
    gen = lambda b: [member_inputs(base, first + b * M + m) for m in range(M)]   # noqa: E731
    batch = gen(0)
    sw = sweep(batch, True)
    sw.run()                                    # warm-up: buffers, streams, kernel attributes
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fails = 0
    for b in range(nb):
        if b > 0:
            sw.load_inputs([w["sic"] for w in batch], [w["sst"] for w in batch])
        sw.upload()
        sw.compute()
        nxt = gen(b + 1) if b + 1 < nb else None   # host generation of the next batch overlaps the device step
        out = sw.plan.assemble(sw.download(), selection=sw.selection)
        assert len(out) == M
        fails += int((sw.raw["info"] == -1).sum())
        batch = nxt
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    t = torch.tensor([wall], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    wall_max = float(t.item())
    total = nb * M * world * 432
    result["stream"] = {"members_total": nb * M * world, "members_per_rank": nb * M, "batches_per_rank": nb,
                        "gpus": world, "scaling": "weak", "forecasts": total, "wall_s": wall_max,
                        "forecasts_per_s": total / wall_max,
                        "timing": "host clock around the whole stream on every rank (max over ranks): per batch "
                                  "load_inputs + H2D + tuned step + D2H + assemble; next batch generated on the host "
                                  "while the device computes",
                        "info_minus1_rank0": fails}
    if rank == 0:
        line = json.dumps(result)
        print(line)
        if args.out:
            with open(args.out, "w") as f:
                f.write(line + "\n")
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
