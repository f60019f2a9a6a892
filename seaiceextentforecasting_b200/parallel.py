"""Multi-GPU glue (SURVEY.md 8(e)): one process per GPU, `torch.distributed` (NCCL on the box, gloo in the CPU tests).

Ways the path shards, all without moving `R`:
  * independent (config, year) tasks: `SweepPlan(rank, world)` owns whole tasks, ranks exchange nothing during the
    step; `gather_results` all-gathers the GP records (80-byte structs, tensor collective) at the end;
  * one large network (25 km grid): `sie_corr_tau(shard_rank, shard_count)` computes the 128-row tile rows
    `bi % shard_count == shard_rank` of the upper triangle, so every rank holds a partial (sum, count) of the
    significant correlations; `tau_from_shards` all-reduces those 16 bytes per network; `build_networks_sharded` then
    grows the domains on one rank from the replicated z rows and broadcasts labels + node series;
  * many large networks (a 25 km retrospective sweep): rank r builds networks r, r + world, ... locally and
    `all_gather_networks` gives every rank all labels / node series (the north_star's all-gather).
"""
from __future__ import annotations

import numpy as np
import torch
import torch.distributed as dist

TILE_ROWS = 128     # csrc/corr.cu TILE


def shard_tile_rows(n_nodes, rank, count):
    """Tile rows (128 nodes each) of the upper triangle computed by `rank` of `count` (csrc/corr.cu shard_rows)."""
    nb = (int(n_nodes) + TILE_ROWS - 1) // TILE_ROWS
    return list(range(rank, nb, count))


def tau_from_shards(tau_sum, tau_cnt, group=None):
    """tau_sum (float64 [B]), tau_cnt (int64 [B]): this rank's partials -> the global tau [B] on every rank
    (ComplexNetworks.py:45-47: mean of the significant non-negative correlations over both triangles)."""
    s = tau_sum.clone()
    c = tau_cnt.clone()
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(s, op=dist.ReduceOp.SUM, group=group)
        dist.all_reduce(c, op=dist.ReduceOp.SUM, group=group)
    return s / c.to(torch.float64)


NETWORK_TENSORS = ("n_areas", "area_key", "area_start", "area_cells", "label", "status", "anomaly")


def network_state(eng):
    """The result of a network build that other ranks need: domain labels (area tables + per-cell label) and the node
    series -- `labels (C x int32)` and `nA x T x f64` per network (SURVEY.md C2); R and z never leave the GPU."""
    return {k: getattr(eng, k) for k in NETWORK_TENSORS}


def broadcast_networks(state, src=0, group=None):
    """Broadcast every tensor of `state` (network_state of an engine, or CPU tensors under gloo) from rank `src`
    in place.  Used after a network whose correlation pass was row-sharded has been grown on one rank."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        for k in NETWORK_TENSORS:
            dist.broadcast(state[k], src=src, group=group)
    return state


def all_gather_networks(state, n_jobs_total, group=None):
    """Rank r built the networks (jobs) r, r + world, r + 2 world, ... of a sweep in a LOCAL batch (`state`: its
    network_state, job-major).  Returns the same tensors for ALL `n_jobs_total` jobs in global job order on every rank:
    one all-gather per tensor of labels / area tables / node series (a few hundred KB per 25 km network)."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return {k: state[k][:n_jobs_total] for k in NETWORK_TENSORS}
    world = dist.get_world_size(group)
    per = (n_jobs_total + world - 1) // world
    out = {}
    for k in NETWORK_TENSORS:
        t = state[k]
        pad = torch.zeros((per,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
        n = min(per, t.shape[0])
        pad[:n] = t[:n]
        parts = [torch.empty_like(pad) for _ in range(world)]
        dist.all_gather(parts, pad, group=group)
        stacked = torch.stack(parts, dim=1)                      # [per][world][...]: job = i * world + rank
        out[k] = stacked.reshape((per * world,) + tuple(t.shape[1:]))[:n_jobs_total]
    return out


def build_networks_sharded(eng, fields, job_field, job_T, r_crit, scale, do_detrend=True, group=None, grow_rank=0):
    """Multi-GPU build of the networks of ONE batch held identically by every rank (the 25 km configuration: a single
    network is a sequential algorithm, only its all-pairs correlation pass shards).  `eng`: NetworkBatch(keep_R=False).
      K1 on every rank (the unit-norm rows z, <= 46 MB per network, are replicated by recomputing them);
      K2 tau-only, rank r computes the 128-row tile rows bi % world == r of the upper triangle; the (sum, count) partials
         are all-reduced -- 16 bytes per network over NCCL; the matrix is never stored and never crosses NVLink;
      K3-K5 (domain growth, correlations recomputed from z) and K6 on `grow_rank`;
      labels / area tables / node series are broadcast from `grow_rank` (<= 1 MB per network).
    Every rank returns with the same tau and network_state."""
    world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
    rank = dist.get_rank(group) if world > 1 else 0
    assert eng.R is None, "the sharded build never stores R: construct the NetworkBatch with keep_R=False"
    eng.detrend_zscore(fields, job_field, job_T, do_detrend)
    eng.corr_tau(r_crit, store_R=False, shard_rank=rank, shard_count=world)
    tau = tau_from_shards(eng.tau_sum, eng.tau_cnt, group)
    eng.tau.copy_(tau)
    if rank == grow_rank:
        eng.area_level()
        eng.intra_links(scale)
    broadcast_networks(network_state(eng), src=grow_rank, group=group)
    return eng.tau


def gather_records(plan, raw, group=None, device=None, raw_dev=None):
    """Tensor all-gather of every rank's GP records (80 B each) and their (config, region, year, member) keys: ranks
    own different numbers of problems, so the counts are gathered first and the payloads padded to the largest.
    Returns (raw_all, meta_all [P,3], member_all [P]) in rank order.  `device`: where the collective runs ("cuda" under
    NCCL, "cpu" under gloo); default = CUDA when the backend is NCCL.  `raw_dev`: the records as a uint8 device tensor
    (GpBatch.out) instead of `raw` -- the payload then goes GPU -> NVLink -> GPU without a host round trip."""
    from .forecast import GP_RESULT_DTYPE
    if raw is None:
        raw = np.zeros(plan.P, dtype=GP_RESULT_DTYPE) if raw_dev is not None else np.zeros(0, dtype=GP_RESULT_DTYPE)
        if raw_dev is not None and not (dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1):
            raw = raw_dev.cpu().numpy().view(GP_RESULT_DTYPE)[:plan.P]
    raw = np.ascontiguousarray(raw)
    meta = np.asarray(plan.prob_meta, dtype=np.int32).reshape(-1, 3)
    keys = np.concatenate([meta, np.asarray(plan.prob_member, dtype=np.int32).reshape(-1, 1)], axis=1)
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return raw, keys[:, :3], keys[:, 3]
    world = dist.get_world_size(group)
    if device is None:
        device = "cuda" if dist.get_backend(group) == "nccl" else "cpu"
    isz = raw.dtype.itemsize
    n = torch.tensor([len(raw)], dtype=torch.int64, device=device)
    counts = [torch.zeros_like(n) for _ in range(world)]
    dist.all_gather(counts, n, group=group)
    counts = [int(c.item()) for c in counts]
    cap = max(max(counts), 1)
    pay = torch.zeros(cap * isz, dtype=torch.uint8, device=device)
    if raw_dev is not None:
        pay[:len(raw) * isz] = raw_dev[:len(raw) * isz].to(device)
    else:
        pay[:len(raw) * isz] = torch.from_numpy(raw.view(np.uint8).reshape(-1).copy()).to(device)
    key = torch.zeros((cap, 4), dtype=torch.int32, device=device)
    key[:len(raw)] = torch.from_numpy(np.ascontiguousarray(keys)).to(device)
    pays = [torch.empty_like(pay) for _ in range(world)]
    keyl = [torch.empty_like(key) for _ in range(world)]
    dist.all_gather(pays, pay, group=group)
    dist.all_gather(keyl, key, group=group)
    raw_all = np.concatenate([p.cpu().numpy()[:c * isz].view(raw.dtype) for p, c in zip(pays, counts)])
    key_all = np.concatenate([k.cpu().numpy()[:c] for k, c in zip(keyl, counts)])
    return raw_all, key_all[:, :3], key_all[:, 3]


def gather_selection(selection, group=None, device=None):
    """Tensor all-gather of every rank's tuned-sweep selection (RetrospectiveSweep.selection: the (l, sigma_n~, grid
    index) each of its problems was forecast with), concatenated in the rank order of gather_records, so that every
    rank assembles the same tuned dict.  Any structured per-problem array gathers the same way (the marginal records
    of a marginalised sweep)."""
    sel = np.ascontiguousarray(selection)
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return sel
    world = dist.get_world_size(group)
    if device is None:
        device = "cuda" if dist.get_backend(group) == "nccl" else "cpu"
    isz = sel.dtype.itemsize
    n = torch.tensor([len(sel)], dtype=torch.int64, device=device)
    counts = [torch.zeros_like(n) for _ in range(world)]
    dist.all_gather(counts, n, group=group)
    counts = [int(c.item()) for c in counts]
    pay = torch.zeros(max(max(counts), 1) * isz, dtype=torch.uint8, device=device)
    pay[:len(sel) * isz] = torch.from_numpy(sel.view(np.uint8).reshape(-1).copy()).to(device)
    pays = [torch.empty_like(pay) for _ in range(world)]
    dist.all_gather(pays, pay, group=group)
    return np.concatenate([p.cpu().numpy()[:c * isz].view(sel.dtype) for p, c in zip(pays, counts)])


def gather_results(plan, raw, group=None, device=None, selection=None, marginal=None):
    """Every rank's GP records -> the assembled GPR dict of the whole sweep (SweepPlan.assemble) on every rank.
    `selection`: this rank's tuned-sweep selection (RetrospectiveSweep.selection), `marginal`: this rank's
    marginal-sweep records (RetrospectiveSweep.marginal), gathered alongside."""
    raw_all, meta, member = gather_records(plan, raw, group, device)
    sel_all = None if selection is None else gather_selection(selection, group, device)
    marg_all = None if marginal is None else gather_selection(marginal, group, device)
    return plan.assemble(raw_all, meta, member, selection=sel_all, marginal=marg_all)
