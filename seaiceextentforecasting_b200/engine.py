"""Device-resident batch engine: B network builds of one grid shape through K1..K6 of libsie_b200.

PyTorch is used for device memory, pinned host staging and streams only; every number is produced by the
CUDA kernels behind the C ABI (include/sie_b200.h).  There is no CPU implementation to fall back to.
"""
from __future__ import annotations

import ctypes as C
import functools

import numpy as np
import torch

from . import _lib


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def require_cuda():
    if not torch.cuda.is_available():
        raise _lib.SieError("seaiceextentforecasting_b200 needs a CUDA device (sm_100a); there is no CPU path")


@functools.lru_cache(maxsize=None)
def r_crit_ttest(T, alpha):
    """Critical correlation for the one-sided t-test of ComplexNetworks.py:41-45:
    P = t.sf(R*sqrt(df/(1-R^2)), df) < alpha  <=>  R > t_c/sqrt(df+t_c^2), t_c = t.isf(alpha, df), df = T-2."""
    from scipy import stats
    df = T - 2
    if df <= 0:
        return float("nan")
    tc = stats.t.isf(alpha, df)
    return float(tc / np.sqrt(df + tc * tc))


@functools.lru_cache(maxsize=None)
def r_crit_pearson(n, alpha):
    """Critical r of scipy.stats.pearsonr's p-value: (r>0)&(p/2<alpha) <=> r > beta(n/2-1,n/2-1,-1,2).isf(alpha)
    (north/August1st.py:178-181)."""
    from scipy import stats
    if n <= 2:
        return float("nan")
    return float(stats.beta(n / 2.0 - 1.0, n / 2.0 - 1.0, loc=-1.0, scale=2.0).isf(alpha))


def pad_T(T):
    """Row length of z: the smallest Tp >= T with Tp = 4 (mod 8): k-steps of 4 for DMMA.8x8x4 and a row stride
    whose 64-bit fragment loads fall in distinct shared-memory banks."""
    Tp = max(4, (T + 3) // 4 * 4)
    while Tp % 8 != 4:
        Tp += 4
    return Tp


def h2d(arr, dtype=None):
    """numpy -> pinned staging -> device (async on the current stream)."""
    a = np.ascontiguousarray(arr, dtype=dtype)
    t = torch.from_numpy(a)
    try:
        t = t.pin_memory()
    except RuntimeError:
        pass
    return t.to("cuda", non_blocking=True)


class NetworkBatch:
    """B jobs (network builds) on one (X, Y) grid.  All buffers are allocated once and reused."""

    def __init__(self, X, Y, Tstride, B, latlon, n_upper=None, max_areas=None, keep_R=True):
        require_cuda()
        self.lib = _lib.load()
        self.X, self.Y, self.C = int(X), int(Y), int(X) * int(Y)
        self.Tstride, self.B, self.latlon = int(Tstride), int(B), bool(latlon)
        self.Tp = pad_T(self.Tstride)
        n_upper = self.C if n_upper is None else int(n_upper)
        self.ldn = max(128, (n_upper + 127) // 128 * 128)
        # area capacity (step-1 areas per network).  768 keeps the per-area tables of the 57x57 / 26x90 grids small enough
        # for two domain-growth CTAs per SM (csrc/area.cu plan_area); a job that needs more reports SIE_JOB_CAPACITY
        self.MA = int(max_areas) if max_areas else min(self.C // 2 + 1, 768)
        dev = "cuda"
        f64, i32 = torch.float64, torch.int32
        B_, C_, ldn, MA, Ts, Tp = self.B, self.C, self.ldn, self.MA, self.Tstride, self.Tp
        self.dt = torch.empty((B_, C_, Ts), dtype=f64, device=dev)
        self.trend = torch.empty((B_, C_, 2), dtype=f64, device=dev)
        self.z = torch.empty((B_, ldn, Tp), dtype=f64, device=dev)
        self.node_cell = torch.empty((B_, ldn), dtype=i32, device=dev)
        self.cell_node = torch.empty((B_, C_), dtype=i32, device=dev)
        self.n_nodes = torch.empty((B_,), dtype=i32, device=dev)
        self.first_nan = torch.empty((B_,), dtype=i32, device=dev)
        self.status = torch.zeros((B_,), dtype=i32, device=dev)
        self.R = torch.empty((B_, ldn, ldn), dtype=f64, device=dev) if keep_R else None
        self.tau_scratch_bytes = int(self.lib.sie_corr_tau_scratch_bytes(B_, ldn)) + \
            B_ * int(self.lib.sie_corr_tau_scratch_bytes(1, ldn)) + 4096   # room for per-range slices
        self.tau_scratch = torch.empty((self.tau_scratch_bytes + 7) // 8, dtype=f64, device=dev)
        self.tau_sum = torch.empty((B_,), dtype=f64, device=dev)
        self.tau_cnt = torch.empty((B_,), dtype=torch.int64, device=dev)
        self.tau = torch.empty((B_,), dtype=f64, device=dev)
        self.stencil = torch.empty((B_, ldn, 4), dtype=f64, device=dev)
        self.area_cells = torch.empty((B_, C_), dtype=i32, device=dev)
        self.area_start = torch.empty((B_, MA + 1), dtype=i32, device=dev)
        self.area_key = torch.empty((B_, MA), dtype=i32, device=dev)
        self.n_areas = torch.zeros((B_,), dtype=i32, device=dev)
        self.label = torch.empty((B_, C_), dtype=i32, device=dev)
        self._area_scratch = {}          # job range -> scratch of the persistent domain-growth grid (per CTA, not per job)
        self.area_work = torch.zeros((B_, _lib.SIE_AREA_WORK), dtype=torch.int64, device=dev)
        self.anomaly = torch.zeros((B_, MA, Ts), dtype=f64, device=dev)
        self.links = torch.zeros((B_, MA, MA), dtype=f64, device=dev)
        self.strength = torch.zeros((B_, MA), dtype=f64, device=dev)
        self.strengthmap = torch.empty((B_, C_), dtype=f64, device=dev)
        self.job_T = None
        self.launches = 0

    # ---- stages -------------------------------------------------------------------------------
    # Every stage takes an optional job range `jr = (j0, j1)`: jobs are independent and every per-job array is
    # job-major, so a sub-batch is the same C-ABI call on offset pointers.  The retrospective sweep uses this to run
    # two waves (short / long windows) on separate streams.
    def _range(self, jr):
        j0, j1 = (0, self.B) if jr is None else (int(jr[0]), int(jr[1]))
        assert 0 <= j0 < j1 <= self.B
        return j0, j1

    def detrend_zscore(self, fields, job_field, job_T, do_detrend=True, jr=None):
        """K1.  fields: device [F, C, Tstride]; job_field/job_T: device int32 [B]."""
        j0, j1 = self._range(jr)
        self.job_T = job_T
        dt = self.dt if do_detrend else fields
        if not do_detrend:
            assert fields.shape[0] == self.B, "pass-through mode needs one field per job"
            self.dt = fields
        rc = self.lib.sie_detrend_zscore(_ptr(fields), _ptr(job_field[j0:]), _ptr(job_T[j0:]), j1 - j0, self.C,
                                         self.Tstride, self.Tp, 1 if do_detrend else 0, _ptr(dt[j0:]),
                                         _ptr(self.trend[j0:]), _ptr(self.z[j0:]), _ptr(self.node_cell[j0:]),
                                         _ptr(self.cell_node[j0:]), _ptr(self.n_nodes[j0:]), _ptr(self.first_nan[j0:]),
                                         _ptr(self.status[j0:]), self.ldn, _stream())
        _lib.check(rc, "sie_detrend_zscore")
        self.launches += 3

    def corr_tau(self, r_crit, store_R=True, shard_rank=0, shard_count=1, jr=None, kernel=_lib.SIE_CORR_AUTO):
        """K2.  r_crit: device float64 [B].  `kernel`: _lib.SIE_CORR_AUTO / _TILES / _ROWS (include/sie_b200.h)."""
        j0, j1 = self._range(jr)
        R = self.R[j0:] if store_R else None
        # each job range owns a disjoint slice of the tile-partial scratch so ranges can run concurrently
        per_job = int(self.lib.sie_corr_tau_scratch_bytes(1, self.ldn))
        off = (j0 * per_job + 255) // 256 * 256 // 8
        nbytes = int(self.lib.sie_corr_tau_scratch_bytes(j1 - j0, self.ldn))
        scratch = self.tau_scratch[off:]
        assert scratch.numel() * 8 >= nbytes
        rc = self.lib.sie_corr_tau(_ptr(self.z[j0:]), _ptr(self.n_nodes[j0:]), _ptr(self.job_T[j0:]),
                                   _ptr(r_crit[j0:]), j1 - j0, self.ldn, self.Tp, _ptr(R), _ptr(scratch),
                                   scratch.numel() * 8, _ptr(self.tau_sum[j0:]), _ptr(self.tau_cnt[j0:]),
                                   _ptr(self.tau[j0:]), shard_rank, shard_count, int(kernel), _stream())
        _lib.check(rc, "sie_corr_tau")
        self.launches += 5

    def area_level(self, jr=None):
        """K3 + K4/K5.  Without a stored matrix (keep_R=False) every correlation is recomputed from the z rows."""
        j0, j1 = self._range(jr)
        n = j1 - j0
        R = _ptr(self.R[j0:]) if self.R is not None else C.c_void_p(0)
        rc = self.lib.sie_corr_stencil(R, _ptr(self.z[j0:]), _ptr(self.job_T[j0:]), self.Tp,
                                       _ptr(self.node_cell[j0:]), _ptr(self.cell_node[j0:]),
                                       _ptr(self.n_nodes[j0:]), n, self.X, self.Y, self.ldn, int(self.latlon),
                                       _ptr(self.stencil[j0:]), _stream())
        _lib.check(rc, "sie_corr_stencil")
        self.prepare([(j0, j1)])
        scratch = self._area_scratch[(j0, j1)]                # ranges may run concurrently: one scratch each
        rc = self.lib.sie_area_level(R, _ptr(self.z[j0:]), _ptr(self.job_T[j0:]), self.Tp,
                                     _ptr(self.stencil[j0:]), _ptr(self.node_cell[j0:]),
                                     _ptr(self.cell_node[j0:]), _ptr(self.n_nodes[j0:]), _ptr(self.tau[j0:]),
                                     _ptr(self.first_nan[j0:]), n, self.X, self.Y, self.ldn, int(self.latlon),
                                     self.MA, _ptr(self.area_cells[j0:]), _ptr(self.area_start[j0:]),
                                     _ptr(self.area_key[j0:]), _ptr(self.n_areas[j0:]), _ptr(self.label[j0:]),
                                     _ptr(self.status[j0:]), _ptr(scratch), scratch.numel() * 8,
                                     _ptr(self.area_work[j0:]), _stream())
        _lib.check(rc, "sie_area_level")
        self.launches += 2

    def prepare(self, *schedules):
        """Allocate the domain-growth scratch of job ranges (j0, j1) that have none yet; area_level() does so on a
        range's first use, a caller that captures its stages into a CUDA graph calls this up front.  Every schedule is
        a list of ranges that may run concurrently, so they get disjoint scratch; different schedules run one at a time
        (stream order), so they share one allocation."""
        layout, end = {}, 0                     # range -> (offset, float64 count) in the shared allocation
        for ranges in schedules:
            new = [r for r in map(tuple, ranges) if r[1] > r[0] and r not in self._area_scratch]
            off = end if any(r in layout for r in new) else 0      # a range placed by an earlier schedule stays put
            for r in new:
                if r not in layout:
                    n = (int(self.lib.sie_area_level_scratch_bytes(r[1] - r[0], self.C)) + 7) // 8
                    layout[r] = (off, n)
                    off += (n + 63) // 64 * 64                      # 512-byte aligned slices
            end = max(end, off)
        if layout:
            buf = torch.empty(end, dtype=torch.float64, device="cuda")
            for r, (off, n) in layout.items():
                self._area_scratch[r] = buf[off:off + n]

    def intra_links(self, scale, jr=None):
        """K6.  scale: device float64 [C] (already square-rooted weights)."""
        j0, j1 = self._range(jr)
        rc = self.lib.sie_intra_links(_ptr(self.dt[j0:]), _ptr(scale), _ptr(self.job_T[j0:]),
                                      _ptr(self.area_cells[j0:]), _ptr(self.area_start[j0:]),
                                      _ptr(self.n_areas[j0:]), _ptr(self.label[j0:]), j1 - j0, self.C, self.Tstride,
                                      self.MA, _ptr(self.anomaly[j0:]), _ptr(self.links[j0:]),
                                      _ptr(self.strength[j0:]), _ptr(self.strengthmap[j0:]), _stream())
        _lib.check(rc, "sie_intra_links")
        self.launches += 3

    def build(self, fields, job_field, job_T, r_crit, scale, do_detrend=True, jr=None):
        self.detrend_zscore(fields, job_field, job_T, do_detrend, jr)
        self.corr_tau(r_crit, store_R=self.R is not None, jr=jr)
        self.area_level(jr)
        self.intra_links(scale, jr)

    # ---- host views ---------------------------------------------------------------------------
    def areas_to_host(self):
        """-> per job: (status, [(key, [[i,j],...]), ...]) in the reference's dict order."""
        n_areas = self.n_areas.cpu().numpy()
        status = self.status.cpu().numpy()
        starts = self.area_start.cpu().numpy()
        keys = self.area_key.cpu().numpy()
        cells = self.area_cells.cpu().numpy()
        out = []
        Y = self.Y
        for b in range(self.B):
            V = {}
            for a in range(int(n_areas[b])):
                seg = cells[b, starts[b, a]:starts[b, a + 1]]
                V[int(keys[b, a])] = [[int(c // Y), int(c % Y)] for c in seg]
            out.append((int(status[b]), V))
        return out
