/*
 * sie_b200.h -- C ABI of libsie_b200.so: the B200 (sm_100a) implementation of the data-parallel core
 * of the complex-network + Gaussian-process sea-ice-extent forecaster.
 *
 * The reference (William-gregory/SeaIceExtentForecasting) is pure Python and has no FFI; what a
 * maintainer would bind is its Python call surface.  Each entry point below names the reference
 * lines whose arithmetic it replaces (paths relative to the reference checkout).  INTEGRATION.md
 * shows the ctypes stub that sits behind `ComplexNetworks.Network.tau/area_level/intra_links` and
 * the script-level `detrend/networks/forecast/MLII` helpers.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in `_host`; outputs are caller-allocated;
 *   - `stream` is a cudaStream_t passed as void*; calls only enqueue work (no device sync) unless noted;
 *   - return value 0 = enqueued OK, negative = argument/launch error (see sie_last_error());
 *   - per-job data errors (no NaN sentinel cell, fewer than 2 areas, capacity, non-SPD kernel matrix)
 *     are reported through the per-job `status`/`info` device arrays, mirroring LAPACK `info`;
 *   - all floating point is FP64, all indices int32; "cell" = flat grid index i*Y+j, "node" = index
 *     into the ascending list of cells whose series is not identically zero/NaN.
 *   - jobs: one job = one network build (one field window).  B jobs of the same grid are batched.
 */
#ifndef SIE_B200_H
#define SIE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SIE_OK 0
#define SIE_ERR_ARG (-1)          /* bad argument (returned by the call) */
#define SIE_ERR_LAUNCH (-2)       /* CUDA launch/runtime failure (returned by the call) */
#define SIE_ERR_UNSUPPORTED (-3)  /* size outside what this build handles */

/* per-job status codes written to device `status[]` arrays */
#define SIE_JOB_OK 0
#define SIE_JOB_NO_NAN_CELL 1   /* ComplexNetworks.py:50-51 would raise IndexError */
#define SIE_JOB_FEW_AREAS 2     /* ComplexNetworks.py:212/:278 would raise ValueError (<2 areas) */
#define SIE_JOB_CAPACITY 3      /* more areas / nodes than the caller-provided capacity */

#define SIE_AREA_WORK 32        /* uint64 profiling counters per job written by sie_area_level */

int sie_abi_version(void);          /* 2 */
const char* sie_last_error(void);
/* device facts used by the host layer for launch sizing; returns 0 on success */
int sie_device_info(int* sm_count, int* max_smem_optin, size_t* l2_bytes);

/* ---------------------------------------------------------------------------------------------
 * K1  per-cell OLS detrend + unit-norm rows + node compaction.
 * Replaces: detrend()            north/June1st.py:179-194, retro north/retrospective_forecasts/June1st_retro.py:178-195
 *           node mask + the row centring/scaling inside np.corrcoef   ComplexNetworks.py:32-34, :37
 *           first-NaN sentinel cell                                   ComplexNetworks.py:50-51
 * fields      [F][C][Tstride]  input series per cell (NaN = land)
 * job_field   [B]  which field job b windows;  job_T [B] window length (prefix of the series)
 * do_detrend  1: remove the OLS line (detrend()), 0: input already detrended (Network(data=dt))
 * dt          [B][C][Tstride]  residuals (all-NaN for cells with any NaN); may alias nothing; required
 * trend       [B][C][2] slope,intercept (NaN for cells with any NaN) or NULL
 * z           [B][ldn][Tp]  unit-norm centred rows, node-compacted, zero padded to Tp (Tp%4==0)
 * node_cell   [B][ldn], cell_node [B][C] (-1 = not a node), n_nodes [B], first_nan_cell [B] (-1 none)
 * status      [B] SIE_JOB_CAPACITY if n_nodes > ldn (ldn: node capacity, a multiple of 4; K2 needs a multiple of 128);
 *             dt is defined for the window [0, T_b) of every series only
 * B <= 65535 jobs per call; Tp <= ~195 (128 series of Tp+1 doubles are staged in shared memory)
 */
int sie_detrend_zscore(const double* fields, const int32_t* job_field, const int32_t* job_T,
                       int B, int C, int Tstride, int Tp, int do_detrend,
                       double* dt, double* trend, double* z,
                       int32_t* node_cell, int32_t* cell_node, int32_t* n_nodes,
                       int32_t* first_nan_cell, int32_t* status, int ldn, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K2  all-pairs Pearson correlation R = Z Z^T on FP64 tensor-core (DMMA m8n8k4) tiles, operands
 *     staged with bulk async copies (TMA engine) + mbarrier, clip to [-1,1], NaN diagonal, mirrored
 *     (bitwise symmetric) store, and the significance threshold tau.
 * Replaces: np.corrcoef + fill_diagonal + t-test + mean      ComplexNetworks.py:34-35, :41-47
 * r_crit   [B]  host-computed critical correlation: P<alpha  <=>  R > r_crit (SURVEY.md App. B)
 * R        [B][ldn][ldn] or NULL (tau only; nothing but Z is read and 16 B/tile written).  Only the UPPER TRIANGLE is
 *          defined: R[i][j] for i < j, NaN on the diagonal; element (i, j) is read as R[min(i,j)][max(i,j)] by K3, K4/K5
 *          and the host accessors, which makes the matrix symmetric by construction and halves the bytes K2 stores
 *          (SIE_CORR_ROWS also writes the mirror image; do not rely on it)
 * tile_part scratch of sie_corr_tau_scratch_bytes(B, ldn) bytes: tile table (32 B/tile), deterministic per-warp and
 *           per-tile (sum,count) partials; a job range of a batch may use a disjoint slice
 * tau      [B]; tau_sum [B]; tau_cnt [B] (int64)   -- sums are over BOTH triangles like the reference
 * shard_rank/shard_count: tile-row bi is computed by the rank with bi % shard_count == shard_rank
 *     (multi-GPU row-block split; tau is then finished by the caller after an all-reduce of sum/cnt).
 * kernel   SIE_CORR_AUTO: the TMA-store kernel when R is stored (the 128x64 tile kernel when Tp > ~52), the row-resident
 *          warp-specialised kernel for the tau-only pass (R == NULL); SIE_CORR_TILES / SIE_CORR_ROWS / SIE_CORR_TMA force
 *          one (tiles and rows serve both modes; all give the same upper triangle bit for bit).  There is no
 *          environment variable or other hidden state.
 */
#define SIE_CORR_AUTO 0
#define SIE_CORR_TILES 1
#define SIE_CORR_ROWS 2
#define SIE_CORR_ROWS_MIRROR 3   /* rows kernel that also writes the lower triangle (debug / A-B only) */
#define SIE_CORR_TMA 4           /* stored R only: every consumer warp's sub-tile leaves as one tensor-map bulk store (TMA) */
int sie_corr_tau(const double* z, const int32_t* n_nodes, const int32_t* job_T, const double* r_crit,
                 int B, int ldn, int Tp, double* R,
                 double* tile_part, size_t tile_part_bytes,
                 double* tau_sum, int64_t* tau_cnt, double* tau,
                 int shard_rank, int shard_count, int kernel, void* stream);
size_t sie_corr_tau_scratch_bytes(int B, int ldn);

/* Selected rows of the correlation matrix of ONE network recomputed from its unit-norm rows z [ldn][Tp] (N nodes, window
 * T): out[r][c] = R[rows[r]][c], NaN on the diagonal.  Serves the `corrs[n]` accessor of the drop-in Network when R is not
 * stored (ComplexNetworks.py:36-39 scatters exactly these rows).  rows [n_rows] device int32; out [n_rows][ld_out]. */
int sie_corr_rows(const double* z, const int32_t* rows, int n_rows, int N, int T, int Tp, double* out, int ld_out,
                  void* stream);

/* K3  local stencil: correlation of every node with its 4 von-Neumann neighbours (up,down,left,right;
 *     lat-lon wrap in the second axis), NaN where the neighbour is off-grid or not a node.
 * Replaces: the seed search gathers `corrs[ID,nei]`            ComplexNetworks.py:166-172, :53-78
 * R        [B][ldn][ldn], or NULL: the 4 correlations are then recomputed from the unit-norm rows
 *          z [B][ldn][Tp] (job_T [B] = window lengths) -- no stored matrix is needed (25 km grids)
 * stencil  [B][ldn][4]
 */
int sie_corr_stencil(const double* R, const double* z, const int32_t* job_T, int Tp,
                     const int32_t* node_cell, const int32_t* cell_node,
                     const int32_t* n_nodes, int B, int X, int Y, int ldn, int latlon,
                     double* stencil, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K4+K5  tau-thresholded domain growth (step 1) and largest-first merging (step 2); one persistent
 *        CTA per network, numpy-pairwise-order means so decisions are those of the reference.
 * Replaces: Network.area_level                                 ComplexNetworks.py:49-278
 * R          [B][ldn][ldn] correlations (K2), or NULL: every correlation the growth / merge decisions consume is then
 *            recomputed from the unit-norm rows z [B][ldn][Tp] (42 FMAs each; z stays L2-resident), so a network
 *            whose N x N matrix does not fit in HBM can still be built.  job_T [B], Tp: as for K1/K2 (only read
 *            when R == NULL).  Jobs are popped from a queue in index order by a persistent grid: put the slowest
 *            (longest-window) jobs first.  The job statuses written by K1 are read here (a job K1 flagged
 *            SIE_JOB_CAPACITY is skipped), so K1 must have run on the same `status` array.
 * area_cells [B][C]  member cells, area after area in dict order, each area in its list order
 * area_start [B][max_areas+1], area_key [B][max_areas] (the reference's dict keys), n_areas [B]
 * label      [B][C]  index into area_key (dict position) or -1
 * status     [B]  SIE_JOB_* (areas are still written when status == SIE_JOB_FEW_AREAS, like the
 *            reference leaves V populated when it raises at :278)
 * scratch    at least sie_area_level_scratch_bytes(B, X*Y) bytes: the job-queue counter + one block per CTA of the
 *            persistent grid (NOT per job); concurrent calls need disjoint scratch
 * work       [B][SIE_AREA_WORK] or NULL: per job {0: correlations consumed (the algorithmic gather count, 8 B
 *            each), 1: SM cycles in step 1, 2: SM cycles in step 2, 3: (growth steps << 32) | merge rounds,
 *            4..14: SM cycles per phase (step 1: seed search, evaluate+argmax, frontier update, gathers;
 *            step 2: select/materialise, neighbour discovery, neighbour lists, row means, statistic,
 *            merge/finalise; 14 unused), 15: growth steps that took the re-summing path}; the per-phase entries
 *            4..14 and 16..25 are only filled by a build with -DSIE_AREA_PHASE_TIMERS (they cost ~6 % of the kernel)
 */
int sie_area_level(const double* R, const double* z, const int32_t* job_T, int Tp,
                   const double* stencil, const int32_t* node_cell,
                   const int32_t* cell_node, const int32_t* n_nodes, const double* tau,
                   const int32_t* first_nan_cell, int B, int X, int Y, int ldn, int latlon,
                   int max_areas, int32_t* area_cells, int32_t* area_start, int32_t* area_key,
                   int32_t* n_areas, int32_t* label, int32_t* status,
                   void* scratch, size_t scratch_bytes, uint64_t* work, void* stream);
size_t sie_area_level_scratch_bytes(int B, int C);

/* ---------------------------------------------------------------------------------------------
 * K6  area-weighted node series (deterministic row-major segmented sums), population-covariance
 *     links, strength, strength map.
 * Replaces: Network.intra_links                                ComplexNetworks.py:283-326
 * scale      [C]  sqrt(area) or sqrt(cos(lat)) or ones (host computes the square root, :296-301)
 * area_cells [B][C], area_start [B][max_areas+1], n_areas [B], label [B][C]: the outputs of sie_area_level (the member
 *            list of an area is rank-sorted into ascending cell order on the device: numpy's reduction order)
 * anomaly    [B][max_areas][Tstride]; links [B][max_areas][max_areas]; strength [B][max_areas];
 * strengthmap [B][C] (NaN outside areas)
 */
int sie_intra_links(const double* dt, const double* scale, const int32_t* job_T,
                    const int32_t* area_cells, const int32_t* area_start, const int32_t* n_areas,
                    const int32_t* label, int B, int C, int Tstride, int max_areas,
                    double* anomaly, double* links, double* strength, double* strengthmap,
                    void* stream);

/* ---------------------------------------------------------------------------------------------
 * K7-K9  batched GP forecast: predictor selection, optional z-score, graph-Laplacian prior,
 *        expm (Al-Mohy & Higham scaling-and-squaring Pade, the algorithm behind scipy.linalg.expm),
 *        Cholesky fit, predictive mean/variance, negative log marginal likelihood (+ MLII gradient).
 * Replaces: forecast()  north/June1st.py:208-279 (and the 13 sibling scripts), MLII :235-257
 *
 * One problem = one (network set, region, hyper-parameter pair).  Problem p reads:
 *   y            y_all + prob[p].y_off, n = prob[p].n training targets
 *   predictors   up to two series sets (SIC, SST): set s has n_areas[job_s] series of length n+1 at
 *                anomaly + (job_s*max_areas + a)*Tstride
 * and writes out[p] = {fmean, fvar, sigma_f, nlml, g_ell, g_sig, n_pred, expm_m, expm_s, info, cycles...}.
 */
typedef struct SieGpProblem {
  int32_t job_sic;      /* index into the first anomaly set (required) */
  int32_t job_sst;      /* index into the second anomaly set, or -1 */
  int32_t n;            /* training rows; series provide n+1 samples (last = test year) */
  int32_t y_off;        /* offset of y[0..n) in y_all */
  int32_t rule;         /* 0: r>0, 1: all, 2: (r>0)&(p/2<alpha) i.e. r > r_sel */
  int32_t zscore;       /* 1: column z-score over the n+1 rows (June scripts) */
  int32_t want_grad;    /* 1: also evaluate the MLII gradient */
  int32_t pad_;
  double r_sel;         /* critical r for rule 2 (host: beta(n/2-1,n/2-1,-1,2).isf(alpha)) */
  double ell;           /* l */
  double sig;           /* sigma_n tilde */
} SieGpProblem;

typedef struct SieGpResult {
  double fmean, fvar, sigma_f, nlml, g_ell, g_sig;
  int32_t n_pred, expm_m, expm_s, info; /* info: 0 ok, k>0 Cholesky failed at pivot k (LinAlgError), -1 fewer than 2 predictors selected (the reference raises IndexError / ValueError), -2 capacity */
  int64_t cycles_total, cycles_expm;    /* SM cycles this problem took (whole / expm only), for profiling */
} SieGpResult;

int sie_gp_forecast(const SieGpProblem* prob, int P, const double* y_all,
                    const double* anom_sic, const int32_t* n_areas_sic, int max_areas_sic, int Tstride_sic,
                    const double* anom_sst, const int32_t* n_areas_sst, int max_areas_sst, int Tstride_sst,
                    int max_pred, SieGpResult* out, void* scratch, size_t scratch_bytes, void* stream);
size_t sie_gp_scratch_bytes(int P, int max_pred, int max_n);
/* Profiling aid, not part of the reference-facing interface: reads and clears 16 per-phase SM-cycle counters of the GP kernel
 * (all zero unless the library was built with -DSIE_GP_TIMERS; tools/gp_phases.py). */
int sie_debug_gp_phases(unsigned long long* out16);

/* Hyper-parameter grid (the search the reference leaves commented out at north/June1st.py:259-262, done over the
 * `ls` x `ss` grids of :210-211): problem p fixes (network set, region, l = prob[p].ell); Sigma~ = expm(l M) and
 * W = X Sigma~ X^T are built once and the fit / nlML (MLII :235-257) is evaluated for every sig_grid[k].
 * prob[p].sig is ignored.  out [P][n_sig].  Same scratch as sie_gp_forecast. */
int sie_gp_hyper_grid(const SieGpProblem* prob, int P, const double* sig_grid, int n_sig, const double* y_all,
                      const double* anom_sic, const int32_t* n_areas_sic, int max_areas_sic, int Tstride_sic,
                      const double* anom_sst, const int32_t* n_areas_sst, int max_areas_sst, int Tstride_sst,
                      int max_pred, SieGpResult* out, void* scratch, size_t scratch_bytes, void* stream);

/* Grid minimum of MLII per problem (type-II maximum likelihood on the grid).  grid [P][n_ell][n_sig] are records of
 * sie_gp_hyper_grid over the problems prob[p] with l = ell_grid[i].  A point is admissible when info == 0 and nlml is
 * finite.  best[p] = i*n_sig + j of the smallest admissible nlml; ties go to the smallest flat index (np.argmin over
 * [n_ell][n_sig]).  best[p] = -1 when no point is admissible.  tuned[p] = prob[p] with ell/sig replaced by the
 * selected pair (unchanged when best[p] = -1), ready for sie_gp_forecast.  Reads only nlml and info of the records;
 * the result is bit-reproducible.  Enqueue only. */
int sie_gp_grid_select(const SieGpResult* grid, const SieGpProblem* prob, int P,
                       const double* ell_grid, int n_ell, const double* sig_grid, int n_sig,
                       SieGpProblem* tuned, int32_t* best, void* stream);

/* Grid marginal of the forecast per problem: the average over the (l, sigma_n~) grid of every grid point's forecast,
 * weighted by its marginal likelihood (the Bayesian completion of type-II maximum likelihood on the grid).
 * grid [P][n_grid] are records of sie_gp_hyper_grid (as for sie_gp_grid_select, n_grid = n_ell * n_sig).
 *   A    = {k : info_k == 0 and nlml_k finite} (sie_gp_grid_select's rule), m = min over A of nlml_k
 *   e_k  = exp(m - nlml_k), S0 = sum_A e_k, w_k = e_k / S0: a uniform prior over the admissible grid points -- on the
 *          reference's log-spaced grids, log-uniform in l and in sigma_n~.  nlml profiles sigma_f out (sigma_f =
 *          y^T K~^-1 y / n at each point), so these are profile-likelihood weights.
 *   out[p] = record argmax with fmean = sum w mu, fvar = sum w (v + (mu - fmean)^2) (law of total variance, second
 *          pass) and nlml = m - log S0 + log|A| (-log of the grid-averaged marginal likelihood)
 *   stats[p] = {ess = S0^2 / sum e^2, w_max = 1 / S0, n_admissible = |A|, argmax = sie_gp_grid_select's best}
 *   quant [P][n_q]: quantiles of F(x) = sum w Phi((x - mu) / sqrt(v)) at the levels q [n_q] (0 < q < 1; a component
 *          with v <= 0 is a point mass at mu), by bisection on [min(mu - 40 sqrt(v)), max(mu + 40 sqrt(v))] over the
 *          points with w > 0, keeping F(lo) < q <= F(hi), at most 128 halvings; the result is hi
 * With A empty: out[p] = record 0 with fmean, fvar and nlml NaN (info stays the record's, e.g. -1), stats = {NaN, NaN,
 * 0, -1}, quantiles NaN.  n_q == 0: q and quant may be NULL.  One warp per problem, fixed-order reductions: the result
 * is bit-reproducible.  Enqueue only. */
typedef struct SieGpMarginal {
  double ess;            /* effective number of grid points, S0^2 / sum e_k^2 */
  double w_max;          /* largest posterior weight, 1 / S0 */
  int32_t n_admissible;  /* |A| */
  int32_t argmax;        /* flat index of the largest weight; -1 when A is empty */
} SieGpMarginal;         /* 24 bytes */

int sie_gp_grid_marginal(const SieGpResult* grid, int P, int n_grid, const double* q, int n_q,
                         SieGpResult* out, SieGpMarginal* stats, double* quant, void* stream);

/* Ensemble pool per problem: the forecasts of M input-perturbed ensemble members pooled into one predictive
 * distribution, each contributing member with weight 1 / M'.  rec [E][M][n_grid]: E ensemble problems (config, region,
 * year) x M member slots x n_grid records per member -- n_grid = 1 for the forecast records of plain or tuned sweeps,
 * n_grid = n_ell * n_sig for the grid records of marginalised sweeps.  Per member m, sie_gp_grid_marginal's
 * arithmetic (A_m, e_k = exp(min - nlml_k), S0_m; same lane order): its mean mu_m = sum e mu / S0_m and variance
 * v_m = sum e (v + (mu - mu_m)^2) / S0_m have the bits of that member's marginal record.  A member with A_m empty does
 * not contribute; M' = the members that do.
 *   out[e] = {fmean = sum mu_m / M', var_within = sum v_m / M', var_between = sum (mu_m - fmean)^2 / M' (second pass),
 *             fvar = var_within + var_between, n_members = M'}
 *   quant [E][n_q]: quantiles of F(x) = (1/M') sum_m (1/S0_m) sum_k e_mk Phi((x - mu_mk) / sd_mk) at the levels q
 *          (0 < q < 1; v <= 0 is a point mass), by sie_gp_grid_marginal's bisection rule over the components with e > 0
 * M' = 0: fmean, fvar, both variance terms and the quantiles NaN, n_members 0.  n_q == 0: q and quant may be NULL.
 * scratch: at least sie_gp_ensemble_scratch_bytes(E, M, n_grid) bytes (the weighted components of every problem,
 * 24 B per record).  Limits: M <= 1024 and M * n_grid < 2^31, else SIE_ERR_UNSUPPORTED.  One CTA per problem,
 * sums in an order fixed by (M, n_grid): bit-reproducible, whichever launch filled which member slot.  Enqueue only. */
typedef struct SieGpEnsemble {
  double fmean;          /* mean of the pooled predictive distribution */
  double fvar;           /* var_within + var_between */
  double var_within;     /* mean over the contributing members of their predictive variance */
  double var_between;    /* mean over the contributing members of (member mean - fmean)^2 */
  int32_t n_members;     /* M' = members with at least one admissible record */
  int32_t pad_;
} SieGpEnsemble;         /* 40 bytes */

int sie_gp_ensemble(const SieGpResult* rec, int E, int M, int n_grid, const double* q, int n_q,
                    SieGpEnsemble* out, double* quant, void* scratch, size_t scratch_bytes, void* stream);
size_t sie_gp_ensemble_scratch_bytes(int E, int M, int n_grid);

/* ---------------------------------------------------------------------------------------------
 * Ingest (SURVEY.md 8(f) rows 1 and 4: the steps immediately before the hot path).
 * Replaces: readNSIDC                                          north/September1st.py:72-139
 *
 * sie_nsidc_monthly   files [n_files][file_stride] raw NSIDC .bin images (300-byte header + C bytes, :93-104/:121-127)
 *                     -> monthly [C] = nanmean over the files of byte/250, values > 1 (flags) -> NaN (:128)
 * sie_polar_hole_fill phole = nanmean(monthly[hole-0.5 < lat < hole]); filled = where(lat >= hole-0.5, phole, monthly)
 *                     (:129-136); scratch [C] doubles; phole is also returned through *phole (device)
 * sie_regrid_linear   scipy griddata(..., 'linear') (:137-138) as a 3-nnz-per-row SpMV: vert [Ct][3] source cells of
 *                     the enclosing Delaunay triangle (-1 = outside the hull -> NaN), bary [Ct][3] barycentric
 *                     weights; src [F][C] -> dst [F][Ct]
 */
int sie_nsidc_monthly(const uint8_t* files, int n_files, size_t file_stride, int header_bytes, int C,
                      double* monthly, void* stream);
int sie_polar_hole_fill(const double* monthly, const double* lat, double hole, int C, double* filled,
                        double* phole, double* scratch, void* stream);
int sie_regrid_linear(const double* src, int F, int C, const int32_t* vert, const double* bary, int Ct,
                      double* dst, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SIE_B200_H */
