// K7-K9: batched GP forecast -- predictor selection, optional z-score, graph-Laplacian prior, expm,
// Cholesky fit / predict / negative log marginal likelihood (+ MLII gradient).
// Reference: forecast() north/June1st.py:208-279 (13 sibling scripts differ only in the selection rule and
// hyper-parameters), nested MLII() north/June1st.py:235-257.
//
// One CTA per problem (persistent grid, problems strided).  Np x Np matrices (Np = selected predictors,
// up to max_pred) live in a per-CTA global scratch slab that stays L2-resident; the n x n kernel matrices
// (n <= 63 training years) live in shared memory.  expm follows the algorithm scipy.linalg.expm runs
// (Al-Mohy & Higham 2009: Pade order m in {3,5,7,9,13} chosen from ||A^k||_1 of explicit powers, the
// exact ||(|A|)^(2m+1)||_1 backward-error check, 2^-s scaling and s squarings; constants and control flow
// validated against scipy 1.18.1 in tests/test_expm_spec.py), because GP parity at large l*||M|| needs the same
// (m, s) -- an eigendecomposition would be *more* accurate there but would not match the reference.
// FP64 FMA work: ~2 Np^3 (6 + s) flop per expm dominates; Cholesky is 2 n^3/3.
#include "common.cuh"

namespace {

constexpr int GT = 256;          // threads per CTA
constexpr int MAXN = 64;         // n+1 <= 64 samples
constexpr int LDS = MAXN + 1;    // padded leading dimension of the shared n x n matrices

__device__ const double kTheta[5] = {1.495585217958292e-002, 2.539398330063230e-001, 9.504178996162932e-001,
                                     2.097847961257068e+000, 4.25};
// u * c_m, the backward-error constants of Al-Mohy & Higham (u = 2^-53)
__device__ const double kCoeff[5] = {1.1102230246251565e-16 * 100800.0, 1.1102230246251565e-16 * 10059033600.0,
                                     1.1102230246251565e-16 * 4487938430976000.0,
                                     1.1102230246251565e-16 * 5914384781877411840000.0,
                                     1.1102230246251565e-16 * 113250775606021113483283660800000000.0};
__device__ const double kB3[4] = {120., 60., 12., 1.};
__device__ const double kB5[6] = {30240., 15120., 3360., 420., 30., 1.};
__device__ const double kB7[8] = {17297280., 8648640., 1995840., 277200., 25200., 1512., 56., 1.};
__device__ const double kB9[10] = {17643225600., 8821612800., 2075673600., 302702400., 30270240.,
                                   2162160., 110880., 3960., 90., 1.};
__device__ const double kB13[14] = {64764752532480000., 32382376266240000., 7771770303897600., 1187353796428800.,
                                    129060195264000., 10559470521600., 670442572800., 33522128640., 1323241920.,
                                    40840800., 960960., 16380., 182., 1.};

// per-phase SM cycles summed over all problems (thread 0 of every CTA; -DSIE_GP_TIMERS builds only; tools/gp_phases.py)
__device__ unsigned long long g_gp_phase[16];
#ifdef SIE_GP_TIMERS
#define GP_TICK(i) do { if (threadIdx.x == 0) { const long long t__ = clock64(); atomicAdd(&g_gp_phase[i], (unsigned long long)(t__ - gp_t_last)); gp_t_last = t__; } } while (0)
#else
#define GP_TICK(i) do { } while (0)
#endif
constexpr int KC = 16;            // GEMM k-chunk
constexpr int LDA_S = 20;         // As[64][20]: row stride = 4 (mod 16) doubles -> conflict-free DMMA A fragments
constexpr int LDB_S = 68;         // Bs[16][68]: same property for B fragments
constexpr int PANEL = 16;         // LU panel width

struct Smem {
  double As[2][64 * LDA_S];
  double Bs[2][KC * LDB_S];
  union {
    struct {
      double K[MAXN * LDS];       // kernel matrix / Cholesky factor
      double W[MAXN * LDS];       // X Sigma~ X^T
    } gp;
    double panel[2 * MAXN * LDS]; // LU panel (rows x PANEL), only live inside cta_lu_solve
  } u;
  double y[MAXN], ya[MAXN], alpha[MAXN], kxs[MAXN], v[MAXN];
  double red[GT / 32];
  int ired[GT / 32];
  int misc[8];
  double dmisc[8];
  int piv[PANEL];
};

__device__ __forceinline__ double block_sum(double v, Smem& sm) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sm.red[threadIdx.x >> 5] = v;
  __syncthreads();
  double r = 0.0;
#pragma unroll
  for (int w = 0; w < GT / 32; ++w) r += sm.red[w];
  return r;
}
__device__ __forceinline__ double block_max(double v, Smem& sm) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sm.red[threadIdx.x >> 5] = v;
  __syncthreads();
  double r = sm.red[0];
#pragma unroll
  for (int w = 1; w < GT / 32; ++w) r = fmax(r, sm.red[w]);
  return r;
}

__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

// C[m x n2] (op)= A[m x k] * B[k x n2]; row-major with leading dimensions; C must not alias A or B.
//   mode 0: C = A*B      mode 1: C -= A*B
// 64x64 output tiles, 8 warps in a 4x2 grid (16x32 per warp = 2x4 DMMA.8x8x4 blocks), k in chunks of 16.
// The (tile, k-chunk) steps are flattened into one software pipeline: the global loads of step s+1 are issued into
// registers before the tensor work of step s and parked in the other shared-memory buffer afterwards, so one
// barrier per step suffices and L2 latency hides behind the MMAs even when k = 16 (the LU trailing updates).
__device__ __noinline__ void cta_gemm(double* __restrict__ Cm, int ldc, const double* __restrict__ A, int lda,
                         const double* __restrict__ Bm, int ldb, int m, int k, int n2, Smem& sm, int mode = 0) {
  if (m <= 0 || n2 <= 0 || k <= 0) { __syncthreads(); return; }
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wr = warp >> 1, wc = warp & 1;
  const int tm = (m + 63) >> 6, tn = (n2 + 63) >> 6, kc = (k + KC - 1) / KC;
  const int nsteps = tm * tn * kc;
  // loader roles: A tile 64 x 16: thread -> (row = tid/4, 4 consecutive k); B tile 16 x 64: (kk = tid/16, 4 cols)
  const int ar = tid >> 2, ak = (tid & 3) * 4;
  const int bk = tid >> 4, bc = (tid & 15) * 4;
  double ra[4], rb[4];
  auto gload = [&](int step) {
    const int t = step / kc, c = step - t * kc;
    const int ti = t / tn, tj = t - ti * tn;
    const int gr = ti * 64 + ar, gk = c * KC + ak;
    const double* pa = A + (size_t)gr * lda + gk;
#pragma unroll
    for (int q = 0; q < 4; ++q) ra[q] = (gr < m && gk + q < k) ? pa[q] : 0.0;
    const int gkb = c * KC + bk, gc = tj * 64 + bc;
    const double* pb = Bm + (size_t)gkb * ldb + gc;
#pragma unroll
    for (int q = 0; q < 4; ++q) rb[q] = (gkb < k && gc + q < n2) ? pb[q] : 0.0;
  };
  auto spark = [&](int bufi) {
    double* as = sm.As[bufi] + ar * LDA_S + ak;
    double* bs = sm.Bs[bufi] + bk * LDB_S + bc;
    *reinterpret_cast<double2*>(as) = make_double2(ra[0], ra[1]);
    *reinterpret_cast<double2*>(as + 2) = make_double2(ra[2], ra[3]);
    *reinterpret_cast<double2*>(bs) = make_double2(rb[0], rb[1]);
    *reinterpret_cast<double2*>(bs + 2) = make_double2(rb[2], rb[3]);
  };
  double acc[2][4][2];
  gload(0);
  spark(0);
  __syncthreads();
  for (int step = 0; step < nsteps; ++step) {
    const int bufi = step & 1;
    const int t = step / kc, c = step - t * kc;
    if (step + 1 < nsteps) gload(step + 1);
    if (c == 0) {
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) acc[i][jj][0] = acc[i][jj][1] = 0.0;
    }
    const double* as = sm.As[bufi] + (wr * 16 + (lane >> 2)) * LDA_S + (lane & 3);
    const double* bs = sm.Bs[bufi] + (lane & 3) * LDB_S + wc * 32 + (lane >> 2);
#pragma unroll
    for (int ks = 0; ks < KC / 4; ++ks) {
      double af[2], bf[4];
#pragma unroll
      for (int i = 0; i < 2; ++i) af[i] = as[i * 8 * LDA_S + ks * 4];
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) bf[jj] = bs[ks * 4 * LDB_S + jj * 8];
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) dmma884(acc[i][jj][0], acc[i][jj][1], af[i], bf[jj]);
    }
    if (c == kc - 1) {   // tile finished: write / update C straight from the accumulator fragments
      const int ti = t / tn, tj = t - ti * tn;
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const int gr = ti * 64 + wr * 16 + i * 8 + (lane >> 2);
        if (gr >= m) continue;
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
          const int gc = tj * 64 + wc * 32 + jj * 8 + 2 * (lane & 3);
          double* pc = Cm + (size_t)gr * ldc + gc;
          // (starting the accumulator from C instead - no read-modify-write here - is 1.5 % faster on the north
          // sweep's Np <= 160 and 9 % slower on the south sweep's Np ~ 300: not worth a second path)
          if (gc < n2) pc[0] = mode ? pc[0] - acc[i][jj][0] : acc[i][jj][0];
          if (gc + 1 < n2) pc[1] = mode ? pc[1] - acc[i][jj][1] : acc[i][jj][1];
        }
      }
    }
    if (step + 1 < nsteps) spark(bufi ^ 1);
    __syncthreads();
  }
}

// ||A||_1 = max column sum of |A| (Np x Np)
__device__ __noinline__ double cta_norm1(const double* __restrict__ A, int ld, int np_, Smem& sm) {
  double best = 0.0;
  for (int j = threadIdx.x; j < np_; j += GT) {
    double s = 0.0;
    for (int i = 0; i < np_; ++i) s += fabs(A[(size_t)i * ld + j]);
    best = fmax(best, s);
  }
  return block_max(best, sm);
}

// exact || (scale*|A|)^p ||_1 by p transposed mat-vecs on the ones vector (non-negative matrix)
__device__ __noinline__ double cta_absnorm_power(const double* __restrict__ A, int ld, int np_, double scale, int p,
                                    double* __restrict__ v0, double* __restrict__ v1, Smem& sm) {
  // every thread works: column j's dot product is split over `parts` row slices (thread = (slice, column)), the slice
  // partials go through shared memory (the GEMM staging buffer, idle here) and are added in slice order
  const int parts = (np_ <= GT / 8) ? 8 : (np_ <= GT / 4) ? 4 : (np_ <= GT / 2) ? 2 : 1;
  double* part = &sm.As[0][0];                       // [parts][np_] <= GT doubles
  const int jc = threadIdx.x % np_, sl = threadIdx.x / np_;
  for (int j = threadIdx.x; j < np_; j += GT) v0[j] = 1.0;
  __syncthreads();
  double* src = v0;
  double* dst = v1;
  for (int it = 0; it < p; ++it) {
    if (parts > 1) {
      if (sl < parts) {
        double s = 0.0;
#pragma unroll 4
        for (int i = sl; i < np_; i += parts) s = fma(scale * fabs(A[(size_t)i * ld + jc]), src[i], s);
        part[sl * np_ + jc] = s;
      }
      __syncthreads();
      if (threadIdx.x < np_) {
        double s = part[threadIdx.x];
        for (int q = 1; q < parts; ++q) s += part[q * np_ + threadIdx.x];
        dst[threadIdx.x] = s;
      }
    } else {
      for (int j = threadIdx.x; j < np_; j += GT) {
        double s = 0.0;
#pragma unroll 4
        for (int i = 0; i < np_; ++i) s = fma(scale * fabs(A[(size_t)i * ld + j]), src[i], s);
        dst[j] = s;
      }
    }
    __syncthreads();
    double* t = src; src = dst; dst = t;
  }
  double best = 0.0;
  for (int j = threadIdx.x; j < np_; j += GT) best = fmax(best, src[j]);
  return block_max(best, sm);
}

__device__ __forceinline__ int ell_of(double t, double normA, int idx, int m) {
  // lm = max(ceil(log2(t / normA / coeff) / (2m)), 0)
  if (!(t > 0.0)) return 0;
  const double val = ceil(log2(t / normA / kCoeff[idx]) / (double)(2 * m));
  if (val != val) return 1 << 20;
  if (val > 1.0e6) return 1 << 20;
  return val > 0.0 ? (int)val : 0;
}

// dst = c0*I + c1*P1 + c2*P2 + c3*P3 (+ add) ; any pointer may be null
__device__ __noinline__ void cta_lincomb(double* __restrict__ dst, int ld, int np_, double cI, const double* P1, double c1,
                            const double* P2, double c2, const double* P3, double c3, const double* add) {
#pragma unroll 4
  for (int idx = threadIdx.x; idx < np_ * np_; idx += GT) {
    const int i = idx / np_, jj = idx - i * np_;
    const size_t o = (size_t)i * ld + jj;
    double v = (i == jj) ? cI : 0.0;
    if (P1) v += c1 * P1[o];
    if (P2) v += c2 * P2[o];
    if (P3) v += c3 * P3[o];
    if (add) v += add[o];
    dst[o] = v;
  }
  __syncthreads();
}

// Solve P X = Q in place (X overwrites Q): right-looking blocked LU with partial pivoting (panel width 16, the
// panel factored in shared memory, trailing updates of [P | Q] as rank-16 DMMA GEMMs), then a blocked back
// substitution.  P is destroyed.  Same algorithm family as LAPACK dgesv (scipy's solve step inside expm).
__device__ __noinline__ void cta_lu_solve(double* __restrict__ P, double* __restrict__ Q, int ld, int np_, Smem& sm) {
  const int tid = threadIdx.x;
  double* pan = sm.u.panel;                       // [rows][PANEL]
  for (int k0 = 0; k0 < np_; k0 += PANEL) {
    const int kb = min(PANEL, np_ - k0);
    const int rows = np_ - k0;
    for (int idx = tid; idx < rows * PANEL; idx += GT) {
      const int r = idx / PANEL, c = idx - r * PANEL;
      pan[idx] = (c < kb) ? P[(size_t)(k0 + r) * ld + k0 + c] : 0.0;
    }
    __syncthreads();
    for (int c = 0; c < kb; ++c) {
      double bv = -1.0; int bi = c;
      for (int r = c + tid; r < rows; r += GT) {
        const double a = fabs(pan[r * PANEL + c]);
        if (a > bv) { bv = a; bi = r; }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
      }
      if ((tid & 31) == 0) { sm.red[tid >> 5] = bv; sm.ired[tid >> 5] = bi; }
      __syncthreads();
      bv = sm.red[0]; bi = sm.ired[0];
#pragma unroll
      for (int w = 1; w < GT / 32; ++w)
        if (sm.red[w] > bv || (sm.red[w] == bv && sm.ired[w] < bi)) { bv = sm.red[w]; bi = sm.ired[w]; }
      if (tid == 0) sm.piv[c] = bi;
      if (bi != c && tid < PANEL) {
        const double t = pan[c * PANEL + tid]; pan[c * PANEL + tid] = pan[bi * PANEL + tid]; pan[bi * PANEL + tid] = t;
      }
      __syncthreads();
      const double inv = 1.0 / pan[c * PANEL + c];
      for (int r = c + 1 + tid; r < rows; r += GT) pan[r * PANEL + c] *= inv;
      __syncthreads();
      const int cw = kb - c - 1;
      if (cw > 0) {
        for (int idx = tid; idx < (rows - c - 1) * cw; idx += GT) {
          const int r = c + 1 + idx / cw, c2 = c + 1 + idx % cw;
          pan[r * PANEL + c2] = fma(-pan[r * PANEL + c], pan[c * PANEL + c2], pan[r * PANEL + c2]);
        }
      }
      __syncthreads();
    }
    // panel back to global; row swaps + L11^-1 applied to the columns right of the panel and to all of Q
    for (int idx = tid; idx < rows * kb; idx += GT) {
      const int r = idx / kb, c = idx - r * kb;
      P[(size_t)(k0 + r) * ld + k0 + c] = pan[r * PANEL + c];
    }
    const int rightw = np_ - k0 - kb;
    for (int col = tid; col < rightw + np_; col += GT) {
      double* base = (col < rightw) ? P + (k0 + kb + col) : Q + (col - rightw);
      for (int c = 0; c < kb; ++c) {
        const int pr = sm.piv[c];
        if (pr != c) {
          const double t = base[(size_t)(k0 + c) * ld]; base[(size_t)(k0 + c) * ld] = base[(size_t)(k0 + pr) * ld];
          base[(size_t)(k0 + pr) * ld] = t;
        }
      }
      double x[PANEL];
#pragma unroll
      for (int c = 0; c < PANEL; ++c) x[c] = (c < kb) ? base[(size_t)(k0 + c) * ld] : 0.0;
#pragma unroll
      for (int c = 1; c < PANEL; ++c) {
        if (c < kb) {
          double sacc = x[c];
#pragma unroll
          for (int d = 0; d < PANEL; ++d)
            if (d < c) sacc = fma(-pan[c * PANEL + d], x[d], sacc);
          x[c] = sacc;
        }
      }
#pragma unroll
      for (int c = 0; c < PANEL; ++c)
        if (c < kb) base[(size_t)(k0 + c) * ld] = x[c];
    }
    __syncthreads();
    const int below = np_ - k0 - kb;
    if (below > 0) {
      const double* L21 = P + (size_t)(k0 + kb) * ld + k0;
      cta_gemm(P + (size_t)(k0 + kb) * ld + k0 + kb, ld, L21, ld, P + (size_t)k0 * ld + k0 + kb, ld, below, kb, rightw,
               sm, 1);
      cta_gemm(Q + (size_t)(k0 + kb) * ld, ld, L21, ld, Q + (size_t)k0 * ld, ld, below, kb, np_, sm, 1);
    }
  }
  // back substitution U X = Y, block rows from the bottom
  const int nblk = (np_ + PANEL - 1) / PANEL;
  for (int b = nblk - 1; b >= 0; --b) {
    const int k0 = b * PANEL, kb = min(PANEL, np_ - k0);
    for (int idx = tid; idx < PANEL * PANEL; idx += GT) {
      const int r = idx / PANEL, c = idx - r * PANEL;
      pan[idx] = (r < kb && c < kb) ? P[(size_t)(k0 + r) * ld + k0 + c] : 0.0;
    }
    __syncthreads();
    for (int col = tid; col < np_; col += GT) {
      double x[PANEL];
#pragma unroll
      for (int c = 0; c < PANEL; ++c) x[c] = (c < kb) ? Q[(size_t)(k0 + c) * ld + col] : 0.0;
#pragma unroll
      for (int c = PANEL - 1; c >= 0; --c) {
        if (c < kb) {
          double sacc = x[c];
#pragma unroll
          for (int d = 0; d < PANEL; ++d)
            if (d > c && d < kb) sacc = fma(-pan[c * PANEL + d], x[d], sacc);
          x[c] = sacc / pan[c * PANEL + c];
        }
      }
#pragma unroll
      for (int c = 0; c < PANEL; ++c)
        if (c < kb) Q[(size_t)(k0 + c) * ld + col] = x[c];
    }
    __syncthreads();
    if (k0 > 0) cta_gemm(Q, ld, P + k0, ld, Q + (size_t)k0 * ld, ld, k0, kb, np_, sm, 1);
  }
}

// expm(A) for the Np x Np matrix in buf[1]; buf[0..8] are Np x Np slabs (ld).  Returns pointer to result.
__device__ __noinline__ double* cta_expm(double** buf, int ld, int np_, double* v0, double* v1, int* m_out, int* s_out,
                            Smem& sm) {
  double* A = buf[1]; double* A2 = buf[2]; double* A4 = buf[3]; double* A6 = buf[4];
  double* B5 = buf[5]; double* B6 = buf[6]; double* B7 = buf[7]; double* B8 = buf[8];
  long long gp_t_last = clock64();
  (void)gp_t_last;
  cta_gemm(A2, ld, A, ld, A, ld, np_, np_, np_, sm);
  cta_gemm(A4, ld, A2, ld, A2, ld, np_, np_, np_, sm);
  cta_gemm(A6, ld, A4, ld, A2, ld, np_, np_, np_, sm);
  const double normA = cta_norm1(A, ld, np_, sm);
  const double d4 = pow(cta_norm1(A4, ld, np_, sm), 0.25);
  const double d6 = pow(cta_norm1(A6, ld, np_, sm), 1.0 / 6.0);
  const double eta0 = fmax(d4, d6);
  GP_TICK(1);                               // A^2, A^4, A^6 and their norms
  int m = 0, s = 0;
  if (eta0 < kTheta[0] && ell_of(cta_absnorm_power(A, ld, np_, 1.0, 7, v0, v1, sm), normA, 0, 3) == 0) m = 3;
  if (!m && eta0 < kTheta[1] && ell_of(cta_absnorm_power(A, ld, np_, 1.0, 11, v0, v1, sm), normA, 1, 5) == 0) m = 5;
  double d8 = 0.0, eta2 = 0.0;
  if (!m) {
    cta_gemm(B5, ld, A4, ld, A4, ld, np_, np_, np_, sm);   // A^8
    d8 = pow(cta_norm1(B5, ld, np_, sm), 0.125);
    eta2 = fmax(d6, d8);
    if (eta2 < kTheta[2] && ell_of(cta_absnorm_power(A, ld, np_, 1.0, 15, v0, v1, sm), normA, 2, 7) == 0) m = 7;
    if (!m && eta2 < kTheta[3] && ell_of(cta_absnorm_power(A, ld, np_, 1.0, 19, v0, v1, sm), normA, 3, 9) == 0) m = 9;
  }
  GP_TICK(2);                               // order selection: A^8 and the |A|^p power iterations of orders 3..9
  double* U = B7; double* V = B8;
  if (m == 3) {
    cta_lincomb(B5, ld, np_, kB3[1], A2, kB3[3], nullptr, 0, nullptr, 0, nullptr);
    cta_gemm(U, ld, A, ld, B5, ld, np_, np_, np_, sm);
    cta_lincomb(V, ld, np_, kB3[0], A2, kB3[2], nullptr, 0, nullptr, 0, nullptr);
  } else if (m == 5) {
    cta_lincomb(B5, ld, np_, kB5[1], A4, kB5[5], A2, kB5[3], nullptr, 0, nullptr);
    cta_gemm(U, ld, A, ld, B5, ld, np_, np_, np_, sm);
    cta_lincomb(V, ld, np_, kB5[0], A4, kB5[4], A2, kB5[2], nullptr, 0, nullptr);
  } else if (m == 7) {
    cta_lincomb(B5, ld, np_, kB7[1], A6, kB7[7], A4, kB7[5], A2, kB7[3], nullptr);
    cta_gemm(U, ld, A, ld, B5, ld, np_, np_, np_, sm);
    cta_lincomb(V, ld, np_, kB7[0], A6, kB7[6], A4, kB7[4], A2, kB7[2], nullptr);
  } else if (m == 9) {
    // B5 holds A^8
    cta_lincomb(B6, ld, np_, kB9[1], A6, kB9[7], A4, kB9[5], A2, kB9[3], nullptr);
    for (int idx = threadIdx.x; idx < np_ * np_; idx += GT) {
      const int i = idx / np_, jj = idx - i * np_; const size_t o = (size_t)i * ld + jj;
      B6[o] += kB9[9] * B5[o];
    }
    __syncthreads();
    cta_gemm(U, ld, A, ld, B6, ld, np_, np_, np_, sm);
    cta_lincomb(V, ld, np_, kB9[0], A6, kB9[6], A4, kB9[4], A2, kB9[2], nullptr);
    for (int idx = threadIdx.x; idx < np_ * np_; idx += GT) {
      const int i = idx / np_, jj = idx - i * np_; const size_t o = (size_t)i * ld + jj;
      V[o] += kB9[8] * B5[o];
    }
    __syncthreads();
  } else {
    m = 13;
    cta_gemm(B6, ld, A4, ld, A6, ld, np_, np_, np_, sm);   // A^10
    const double d10 = pow(cta_norm1(B6, ld, np_, sm), 0.1);
    const double eta3 = fmax(d8, d10), eta4 = fmin(eta2, eta3);
    double sv = ceil(log2(eta4 / kTheta[4]));
    s = (sv > 0.0) ? (int)sv : 0;
    if (!(sv == sv) || sv > 2000.0) s = 2000;
    const double sc = ldexp(1.0, -s);
    GP_TICK(2);
    s += ell_of(cta_absnorm_power(A, ld, np_, sc, 27, v0, v1, sm), normA * sc, 4, 13);
    GP_TICK(3);                             // the 27-step |A|^27 power iteration of order 13
    if (s > 2000) s = 2000;
    const double s1 = ldexp(1.0, -s), s2 = ldexp(1.0, -2 * s), s4 = ldexp(1.0, -4 * s), s6 = ldexp(1.0, -6 * s);
#pragma unroll 2
    for (int idx = threadIdx.x; idx < np_ * np_; idx += GT) {
      const int i = idx / np_, jj = idx - i * np_; const size_t o = (size_t)i * ld + jj;
      A[o] *= s1; A2[o] *= s2; A4[o] *= s4; A6[o] *= s6;
    }
    __syncthreads();
    cta_lincomb(B5, ld, np_, 0.0, A6, kB13[13], A4, kB13[11], A2, kB13[9], nullptr);
    cta_gemm(B6, ld, A6, ld, B5, ld, np_, np_, np_, sm);                                   // U2
    cta_lincomb(B5, ld, np_, kB13[1], A6, kB13[7], A4, kB13[5], A2, kB13[3], B6);
    cta_gemm(U, ld, A, ld, B5, ld, np_, np_, np_, sm);
    cta_lincomb(B5, ld, np_, 0.0, A6, kB13[12], A4, kB13[10], A2, kB13[8], nullptr);
    cta_gemm(B6, ld, A6, ld, B5, ld, np_, np_, np_, sm);                                   // V2
    cta_lincomb(V, ld, np_, kB13[0], A6, kB13[6], A4, kB13[4], A2, kB13[2], B6);
  }
  GP_TICK(4);                               // Pade numerator / denominator (element-wise passes + 1-3 GEMMs)
  // P = V - U -> B5 ; Q = V + U -> B6 ; solve P X = Q
#pragma unroll 4
  for (int idx = threadIdx.x; idx < np_ * np_; idx += GT) {
    const int i = idx / np_, jj = idx - i * np_; const size_t o = (size_t)i * ld + jj;
    const double u = U[o], vv = V[o];
    B5[o] = vv - u; B6[o] = vv + u;
  }
  __syncthreads();
  cta_lu_solve(B5, B6, ld, np_, sm);
  GP_TICK(5);                               // LU solve
  double* Xc = B6; double* Xn = B7;
  for (int it = 0; it < s; ++it) {
    cta_gemm(Xn, ld, Xc, ld, Xc, ld, np_, np_, np_, sm);
    double* t = Xc; Xc = Xn; Xn = t;
  }
  GP_TICK(6);                               // s squarings
  *m_out = m; *s_out = s;
  return Xc;
}

// in-place lower Cholesky of the n x n matrix K (shared, ld LDS); returns 0 or the 1-based failing pivot
__device__ __noinline__ int cta_cholesky(double* K, int n, Smem& sm) {
  const int tid = threadIdx.x;
  for (int k = 0; k < n; ++k) {
    const double d = K[k * LDS + k];
    if (!(d > 0.0)) return k + 1;      // uniform: every thread reads the same value
    const double r = sqrt(d);
    __syncthreads();
    if (tid == 0) K[k * LDS + k] = r;
    for (int i = k + 1 + tid; i < n; i += GT) K[i * LDS + k] /= r;
    __syncthreads();
    const int rem = n - k - 1;
    for (int idx = tid; idx < rem * rem; idx += GT) {
      const int a = idx / rem, b = idx - a * rem;
      if (b <= a) {
        const int i = k + 1 + a, jj = k + 1 + b;
        K[i * LDS + jj] = fma(-K[i * LDS + k], K[jj * LDS + k], K[i * LDS + jj]);
      }
    }
    __syncthreads();
  }
  return 0;
}
// warp 0: forward substitution tmp = L^-1 b (row dot products split over the 32 lanes)
__device__ __forceinline__ void warp_fwd_solve(const double* L, int n, const double* b, double* tmp, int lane) {
  for (int i = 0; i < n; ++i) {
    double s = 0.0;
    for (int c = lane; c < i; c += 32) s = fma(L[i * LDS + c], tmp[c], s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) tmp[i] = (b[i] - s) / L[i * LDS + i];
    __syncwarp();
  }
}
// warp 0: backward substitution x = L^-T tmp
__device__ __forceinline__ void warp_bwd_solve(const double* L, int n, const double* tmp, double* x, int lane) {
  for (int i = n - 1; i >= 0; --i) {
    double s = 0.0;
    for (int c = i + 1 + lane; c < n; c += 32) s = fma(L[c * LDS + i], x[c], s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) x[i] = (tmp[i] - s) / L[i * LDS + i];
    __syncwarp();
  }
}
// x = L^-T L^-1 b
__device__ void cta_chol_solve(const double* L, int n, const double* b, double* x, double* tmp) {
  if (threadIdx.x < 32) {
    warp_fwd_solve(L, n, b, tmp, threadIdx.x);
    warp_bwd_solve(L, n, tmp, x, threadIdx.x);
  }
  __syncthreads();
}

// ---------------------------------------------------------------------------------------------------------------
// Warp-local fit for the hyper-parameter grid: one warp owns one (problem, l, sigma) evaluation -- its own n x n
// kernel matrix in shared memory (row stride ldw = n | 1), right-looking Cholesky with a row per lane, triangular
// solves with lane-split dot products -- so the 8 warps of a CTA factor 8 different sigma at once instead of taking
// turns at CTA-wide barriers.  Every element receives the same sequence of fma updates as in cta_cholesky (k = 0, 1,
// ... in order), so the factor is bit-identical to the CTA-wide path.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int warp_cholesky(double* K, int n, int ldw, int lane) {
  for (int k = 0; k < n; ++k) {
    const double d = K[k * ldw + k];
    if (!(d > 0.0)) return k + 1;          // uniform across the warp
    const double r = sqrt(d);
    __syncwarp();
    if (lane == 0) K[k * ldw + k] = r;
    for (int i = k + 1 + lane; i < n; i += 32) K[i * ldw + k] /= r;
    __syncwarp();
    for (int i = k + 1 + lane; i < n; i += 32) {
      const double aik = K[i * ldw + k];
      for (int jj = k + 1; jj <= i; ++jj) K[i * ldw + jj] = fma(-aik, K[jj * ldw + k], K[i * ldw + jj]);
    }
    __syncwarp();
  }
  return 0;
}
__device__ __forceinline__ void warp_fwd_solve_ld(const double* L, int n, int ldw, const double* b, double* tmp, int lane) {
  for (int i = 0; i < n; ++i) {
    double s = 0.0;
    for (int c = lane; c < i; c += 32) s = fma(L[i * ldw + c], tmp[c], s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) tmp[i] = (b[i] - s) / L[i * ldw + i];
    __syncwarp();
  }
}
__device__ __forceinline__ void warp_bwd_solve_ld(const double* L, int n, int ldw, const double* tmp, double* x, int lane) {
  for (int i = n - 1; i >= 0; --i) {
    double s = 0.0;
    for (int c = i + 1 + lane; c < n; c += 32) s = fma(L[c * ldw + i], x[c], s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) x[i] = (tmp[i] - s) / L[i * ldw + i];
    __syncwarp();
  }
}

// One (sigma) evaluation by one warp.  W: n x n (stride LDS, shared, read-only); y, kxs_raw: shared, read-only;
// Kw / vec: this warp's workspace (n x ldw and 4 x MAXN doubles); G1raw: X (M Sigma~) X^T (stride LDS, global) or null.
__device__ void warp_sigma_fit(const double* __restrict__ W, const double* __restrict__ y, const double* __restrict__ kxs_raw,
                               double kss_raw, const double* __restrict__ G1raw, int n, double sig, double* Kw, double* vec,
                               SieGpResult& res, long long clk_start, SieGpResult* outp) {
  const int lane = threadIdx.x & 31;
  const int ldw = n | 1;
  double* ya = vec; double* alpha = vec + MAXN; double* kxs = vec + 2 * MAXN; double* v = vec + 3 * MAXN;
  res.fmean = res.fvar = res.sigma_f = res.nlml = res.g_ell = res.g_sig = sie_nan();
  res.info = 0;
  for (int idx = lane; idx < n * n; idx += 32) {
    const int i = idx / n, jj = idx - i * n;
    Kw[i * ldw + jj] = W[i * LDS + jj] + ((i == jj) ? sig : 0.0);
  }
  __syncwarp();
  int info = warp_cholesky(Kw, n, ldw, lane);
  if (info) { if (lane == 0) { res.info = info; res.cycles_total = clock64() - clk_start; *outp = res; } return; }
  warp_fwd_solve_ld(Kw, n, ldw, y, v, lane);
  warp_bwd_solve_ld(Kw, n, ldw, v, ya, lane);
  double sf = 0.0;
  for (int t = 0; t < n; ++t) sf = fma(y[t], ya[t], sf);
  sf /= (double)n;
  const double sn = sf * sig;
  res.sigma_f = sf;
  __syncwarp();
  for (int idx = lane; idx < n * n; idx += 32) {
    const int i = idx / n, jj = idx - i * n;
    Kw[i * ldw + jj] = sf * W[i * LDS + jj] + ((i == jj) ? sn : 0.0);
  }
  __syncwarp();
  info = warp_cholesky(Kw, n, ldw, lane);
  if (info) { if (lane == 0) { res.info = info; res.cycles_total = clock64() - clk_start; *outp = res; } return; }
  warp_fwd_solve_ld(Kw, n, ldw, y, v, lane);
  warp_bwd_solve_ld(Kw, n, ldw, v, alpha, lane);
  for (int i = lane; i < n; i += 32) kxs[i] = sf * kxs_raw[i];
  __syncwarp();
  const double kss = sf * kss_raw + sn;
  warp_fwd_solve_ld(Kw, n, ldw, kxs, v, lane);
  double vv = 0.0, fm = 0.0, yal = 0.0, ld_sum = 0.0;
  for (int i = lane; i < n; i += 32) {
    vv = fma(v[i], v[i], vv);
    fm = fma(kxs[i], alpha[i], fm);
    yal = fma(y[i], alpha[i], yal);
    ld_sum += log(Kw[i * ldw + i]);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    vv += __shfl_xor_sync(0xffffffffu, vv, o);
    fm += __shfl_xor_sync(0xffffffffu, fm, o);
    yal += __shfl_xor_sync(0xffffffffu, yal, o);
    ld_sum += __shfl_xor_sync(0xffffffffu, ld_sum, o);
  }
  res.fmean = fm; res.fvar = kss - vv;
  res.nlml = yal / 2 + ld_sum + n * log(2 * 3.141592653589793238462643383279502884) / 2;
  if (G1raw) {
    // MLII gradient as written (:248-252): dK/dl = sf G1raw + sn I, dK/dsigma = sf W + sf I
    for (int which = 0; which < 2; ++which) {
      auto dK = [&](int i, int jj) -> double {
        return which == 0 ? sf * G1raw[i * LDS + jj] + ((i == jj) ? sn : 0.0) : sf * W[i * LDS + jj] + ((i == jj) ? sf : 0.0);
      };
      double quad = 0.0;
      for (int idx = lane; idx < n * n; idx += 32) {
        const int i = idx / n, jj = idx - i * n;
        quad = fma(alpha[i] * dK(i, jj), alpha[jj], quad);
      }
      double tr = 0.0;
      for (int jj = lane; jj < n; jj += 32) {          // column jj of K^-1 dK, down to its diagonal entry
        double col[MAXN];
        for (int i = 0; i < n; ++i) {
          double sacc = dK(i, jj);
          for (int c = 0; c < i; ++c) sacc = fma(-Kw[i * ldw + c], col[c], sacc);
          col[i] = sacc / Kw[i * ldw + i];
        }
        for (int i = n - 1; i >= jj; --i) {
          double sacc = col[i];
          for (int c = i + 1; c < n; ++c) sacc = fma(-Kw[c * ldw + i], col[c], sacc);
          col[i] = sacc / Kw[i * ldw + i];
        }
        tr += col[jj];
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        quad += __shfl_xor_sync(0xffffffffu, quad, o);
        tr += __shfl_xor_sync(0xffffffffu, tr, o);
      }
      const double gval = tr / 2 - quad / 2;
      if (which == 0) res.g_ell = gval; else res.g_sig = gval;
    }
  }
  if (lane == 0) { res.cycles_total = clock64() - clk_start; *outp = res; }
}

__global__ void __launch_bounds__(GT, 2)
k_gp_forecast(const SieGpProblem* __restrict__ prob, int P, const double* __restrict__ y_all,
              const double* __restrict__ anom_sic, const int32_t* __restrict__ n_areas_sic, int ma_sic, int ts_sic,
              const double* __restrict__ anom_sst, const int32_t* __restrict__ n_areas_sst, int ma_sst, int ts_sst,
              int max_pred, SieGpResult* __restrict__ out, unsigned char* __restrict__ scratch, size_t per_cta,
              const int32_t* __restrict__ order, int* __restrict__ queue, const double* __restrict__ sig_grid,
              int n_sig) {
  // hyper-parameter grid mode (sig_grid != nullptr): problem p is one (network set, region, l); Sigma~ = expm(l M) and
  // W = X Sigma~ X^T are built once and the Cholesky fit / nlML is repeated for the n_sig noise values; results go to
  // out[p * n_sig + k].  Otherwise n_sig = 1, sigma_n~ = prob[p].sig and the result goes to out[p].
  const int ns = sig_grid ? n_sig : 1;
  extern __shared__ __align__(16) unsigned char smraw[];
  Smem& sm = *reinterpret_cast<Smem*>(smraw);
  const int tid = threadIdx.x;
  const int ld = max_pred;
  unsigned char* sp = scratch + (size_t)blockIdx.x * per_cta;
  double* buf[9];
  for (int i = 0; i < 9; ++i) buf[i] = reinterpret_cast<double*>(sp) + (size_t)i * ld * ld;
  double* Xg = reinterpret_cast<double*>(sp) + (size_t)9 * ld * ld;   // (n+1) x Np, ld
  double* XE = Xg + (size_t)MAXN * ld;                                 // n x Np
  double* XM = XE + (size_t)MAXN * ld;                                 // n x Np (gradient)
  double* v0 = XM + (size_t)MAXN * ld;
  double* v1 = v0 + ld;
  double* colm = v1 + ld;                                              // column means / scratch [ld]
  double* Gg = colm + ld;                                              // [MAXN*LDS] gradient scratch
  int* sel = reinterpret_cast<int*>(Gg + MAXN * LDS);                  // [ld] selected series (sign in bit 30)

  // dynamic work queue over problems pre-ordered by expected cost (largest first)
  while (true) {
    __syncthreads();
    if (tid == 0) sm.misc[7] = atomicAdd(queue, 1);
    __syncthreads();
    const int qi = sm.misc[7];
    if (qi >= P) break;
    const int p = order ? order[qi] : qi;
    const SieGpProblem pr = prob[p];
    const int n = pr.n;
    SieGpResult res;
    res.fmean = res.fvar = res.sigma_f = res.nlml = res.g_ell = res.g_sig = sie_nan();
    res.n_pred = 0; res.expm_m = 0; res.expm_s = 0; res.info = 0;
    res.cycles_total = 0; res.cycles_expm = 0;
    const long long clk_start = clock64();
    long long gp_t_last = clk_start;
    (void)gp_t_last;
    __syncthreads();
    if (n < 2 || n + 1 > MAXN) {
      if (tid == 0) { res.info = -2; for (int k = 0; k < ns; ++k) out[(size_t)p * ns + k] = res; }
      continue;
    }
    const int na1 = n_areas_sic[pr.job_sic];
    const int na2 = (pr.job_sst >= 0) ? n_areas_sst[pr.job_sst] : 0;
    const double* s1 = anom_sic + (size_t)pr.job_sic * ma_sic * ts_sic;
    const double* s2 = (pr.job_sst >= 0) ? anom_sst + (size_t)pr.job_sst * ma_sst * ts_sst : nullptr;
    // ---- y, centred/normalised copy for pearsonr (scipy: xm/||xm|| . ym/||ym||)
    for (int t = tid; t < n; t += GT) sm.y[t] = y_all[pr.y_off + t];
    __syncthreads();
    double ymean = 0.0;
    for (int t = 0; t < n; ++t) ymean += sm.y[t];
    ymean /= (double)n;
    double ynorm = 0.0;
    for (int t = 0; t < n; ++t) { const double d = sm.y[t] - ymean; ynorm = fma(d, d, ynorm); }
    ynorm = sqrt(ynorm);
    // ---- predictor selection (north/June1st.py:216-224)
    if (tid == 0) sm.misc[0] = 0;
    __syncthreads();
    for (int c0 = 0; c0 < na1 + na2; c0 += GT) {
      const int c = c0 + tid;
      int flag = 0;   // 0 no, 1 take, 2 take negated
      if (c < na1 + na2) {
        const bool sst = c >= na1;
        const double* x = sst ? s2 + (size_t)(c - na1) * ts_sst : s1 + (size_t)c * ts_sic;
        double xm = 0.0;
        for (int t = 0; t < n; ++t) xm += x[t];
        xm /= (double)n;
        double xn = 0.0, dot = 0.0;
        for (int t = 0; t < n; ++t) { const double d = x[t] - xm; xn = fma(d, d, xn); dot = fma(d, sm.y[t] - ymean, dot); }
        double r = dot / (sqrt(xn) * ynorm);
        // pearsonr clips to [-1, 1]; a constant series gives NaN, which must stay NaN (fmin/fmax would return the
        // non-NaN operand): `r > 0` / `r < 0` then reject it like the reference does
        if (r == r) r = fmax(-1.0, fmin(1.0, r));
        if (sst) flag = (r < 0.0) ? 2 : 0;
        else if (pr.rule == 1) flag = 1;
        else if (pr.rule == 0) flag = (r > 0.0) ? 1 : 0;
        else flag = (r > 0.0 && r > pr.r_sel) ? 1 : 0;
      }
      // order-preserving compaction across the CTA
      const unsigned bal = __ballot_sync(0xffffffffu, flag != 0);
      const int lane = tid & 31, w = tid >> 5;
      if (lane == 0) sm.ired[w] = __popc(bal);
      __syncthreads();
      int off = sm.misc[0];
      for (int i = 0; i < w; ++i) off += sm.ired[i];
      if (flag) {
        const int pos = off + __popc(bal & ((1u << lane) - 1u));
        if (pos < ld) sel[pos] = c | (flag == 2 ? (1 << 30) : 0);
      }
      __syncthreads();
      if (tid == 0) { int tot = 0; for (int i = 0; i < GT / 32; ++i) tot += sm.ired[i]; sm.misc[0] += tot; }
      __syncthreads();
    }
    const int np_ = sm.misc[0];
    res.n_pred = np_;
    // fewer than two predictors: the reference's forecast() raises (no column: IndexError at `X[-1,:]`; one column:
    // np.cov is 0-d and np.fill_diagonal raises ValueError, north/June1st.py:228-232)
    if (np_ < 2 || np_ > ld) {
      if (tid == 0) { res.info = (np_ < 2) ? -1 : -2; for (int k = 0; k < ns; ++k) out[(size_t)p * ns + k] = res; }
      continue;
    }
    // ---- X (n+1 rows) with optional column z-score over all n+1 rows (:226-227)
    for (int c = tid; c < np_; c += GT) {
      const int sc = sel[c] & ~(1 << 30);
      const double sign = (sel[c] & (1 << 30)) ? -1.0 : 1.0;
      const double* x = (sc >= na1) ? s2 + (size_t)(sc - na1) * ts_sst : s1 + (size_t)sc * ts_sic;
      if (pr.zscore) {
        double mu = 0.0;
        for (int t = 0; t <= n; ++t) mu += sign * x[t];
        mu /= (double)(n + 1);
        double var = 0.0;
        for (int t = 0; t <= n; ++t) { const double d = sign * x[t] - mu; var = fma(d, d, var); }
        const double sd = sqrt(var / (double)(n + 1));
        for (int t = 0; t <= n; ++t) Xg[(size_t)t * ld + c] = (sign * x[t] - mu) / sd;
      } else {
        for (int t = 0; t <= n; ++t) Xg[(size_t)t * ld + c] = sign * x[t];
      }
      double cm = 0.0;                       // column mean over the n training rows for the covariance
      for (int t = 0; t < n; ++t) cm += Xg[(size_t)t * ld + c];
      colm[c] = cm / (double)n;
    }
    __syncthreads();
    // ---- M = |cov(X, bias=True)|, zero diagonal, diagonal = -column sums (:231-233) -> buf[0]
    double* M = buf[0];
    const double invn = 1.0 / (double)n;
    for (int idx = tid; idx < np_ * np_; idx += GT) {
      const int i = idx / np_, jj = idx - i * np_;
      double sacc = 0.0;
      if (i != jj) {
        const double mi = colm[i], mj = colm[jj];
        for (int t = 0; t < n; ++t) sacc = fma(Xg[(size_t)t * ld + i] - mi, Xg[(size_t)t * ld + jj] - mj, sacc);
        sacc = fabs(sacc * invn);
      }
      M[(size_t)i * ld + jj] = sacc;
    }
    __syncthreads();
    for (int jj = tid; jj < np_; jj += GT) {
      double sacc = 0.0;
      for (int i = 0; i < np_; ++i) sacc += M[(size_t)i * ld + jj];
      colm[jj] = sacc;
    }
    __syncthreads();
    for (int jj = tid; jj < np_; jj += GT) M[(size_t)jj * ld + jj] = -colm[jj];
    __syncthreads();
    // ---- Sigma~ = expm(l*M)
    for (int idx = tid; idx < np_ * np_; idx += GT) {
      const int i = idx / np_, jj = idx - i * np_;
      buf[1][(size_t)i * ld + jj] = pr.ell * M[(size_t)i * ld + jj];
    }
    __syncthreads();
    int em = 0, es = 0;
    GP_TICK(0);                             // selection, design matrix, Laplacian
    const long long clk_e0 = clock64();
    const double* E = cta_expm(buf, ld, np_, v0, v1, &em, &es, sm);
    res.expm_m = em; res.expm_s = es;
    res.cycles_expm = clock64() - clk_e0;
    gp_t_last = clock64();
    // ---- W = X Sigma~ X^T : XE = X E (n x Np), then W = XE X^T (n x n, shared)
    cta_gemm(XE, ld, Xg, ld, E, ld, n, np_, np_, sm);
    for (int idx = tid; idx < n * n; idx += GT) {
      const int i = idx / n, jj = idx - i * n;
      double sacc = 0.0;
      for (int c = 0; c < np_; ++c) sacc = fma(XE[(size_t)i * ld + c], Xg[(size_t)jj * ld + c], sacc);
      sm.u.gp.W[i * LDS + jj] = sacc;
    }
    __syncthreads();
    if (pr.want_grad) {        // sigma-independent part of the MLII gradient: X (M Sigma~) (:248)
      cta_gemm(buf[5], ld, M, ld, E, ld, np_, np_, np_, sm);
      cta_gemm(XM, ld, Xg, ld, buf[5], ld, n, np_, np_, sm);
    }
    if (sig_grid) {
      // ---- hyper-parameter grid: the sigma-independent pieces once, then one warp per sigma
      for (int i = tid; i < n; i += GT) {                      // KXXs / sf = X Sigma~ Xs^T
        double sacc = 0.0;
        for (int c = 0; c < np_; ++c) sacc = fma(XE[(size_t)i * ld + c], Xg[(size_t)n * ld + c], sacc);
        sm.kxs[i] = sacc;
      }
      double kss_part = 0.0;                                   // (KXsXs - sn) / sf = Xs Sigma~ Xs^T
      for (int c = tid; c < np_; c += GT) {
        double row = 0.0;
        for (int d = 0; d < np_; ++d) row = fma(Xg[(size_t)n * ld + d], E[(size_t)d * ld + c], row);
        kss_part = fma(row, Xg[(size_t)n * ld + c], kss_part);
      }
      const double kss_raw = block_sum(kss_part, sm);
      if (pr.want_grad) {                                      // X (M Sigma~) X^T, sigma-independent
        for (int idx = tid; idx < n * n; idx += GT) {
          const int i = idx / n, jj = idx - i * n;
          double sacc = 0.0;
          for (int c = 0; c < np_; ++c) sacc = fma(XM[(size_t)i * ld + c], Xg[(size_t)jj * ld + c], sacc);
          Gg[i * LDS + jj] = sacc;
        }
      }
      __syncthreads();
      // per-warp workspaces over the GEMM staging buffers and the (unused here) CTA-wide K: As | Bs | u.gp.K
      double* wsp = &sm.As[0][0];
      const size_t avail = (size_t)(&sm.u.gp.W[0] - wsp);
      const size_t per_warp = (size_t)n * (n | 1) + 4 * MAXN;
      int nwu = (int)(avail / per_warp);
      if (nwu > GT / 32) nwu = GT / 32;
      const int warp = tid >> 5;
      if (warp < nwu) {
        double* Kw = wsp + (size_t)warp * per_warp;
        for (int ks = warp; ks < ns; ks += nwu)
          warp_sigma_fit(sm.u.gp.W, sm.y, sm.kxs, kss_raw, pr.want_grad ? Gg : nullptr, n, sig_grid[ks], Kw,
                         Kw + (size_t)n * (n | 1), res, clk_start, out + (size_t)p * ns + ks);
      }
      continue;                                                // next problem (the loop head synchronises the CTA)
    }
    GP_TICK(7);                             // X E, W = X E X^T (+ gradient operands)
    for (int ks = 0; ks < ns; ++ks) {
    const double sig = sig_grid ? sig_grid[ks] : pr.sig;
    SieGpResult* const outp = out + (size_t)p * ns + ks;
    res.fmean = res.fvar = res.sigma_f = res.nlml = res.g_ell = res.g_sig = sie_nan();
    res.info = 0;
    __syncthreads();
    // ---- L~ = chol(W + sig I); A~ ; sigma_f = y^T A~ / n  (:265-267)
    for (int idx = tid; idx < n * n; idx += GT) {
      const int i = idx / n, jj = idx - i * n;
      sm.u.gp.K[i * LDS + jj] = sm.u.gp.W[i * LDS + jj] + ((i == jj) ? sig : 0.0);
    }
    __syncthreads();
    int info = cta_cholesky(sm.u.gp.K, n, sm);
    if (info) { if (tid == 0) { res.info = info; res.cycles_total = clock64() - clk_start; *outp = res; } continue; }
    cta_chol_solve(sm.u.gp.K, n, sm.y, sm.ya, sm.v);
    double sf = 0.0;
    for (int t = 0; t < n; ++t) sf = fma(sm.y[t], sm.ya[t], sf);
    sf /= (double)n;
    const double sn = sf * sig;
    res.sigma_f = sf;
    __syncthreads();
    // ---- L = chol(sf*W + sn I); alpha (:269-271)
    for (int idx = tid; idx < n * n; idx += GT) {
      const int i = idx / n, jj = idx - i * n;
      sm.u.gp.K[i * LDS + jj] = sf * sm.u.gp.W[i * LDS + jj] + ((i == jj) ? sn : 0.0);
    }
    __syncthreads();
    info = cta_cholesky(sm.u.gp.K, n, sm);
    if (info) { if (tid == 0) { res.info = info; res.cycles_total = clock64() - clk_start; *outp = res; } continue; }
    cta_chol_solve(sm.u.gp.K, n, sm.y, sm.alpha, sm.v);
    // ---- predictive mean / variance (:272-277)
    for (int i = tid; i < n; i += GT) {
      double sacc = 0.0;
      for (int c = 0; c < np_; ++c) sacc = fma(XE[(size_t)i * ld + c], Xg[(size_t)n * ld + c], sacc);
      sm.kxs[i] = sf * sacc;
    }
    __syncthreads();
    // KXsXs = xs Sigma xs^T + sn : thread per column of E, then a block sum
    double kss_part = 0.0;
    for (int c = tid; c < np_; c += GT) {
      double row = 0.0;
      for (int d = 0; d < np_; ++d) row = fma(Xg[(size_t)n * ld + d], E[(size_t)d * ld + c], row);
      kss_part = fma(row, Xg[(size_t)n * ld + c], kss_part);
    }
    const double kss = sf * block_sum(kss_part, sm) + sn;
    if (tid < 32) {
      warp_fwd_solve(sm.u.gp.K, n, sm.kxs, sm.v, tid);          // v = L^-1 KXXs
      double vv = 0.0, fm = 0.0, ya = 0.0, ld_sum = 0.0;
      for (int i = tid; i < n; i += 32) {
        vv = fma(sm.v[i], sm.v[i], vv);
        fm = fma(sm.kxs[i], sm.alpha[i], fm);
        ya = fma(sm.y[i], sm.alpha[i], ya);
        ld_sum += log(sm.u.gp.K[i * LDS + i]);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        vv += __shfl_xor_sync(0xffffffffu, vv, o);
        fm += __shfl_xor_sync(0xffffffffu, fm, o);
        ya += __shfl_xor_sync(0xffffffffu, ya, o);
        ld_sum += __shfl_xor_sync(0xffffffffu, ld_sum, o);
      }
      if (tid == 0) {
        sm.dmisc[0] = fm; sm.dmisc[1] = kss - vv;
        sm.dmisc[2] = ya / 2 + ld_sum + n * log(2 * 3.141592653589793238462643383279502884) / 2;
      }
    }
    __syncthreads();
    res.fmean = sm.dmisc[0]; res.fvar = sm.dmisc[1]; res.nlml = sm.dmisc[2];
    // ---- MLII gradient as written at :248-252
    if (pr.want_grad) {
      // dKdl = X (M Sigma) X^T + sn I, Sigma = sf * E  (XM = X M Sigma~ was formed before the sigma loop)
      for (int which = 0; which < 2; ++which) {
        for (int idx = tid; idx < n * n; idx += GT) {
          const int i = idx / n, jj = idx - i * n;
          double val;
          if (which == 0) {
            double sacc = 0.0;
            for (int c = 0; c < np_; ++c) sacc = fma(XM[(size_t)i * ld + c], Xg[(size_t)jj * ld + c], sacc);
            val = sf * sacc + ((i == jj) ? sn : 0.0);
          } else {
            val = sf * sm.u.gp.W[i * LDS + jj] + ((i == jj) ? sf : 0.0);
          }
          Gg[i * LDS + jj] = val;
        }
        __syncthreads();
        // quad = alpha^T dK alpha ; trace(K^-1 dK) by solving column by column (thread per column)
        double quad = 0.0;
        for (int idx = tid; idx < n * n; idx += GT) {
          const int i = idx / n, jj = idx - i * n;
          quad = fma(sm.alpha[i] * Gg[i * LDS + jj], sm.alpha[jj], quad);
        }
        quad = block_sum(quad, sm);
        double tr = 0.0;
        if (tid < n) {
          double col[MAXN];
          const int jj = tid;
          for (int i = 0; i < n; ++i) {
            double sacc = Gg[i * LDS + jj];
            for (int c = 0; c < i; ++c) sacc = fma(-sm.u.gp.K[i * LDS + c], col[c], sacc);
            col[i] = sacc / sm.u.gp.K[i * LDS + i];
          }
          for (int i = n - 1; i >= jj; --i) {
            double sacc = col[i];
            for (int c = i + 1; c < n; ++c) sacc = fma(-sm.u.gp.K[c * LDS + i], col[c], sacc);
            col[i] = sacc / sm.u.gp.K[i * LDS + i];
          }
          tr = col[jj];
        }
        tr = block_sum(tr, sm);
        const double gval = tr / 2 - quad / 2;
        if (which == 0) res.g_ell = gval; else res.g_sig = gval;
        __syncthreads();
      }
    }
    GP_TICK(8);                             // two Cholesky factorisations, solves, predictive mean / variance (+ gradient)
    if (tid == 0) { res.cycles_total = clock64() - clk_start; *outp = res; }
    }   // sigma loop
  }
}

// Orders problems by descending candidate-predictor count (a proxy for Np^3 expm cost) with a one-CTA counting
// sort and resets the work-queue counter, so the biggest problems start first (LPT) on the persistent grid.
constexpr int ORDER_BUCKETS = 2048;
__global__ void __launch_bounds__(1024) k_gp_order(const SieGpProblem* __restrict__ prob, int P,
                                                  const int32_t* __restrict__ n_areas_sic,
                                                  const int32_t* __restrict__ n_areas_sst, int32_t* __restrict__ order,
                                                  int* __restrict__ queue) {
  __shared__ int hist[ORDER_BUCKETS];
  for (int i = threadIdx.x; i < ORDER_BUCKETS; i += blockDim.x) hist[i] = 0;
  __syncthreads();
  auto bucket = [&](int p) {
    const SieGpProblem pr = prob[p];
    int na = n_areas_sic[pr.job_sic] + ((pr.job_sst >= 0 && n_areas_sst) ? n_areas_sst[pr.job_sst] : 0);
    if (pr.rule == 2) na = na / 2;                     // significance-filtered problems select fewer series
    na = max(0, min(na, ORDER_BUCKETS - 1));
    return ORDER_BUCKETS - 1 - na;                     // descending cost
  };
  for (int p = threadIdx.x; p < P; p += blockDim.x) atomicAdd(&hist[bucket(p)], 1);
  __syncthreads();
  if (threadIdx.x == 0) {
    int acc = 0;
    for (int i = 0; i < ORDER_BUCKETS; ++i) { const int c = hist[i]; hist[i] = acc; acc += c; }
    *queue = 0;
  }
  __syncthreads();
  for (int p = threadIdx.x; p < P; p += blockDim.x) order[atomicAdd(&hist[bucket(p)], 1)] = p;
}

// Grid minimum of MLII per problem (sie_gp_grid_select, and the weight maximum of sie_gp_grid_marginal).  One warp per
// problem; lanes stride over the n grid records reading only nlml / info.  Each lane keeps the first of its smallest
// admissible values (its indices ascend), then the (value, flat index) pairs are reduced lexicographically with
// shuffles -- an associative, commutative min, so every lane ends with np.argmin's answer whatever the reduction order
// (-0.0 == 0.0 resolves to the smaller index).  bi = SEL_NONE, bv = +inf when no record is admissible.
constexpr int SEL_WARPS = 8;
constexpr int SEL_NONE = 0x7fffffff;
__device__ __forceinline__ bool gp_grid_admissible(const SieGpResult* r, double& nlml) {
  nlml = __ldg(&r->nlml);
  return __ldg(&r->info) == 0 && isfinite(nlml);
}
__device__ __forceinline__ void gp_grid_argmin_warp(const SieGpResult* __restrict__ g, int n, int lane, double& bv,
                                                    int& bi) {
  bv = __longlong_as_double(0x7ff0000000000000LL);   // +inf: no admissible point seen
  bi = SEL_NONE;
  for (int k = lane; k < n; k += 32) {
    double v;
    if (gp_grid_admissible(&g[k], v) && v < bv) { bv = v; bi = k; }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    const double ov = __shfl_xor_sync(0xffffffffu, bv, off);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, off);
    if (ov < bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
  }
}

__global__ void __launch_bounds__(SEL_WARPS * 32)
k_gp_grid_select(const SieGpResult* __restrict__ grid, const SieGpProblem* __restrict__ prob, int P,
                 const double* __restrict__ ell_grid, int n_ell, const double* __restrict__ sig_grid, int n_sig,
                 SieGpProblem* __restrict__ tuned, int32_t* __restrict__ best) {
  const int p = blockIdx.x * SEL_WARPS + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (p >= P) return;                                  // whole warp: p is uniform across it
  const int n = n_ell * n_sig;
  double bv;
  int bi;
  gp_grid_argmin_warp(grid + (size_t)p * n, n, lane, bv, bi);
  if (lane == 0) {
    SieGpProblem t = prob[p];
    if (bi != SEL_NONE) { t.ell = ell_grid[bi / n_sig]; t.sig = sig_grid[bi % n_sig]; }
    tuned[p] = t;
    best[p] = bi == SEL_NONE ? -1 : bi;
  }
}

// Grid marginal of the forecast per problem (sie_gp_grid_marginal).  One warp per problem, like k_gp_grid_select:
//   1. m = min admissible nlml and its flat index (gp_grid_argmin_warp: the argmax of the weights is grid_select's best)
//   2. e_k = exp(m - nlml_k) (0 outside A, 1 at the minimum), S0 = sum e, sum e^2, sum e mu, |A|
//   3. fvar = sum e (v + (mu - fmean)^2) / S0 (second pass over the centred means)
//   4. quantiles of the mixture CDF by bisection, F evaluated by the whole warp
// Every sum is a per-lane sum over k = lane, lane + 32, ... (fixed order) followed by a fixed xor-shuffle tree; IEEE
// addition commutes, so all 32 lanes hold the same bits and every branch on a reduced value is warp-uniform.  The
// (e, mu, sd) of up to MARG_STAGE grid points are staged in shared memory for the bisection; a larger grid recomputes
// them from the records at each step, with the same arithmetic, so both give the same bits.
constexpr int MARG_WARPS = 4;
constexpr int MARG_STAGE = 500;     // 4 warps x 500 points x 3 doubles = 48000 B of static shared memory per CTA

__device__ __forceinline__ double warp_sum_xor(double v) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v = __dadd_rn(v, __shfl_xor_sync(0xffffffffu, v, off));
  return v;
}

// Component k of the mixture: weight e (0 when k is not admissible or its weight underflows), mean, standard deviation
// (0: v <= 0, a point mass at mu).  Reads fmean / fvar only for admissible points.
__device__ __forceinline__ bool marg_component(const SieGpResult* __restrict__ r, double m, double& e, double& mu,
                                               double& sd) {
  double v;
  e = 0.0; mu = 0.0; sd = 0.0;
  if (!gp_grid_admissible(r, v)) return false;
  e = exp(m - v);
  mu = __ldg(&r->fmean);
  const double var = __ldg(&r->fvar);
  sd = var > 0.0 ? sqrt(var) : 0.0;
  return true;
}

// Passes 1-2 of one grid's marginal (k_gp_grid_marginal, and every member of k_gp_ensemble, so that a member's mean and
// variance have the bits of its marginal record): over the records g[0..n) whose admissible minimum is m, the
// warp-reduced S0 = sum e, the mixture mean sum e mu / S0 and variance sum e (v + (mu - mean)^2) / S0 (second pass), |A|
// and the number of e > 0 points.  Left per lane for the caller: s2 += e^2, and the bracket [lo, hi] of the e > 0
// components (extended, not reset).  st not null: (e, mu, sd) of every point are staged in st[0..2][k].
struct MargMoments {
  double s0, fmean, fvar;
  int n_admissible, n_positive;
};
__device__ __forceinline__ MargMoments marg_moments(const SieGpResult* __restrict__ g, int n, int lane, double m,
                                                    double (*st)[MARG_STAGE], double& s2, double& lo, double& hi) {
  double s0 = 0.0, s1 = 0.0;
  int n_adm = 0, n_pos = 0;
  for (int k = lane; k < n; k += 32) {
    double e, mu, sd;
    n_adm += marg_component(&g[k], m, e, mu, sd) ? 1 : 0;
    if (st) { st[0][k] = e; st[1][k] = mu; st[2][k] = sd; }
    if (e > 0.0) {
      s0 = __dadd_rn(s0, e);
      s2 = __fma_rn(e, e, s2);
      s1 = __fma_rn(e, mu, s1);
      lo = fmin(lo, mu - 40.0 * sd);
      hi = fmax(hi, mu + 40.0 * sd);
      ++n_pos;
    }
  }
  s0 = warp_sum_xor(s0);
  s1 = warp_sum_xor(s1);
  n_adm = __reduce_add_sync(0xffffffffu, n_adm);       // integer sums: exact in any order
  n_pos = __reduce_add_sync(0xffffffffu, n_pos);
  const double fmean = s1 / s0;
  double sv = 0.0;
  for (int k = lane; k < n; k += 32) {
    double v;
    if (gp_grid_admissible(&g[k], v)) {
      const double e = exp(m - v);
      if (e > 0.0) {
        const double d = __ldg(&g[k].fmean) - fmean;
        sv = __fma_rn(e, __fma_rn(d, d, __ldg(&g[k].fvar)), sv);
      }
    }
  }
  sv = warp_sum_xor(sv);
  return {s0, fmean, sv / s0, n_adm, n_pos};
}

__global__ void __launch_bounds__(MARG_WARPS * 32)
k_gp_grid_marginal(const SieGpResult* __restrict__ grid, int P, int n, const double* __restrict__ q, int n_q,
                   SieGpResult* __restrict__ out, SieGpMarginal* __restrict__ stats, double* __restrict__ quant) {
  __shared__ double s_c[MARG_WARPS][3][MARG_STAGE];  // staged (e, mu, sd) of each warp's problem
  const int wp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int p = blockIdx.x * MARG_WARPS + wp;
  if (p >= P) return;                                  // whole warp: p is uniform across it
  const SieGpResult* g = grid + (size_t)p * n;
  double m;
  int bi;
  gp_grid_argmin_warp(g, n, lane, m, bi);
  if (bi == SEL_NONE) {                                // A empty: record 0 (its info says why), NaN moments / quantiles
    if (lane == 0) {
      SieGpResult r = g[0];
      r.fmean = r.fvar = r.nlml = sie_nan();
      out[p] = r;
      SieGpMarginal s;
      s.ess = s.w_max = sie_nan();
      s.n_admissible = 0;
      s.argmax = -1;
      stats[p] = s;
    }
    for (int i = lane; i < n_q; i += 32) quant[(size_t)p * n_q + i] = sie_nan();
    return;
  }
  double (*st)[MARG_STAGE] = n <= MARG_STAGE ? s_c[wp] : nullptr;
  double s2 = 0.0, lo = __longlong_as_double(0x7ff0000000000000LL), hi = -lo;
  const MargMoments mo = marg_moments(g, n, lane, m, st, s2, lo, hi);
  const double s0 = mo.s0;
  s2 = warp_sum_xor(s2);
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    lo = fmin(lo, __shfl_xor_sync(0xffffffffu, lo, off));
    hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, off));
  }
  __syncwarp();                                        // the staged components are visible to the whole warp

  // F(x) = sum_k e_k Phi((x - mu_k) / sd_k) / S0, a point mass (sd = 0) counting from x = mu on (right-continuous)
  auto cdf = [&](double x) {
    double f = 0.0;
    for (int k = lane; k < n; k += 32) {
      double e, mu, sd;
      if (st) { e = st[0][k]; mu = st[1][k]; sd = st[2][k]; }
      else marg_component(&g[k], m, e, mu, sd);
      if (e > 0.0) f = __fma_rn(e, sd > 0.0 ? normcdf((x - mu) / sd) : (x >= mu ? 1.0 : 0.0), f);
    }
    return warp_sum_xor(f) / s0;
  };
  for (int i = 0; i < n_q; ++i) {
    const double t = q[i];
    double a = lo, b = hi;
    if (cdf(a) >= t) b = a;                            // a point mass at the lower end already holds q
    else if (cdf(b) >= t) {                            // invariant F(a) < q <= F(b)
      for (int it = 0; it < 128; ++it) {
        const double c = 0.5 * a + 0.5 * b;
        if (c == a || c == b) break;
        if (cdf(c) >= t) b = c; else a = c;
      }
    }                                                  // else: sum w rounds below q; hi is the upper end
    if (lane == 0) quant[(size_t)p * n_q + i] = b;
  }
  if (lane == 0) {
    SieGpResult r = g[bi];
    r.fmean = mo.fmean;
    r.fvar = mo.fvar;
    r.nlml = m - log(s0) + log((double)mo.n_admissible);
    out[p] = r;
    SieGpMarginal s;
    s.ess = s0 * s0 / s2;
    s.w_max = 1.0 / s0;
    s.n_admissible = mo.n_admissible;
    s.argmax = bi;
    stats[p] = s;
  }
}

// Ensemble pool per problem (sie_gp_ensemble).  One CTA per ensemble problem e, whose records are [M][n]:
//   1. one warp per member (members wp, wp + ENS_WARPS, ...): k_gp_grid_marginal's first two passes (marg_moments), so
//      the member mean / variance have the bits of that member's marginal record; plus the member's count of e > 0
//      components and its part of the bracket [lo, hi]
//   2. pooled moments over the contributing members (M' of them, weight 1 / M'), second pass for var_between
//   3. the e > 0 components (w = e / S0_m, mu, sd) compacted into the CTA's slab of the scratch in (member, grid index)
//      order, each member at the exclusive prefix sum of the counts
//   4. bisection on F(x) = sum w Phi((x - mu) / sd) / M' for up to ENS_QB levels at once: one pass over the slab
//      evaluates F at every active level's midpoint, so the slab is read once per halving, not once per level
// Every sum runs over an index order fixed by (M, n) (per-thread strided sums, xor trees, then the warp sums added in
// warp order), so the result does not depend on the schedule or on which batch filled which member slot.
constexpr int ENS_WARPS = 8;
constexpr int ENS_THREADS = ENS_WARPS * 32;
constexpr int ENS_MAX_MEMBERS = 1024;   // per-member stats in static shared memory: 36 KB
constexpr int ENS_QB = 4;               // quantile levels bisected together

// Fixed-order CTA sum of NV values per thread; every thread gets the totals.  red: [NV][ENS_WARPS] shared.
template <int NV>
__device__ __forceinline__ void ens_block_sum(double (&v)[NV], double (*red)[ENS_WARPS]) {
  const int wp = threadIdx.x >> 5;
#pragma unroll
  for (int j = 0; j < NV; ++j) v[j] = warp_sum_xor(v[j]);
  __syncthreads();                                     // the previous call's readers are done with red
  if ((threadIdx.x & 31) == 0) {
#pragma unroll
    for (int j = 0; j < NV; ++j) red[j][wp] = v[j];
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < NV; ++j) {
    double s = red[j][0];
    for (int w = 1; w < ENS_WARPS; ++w) s = __dadd_rn(s, red[j][w]);
    v[j] = s;
  }
}

// f[j] <- F(x[j]) * M' for the levels j with bit j of `act` set, over the n_c compacted components.
__device__ __forceinline__ void ens_cdf(const double* w, const double* mu, const double* sd, int n_c,
                                        const double (&x)[ENS_QB], unsigned act, double (&f)[ENS_QB],
                                        double (*red)[ENS_WARPS]) {
#pragma unroll
  for (int j = 0; j < ENS_QB; ++j) f[j] = 0.0;
  for (int i = threadIdx.x; i < n_c; i += ENS_THREADS) {
    const double wi = w[i], mi = mu[i], si = sd[i];
#pragma unroll
    for (int j = 0; j < ENS_QB; ++j)
      if (act & (1u << j)) f[j] = __fma_rn(wi, si > 0.0 ? normcdf((x[j] - mi) / si) : (x[j] >= mi ? 1.0 : 0.0), f[j]);
  }
  ens_block_sum<ENS_QB>(f, red);
}

__global__ void __launch_bounds__(ENS_THREADS, 2)
k_gp_ensemble(const SieGpResult* __restrict__ rec, int M, int n, const double* __restrict__ q, int n_q,
              SieGpEnsemble* __restrict__ out, double* __restrict__ quant, double* __restrict__ scratch) {
  __shared__ double s_mu[ENS_MAX_MEMBERS], s_v[ENS_MAX_MEMBERS], s_m[ENS_MAX_MEMBERS], s_s0[ENS_MAX_MEMBERS];
  __shared__ int s_off[ENS_MAX_MEMBERS + 1];          // e > 0 components per member, then their exclusive prefix sum
  __shared__ double s_red[ENS_QB][ENS_WARPS];
  const int wp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int e = blockIdx.x;
  const size_t cap = (size_t)M * n;
  const SieGpResult* base = rec + (size_t)e * cap;
  double* sw = scratch + (size_t)e * 3 * cap;          // this CTA's slab: w [cap], mu [cap], sd [cap]
  double* smu = sw + cap;
  double* ssd = smu + cap;

  double lo = __longlong_as_double(0x7ff0000000000000LL), hi = -lo;
  for (int mm = wp; mm < M; mm += ENS_WARPS) {
    const SieGpResult* g = base + (size_t)mm * n;
    double m;
    int bi;
    gp_grid_argmin_warp(g, n, lane, m, bi);
    if (bi == SEL_NONE) {                              // A_m empty: the member does not contribute
      if (lane == 0) s_off[mm] = 0;
      continue;
    }
    double s2 = 0.0;
    const MargMoments mo = marg_moments(g, n, lane, m, nullptr, s2, lo, hi);
    if (lane == 0) {
      s_mu[mm] = mo.fmean;
      s_v[mm] = mo.fvar;
      s_m[mm] = m;
      s_s0[mm] = mo.s0;
      s_off[mm] = mo.n_positive;                       // >= 1: the minimum has e = 1
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    lo = fmin(lo, __shfl_xor_sync(0xffffffffu, lo, off));
    hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, off));
  }
  __syncthreads();
  if (wp == 0) {                                       // exclusive scan of the counts: lane L owns a contiguous chunk
    const int chunk = (M + 31) / 32, m0 = min(M, lane * chunk), m1 = min(M, m0 + chunk);
    int t = 0;
    for (int mm = m0; mm < m1; ++mm) t += s_off[mm];
    int incl = t;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const int o = __shfl_up_sync(0xffffffffu, incl, off);
      if (lane >= off) incl += o;
    }
    int run = incl - t;
    for (int mm = m0; mm < m1; ++mm) {
      const int c = s_off[mm];
      s_off[mm] = run;
      run += c;
    }
    if (lane == 31) s_off[M] = incl;
  }
  __syncthreads();
  double mv[3] = {0.0, 0.0, 0.0};                     // sum of the member means, of their variances, M'
  for (int mm = threadIdx.x; mm < M; mm += ENS_THREADS) {
    if (s_off[mm + 1] > s_off[mm]) {
      mv[0] = __dadd_rn(mv[0], s_mu[mm]);
      mv[1] = __dadd_rn(mv[1], s_v[mm]);
      mv[2] += 1.0;
    }
  }
  ens_block_sum<3>(mv, s_red);
  const double mp = mv[2];
  const int n_members = (int)mp;
  const size_t qo = (size_t)e * n_q;
  if (n_members == 0) {
    if (threadIdx.x == 0) {
      SieGpEnsemble r;
      r.fmean = r.fvar = r.var_within = r.var_between = sie_nan();
      r.n_members = 0;
      r.pad_ = 0;
      out[e] = r;
    }
    for (int i = threadIdx.x; i < n_q; i += ENS_THREADS) quant[qo + i] = sie_nan();
    return;
  }
  const double fmean = mv[0] / mp, vw = mv[1] / mp;
  double vb[1] = {0.0};
  for (int mm = threadIdx.x; mm < M; mm += ENS_THREADS) {
    if (s_off[mm + 1] > s_off[mm]) {
      const double d = s_mu[mm] - fmean;
      vb[0] = __fma_rn(d, d, vb[0]);
    }
  }
  ens_block_sum<1>(vb, s_red);
  if (threadIdx.x == 0) {
    SieGpEnsemble r;
    r.fmean = fmean;
    r.var_within = vw;
    r.var_between = vb[0] / mp;
    r.fvar = r.var_within + r.var_between;
    r.n_members = n_members;
    r.pad_ = 0;
    out[e] = r;
  }
  if (n_q == 0) return;

  // bracket over every contributing component (fmin / fmax are exact: any order gives the same bits)
  __syncthreads();
  if (lane == 0) { s_red[0][wp] = lo; s_red[1][wp] = hi; }
  __syncthreads();
  lo = s_red[0][0];
  hi = s_red[1][0];
  for (int w = 1; w < ENS_WARPS; ++w) { lo = fmin(lo, s_red[0][w]); hi = fmax(hi, s_red[1][w]); }

  for (int mm = wp; mm < M; mm += ENS_WARPS) {         // compaction, in (member, grid index) order
    int off = s_off[mm];
    if (s_off[mm + 1] == off) continue;
    const SieGpResult* g = base + (size_t)mm * n;
    const double m = s_m[mm], s0 = s_s0[mm];
    for (int k0 = 0; k0 < n; k0 += 32) {
      const int k = k0 + lane;
      double ek = 0.0, mu = 0.0, sd = 0.0;
      if (k < n) marg_component(&g[k], m, ek, mu, sd);
      const unsigned bal = __ballot_sync(0xffffffffu, ek > 0.0);
      if (ek > 0.0) {
        const int i = off + __popc(bal & ((1u << lane) - 1u));
        sw[i] = ek / s0;
        smu[i] = mu;
        ssd[i] = sd;
      }
      off += __popc(bal);
    }
  }
  __syncthreads();                                     // the slab is visible to the whole CTA
  const int n_c = s_off[M];

  double x[ENS_QB], f[ENS_QB];
#pragma unroll
  for (int j = 0; j < ENS_QB; ++j) x[j] = j == 0 ? lo : hi;
  ens_cdf(sw, smu, ssd, n_c, x, 3u, f, s_red);
  const double f_lo = f[0] / mp, f_hi = f[1] / mp;
  for (int i0 = 0; i0 < n_q; i0 += ENS_QB) {
    const int nb = min(ENS_QB, n_q - i0);
    double a[ENS_QB], b[ENS_QB], t[ENS_QB];
    unsigned act = 0u;
#pragma unroll
    for (int j = 0; j < ENS_QB; ++j) {
      t[j] = j < nb ? q[i0 + j] : 0.0;
      a[j] = lo;
      b[j] = hi;
      if (j >= nb) continue;
      if (f_lo >= t[j]) b[j] = lo;                     // a point mass at the lower end already holds q
      else if (f_hi >= t[j]) act |= 1u << j;           // invariant F(a) < q <= F(b)
    }                                                  // else: sum w rounds below q; hi is the upper end
    for (int it = 0; it < 128 && act; ++it) {
#pragma unroll
      for (int j = 0; j < ENS_QB; ++j) {
        if (!(act & (1u << j))) continue;
        x[j] = 0.5 * a[j] + 0.5 * b[j];
        if (x[j] == a[j] || x[j] == b[j]) act &= ~(1u << j);
      }
      if (!act) break;
      ens_cdf(sw, smu, ssd, n_c, x, act, f, s_red);
#pragma unroll
      for (int j = 0; j < ENS_QB; ++j) {
        if (!(act & (1u << j))) continue;
        if (f[j] / mp >= t[j]) b[j] = x[j]; else a[j] = x[j];
      }
    }
    if (threadIdx.x == 0) {
#pragma unroll
      for (int j = 0; j < ENS_QB; ++j)
        if (j < nb) quant[qo + i0 + j] = b[j];
    }
  }
}

__host__ size_t gp_per_cta_bytes(int max_pred) {
  size_t d = (size_t)9 * max_pred * max_pred + (size_t)3 * MAXN * max_pred + (size_t)3 * max_pred + (size_t)MAXN * LDS;
  size_t bytes = d * sizeof(double) + (size_t)max_pred * sizeof(int);
  return (bytes + 255) / 256 * 256;
}
__host__ size_t gp_header_bytes(int P) { return ((size_t)256 + (size_t)P * sizeof(int32_t) + 255) / 256 * 256; }
int gp_grid(int P) {
  const SieDevice* dev = sie_device();
  const int sms = (dev && dev->sm_count > 0) ? dev->sm_count : 148;
  const int g = 2 * sms;     // shared memory (~106 KB) and 128 registers/thread allow two CTAs per SM
  return P < g ? P : g;
}

}  // namespace

// Profiling aid (not part of the reference-facing interface): reads and clears the per-phase cycle counters of
// k_gp_forecast; all zero unless the library was built with -DSIE_GP_TIMERS.
extern "C" int sie_debug_gp_phases(unsigned long long* out16) {
  if (!out16) return SIE_ERR_ARG;
  if (cudaMemcpyFromSymbol(out16, g_gp_phase, sizeof(unsigned long long) * 16) != cudaSuccess) return SIE_ERR_LAUNCH;
  unsigned long long zero[16] = {0};
  if (cudaMemcpyToSymbol(g_gp_phase, zero, sizeof(zero)) != cudaSuccess) return SIE_ERR_LAUNCH;
  return SIE_OK;
}

extern "C" size_t sie_gp_scratch_bytes(int P, int max_pred, int max_n) {
  (void)max_n;
  if (P < 1) P = 1;
  return gp_header_bytes(P) + (size_t)gp_grid(P) * gp_per_cta_bytes(max_pred);
}

static int gp_launch(const SieGpProblem* prob, int P, const double* y_all, const double* anom_sic,
                     const int32_t* n_areas_sic, int max_areas_sic, int Tstride_sic, const double* anom_sst,
                     const int32_t* n_areas_sst, int max_areas_sst, int Tstride_sst, int max_pred, SieGpResult* out,
                     void* scratch, size_t scratch_bytes, const double* sig_grid, int n_sig, void* stream) {
  SIE_CHECK_ARG(prob && y_all && anom_sic && n_areas_sic && out && scratch, "null pointer");
  SIE_CHECK_ARG(P > 0 && max_pred > 0 && (max_pred % 4) == 0, "P>0 and max_pred a positive multiple of 4");
  const size_t per = gp_per_cta_bytes(max_pred);
  const size_t head = gp_header_bytes(P);
  SIE_CHECK_ARG(scratch_bytes >= head + per, "scratch too small");
  SIE_CHECK_ARG(max_pred <= 2 * MAXN * LDS / PANEL, "max_pred above the LU panel capacity (520)");
  int grid = gp_grid(P);
  if (head + (size_t)grid * per > scratch_bytes) grid = (int)((scratch_bytes - head) / per);
  SIE_CHECK_ARG(grid >= 1, "scratch too small");
  cudaStream_t st = (cudaStream_t)stream;
  int* queue = reinterpret_cast<int*>(scratch);
  int32_t* order = reinterpret_cast<int32_t*>(reinterpret_cast<unsigned char*>(scratch) + 256);
  k_gp_order<<<1, 1024, 0, st>>>(prob, P, n_areas_sic, n_areas_sst, order, queue);
  SIE_CHECK_LAUNCH();
  const size_t smem = sizeof(Smem);
  const SieDevice* dev = sie_device();
  if (!dev) return SIE_ERR_LAUNCH;
  if (int rc = sie_ensure_smem(dev, SIE_K_GP, (const void*)k_gp_forecast, smem)) return rc;
  k_gp_forecast<<<grid, GT, smem, st>>>(prob, P, y_all, anom_sic, n_areas_sic, max_areas_sic, Tstride_sic, anom_sst,
                                        n_areas_sst, max_areas_sst, Tstride_sst, max_pred, out,
                                        (unsigned char*)scratch + head, per, order, queue, sig_grid, n_sig);
  SIE_CHECK_LAUNCH();
  return SIE_OK;
}

extern "C" int sie_gp_forecast(const SieGpProblem* prob, int P, const double* y_all, const double* anom_sic,
                               const int32_t* n_areas_sic, int max_areas_sic, int Tstride_sic,
                               const double* anom_sst, const int32_t* n_areas_sst, int max_areas_sst,
                               int Tstride_sst, int max_pred, SieGpResult* out, void* scratch,
                               size_t scratch_bytes, void* stream) {
  return gp_launch(prob, P, y_all, anom_sic, n_areas_sic, max_areas_sic, Tstride_sic, anom_sst, n_areas_sst,
                   max_areas_sst, Tstride_sst, max_pred, out, scratch, scratch_bytes, nullptr, 1, stream);
}

extern "C" int sie_gp_hyper_grid(const SieGpProblem* prob, int P, const double* sig_grid, int n_sig,
                                 const double* y_all, const double* anom_sic, const int32_t* n_areas_sic,
                                 int max_areas_sic, int Tstride_sic, const double* anom_sst,
                                 const int32_t* n_areas_sst, int max_areas_sst, int Tstride_sst, int max_pred,
                                 SieGpResult* out, void* scratch, size_t scratch_bytes, void* stream) {
  SIE_CHECK_ARG(sig_grid && n_sig > 0, "sig_grid must hold n_sig > 0 values");
  return gp_launch(prob, P, y_all, anom_sic, n_areas_sic, max_areas_sic, Tstride_sic, anom_sst, n_areas_sst,
                   max_areas_sst, Tstride_sst, max_pred, out, scratch, scratch_bytes, sig_grid, n_sig, stream);
}

extern "C" int sie_gp_grid_select(const SieGpResult* grid, const SieGpProblem* prob, int P, const double* ell_grid,
                                  int n_ell, const double* sig_grid, int n_sig, SieGpProblem* tuned, int32_t* best,
                                  void* stream) {
  SIE_CHECK_ARG(grid && prob && ell_grid && sig_grid && tuned && best, "null pointer");
  SIE_CHECK_ARG(P > 0 && n_ell > 0 && n_sig > 0, "P, n_ell and n_sig must be positive");
  SIE_CHECK_ARG((long long)n_ell * n_sig < SEL_NONE, "n_ell * n_sig must be below 2^31 - 1");
  k_gp_grid_select<<<(P - 1) / SEL_WARPS + 1, SEL_WARPS * 32, 0, (cudaStream_t)stream>>>(
      grid, prob, P, ell_grid, n_ell, sig_grid, n_sig, tuned, best);
  SIE_CHECK_LAUNCH();
  return SIE_OK;
}

extern "C" int sie_gp_grid_marginal(const SieGpResult* grid, int P, int n_grid, const double* q, int n_q,
                                    SieGpResult* out, SieGpMarginal* stats, double* quant, void* stream) {
  SIE_CHECK_ARG(grid && out && stats, "null pointer");
  SIE_CHECK_ARG(P > 0 && n_grid > 0, "P and n_grid must be positive");
  SIE_CHECK_ARG(n_q >= 0, "n_q must not be negative");
  SIE_CHECK_ARG(n_q == 0 || (q && quant), "q and quant must not be null when n_q > 0");
  k_gp_grid_marginal<<<(P - 1) / MARG_WARPS + 1, MARG_WARPS * 32, 0, (cudaStream_t)stream>>>(
      grid, P, n_grid, q, n_q, out, stats, quant);
  SIE_CHECK_LAUNCH();
  return SIE_OK;
}

extern "C" size_t sie_gp_ensemble_scratch_bytes(int E, int M, int n_grid) {
  if (E < 1 || M < 1 || n_grid < 1) return 0;
  return (size_t)E * (size_t)M * (size_t)n_grid * 3 * sizeof(double);
}

extern "C" int sie_gp_ensemble(const SieGpResult* rec, int E, int M, int n_grid, const double* q, int n_q,
                               SieGpEnsemble* out, double* quant, void* scratch, size_t scratch_bytes, void* stream) {
  SIE_CHECK_ARG(rec && out && scratch, "null pointer");
  SIE_CHECK_ARG(E > 0 && M > 0 && n_grid > 0, "E, M and n_grid must be positive");
  SIE_CHECK_ARG(n_q >= 0, "n_q must not be negative");
  SIE_CHECK_ARG(n_q == 0 || (q && quant), "q and quant must not be null when n_q > 0");
  if (M > ENS_MAX_MEMBERS) {
    sie_set_error("%s: M = %d members, at most %d are supported", __func__, M, ENS_MAX_MEMBERS);
    return SIE_ERR_UNSUPPORTED;
  }
  if ((long long)M * n_grid >= (1LL << 31)) {
    sie_set_error("%s: M * n_grid = %lld records per problem, must be below 2^31", __func__, (long long)M * n_grid);
    return SIE_ERR_UNSUPPORTED;
  }
  SIE_CHECK_ARG(scratch_bytes >= sie_gp_ensemble_scratch_bytes(E, M, n_grid), "scratch too small");
  k_gp_ensemble<<<E, ENS_THREADS, 0, (cudaStream_t)stream>>>(rec, M, n_grid, q, n_q, out, quant, (double*)scratch);
  SIE_CHECK_LAUNCH();
  return SIE_OK;
}
