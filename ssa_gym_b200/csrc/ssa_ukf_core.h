// ssa_ukf_core.h — the small fp64 linear algebra of the unscented Kalman filter, element by element.
// Host+device; the sm_100a kernels call these per lane, the host twin (tests/twin) calls them in
// loops, and both therefore execute the same rounded operations in the same order.
//
// Reference behaviour reproduced.  filterpy is a third-party dependency of the reference
// (requirements.txt:14, unpinned; 1.4.5 is the release contemporary with the repo) and is not
// vendored; its published algorithm is restated in SURVEY.md Appendix B.  Call sites in the
// reference: envs/ssa_tasker_simple_2.py:110 (Q_discrete_white_noise), :211-218 (UKF and
// MerweScaledSigmaPoints construction), :275 (predict), :301-306 (update, .y .S .sigmas_h).
//   sigma points   s0 = x, s_{k+1} = x + U[k,:], s_{7+k} = x - U[k,:],  U^T U = (lambda+n) P, U upper
//   sqrt_method    envs/dynamics.py:402-417 robust_cholesky: scipy cholesky, on failure retry with
//                  + I*10**i for i = -6..9, then LinAlgError
//   predict        x = Wm . f(s);  P = sum_k Wc_k y_k y_k^T + Q, y_k = f(s_k) - x;  sigmas re-drawn
//   update         z_k = h(s_k); zp = mean_z; S = sum Wc_k r_k r_k^T + R; Pxz = sum Wc_k dx_k r_k^T;
//                  K = Pxz S^-1; x += K y; P -= K (S K^T)
//
// Packed symmetric storage: the 6x6 covariance keeps its upper triangle only, row-major,
// idx(i,j) = i*6 - i*(i-1)/2 + (j-i) for i <= j (21 doubles).  The reference's Cholesky reads only
// the upper triangle and obs/reward read only the diagonal, so nothing on the path observes the
// lower triangle (SURVEY.md 7.2).
#pragma once
#include "ssa_math.h"

#define SSA_NX 6
#define SSA_NZ 3
#define SSA_NSIG 13
#define SSA_NP 21

// status word of one object (int32)
#define SSA_ST_OK 0
#define SSA_ST_FAILED 0x1      /* filter is in the failed state (sentinels, skipped) — SS2:369-382 */
#define SSA_ST_LINALG 0x2      /* robust_cholesky exhausted its 16 inflation steps -> LinAlgError   */
#define SSA_ST_NAN 0x4         /* predict/update returned NaN in x (SS2:278, :306)                  */
#define SSA_ST_FXEXC 0x8       /* fx raised inside numba (assert / ZeroDivisionError / RuntimeError) */
#define SSA_ST_TRUTHEXC 0x10   /* fx raised while propagating the TRUE state (SS2:266, uncaught)    */
#define SSA_ST_IN_UPDATE 0x20  /* the failure happened in update() rather than predict()            */

#define SSA_XFAIL_POS 1e20 /* SS2:157-158 */
#define SSA_XFAIL_VEL 1e12

SSA_HD int ssa_pidx(int i, int j) { return i * 6 - (i * (i - 1)) / 2 + (j - i); }

// 10**i for i = -6..9 as Python evaluates it (dynamics.py:410): floats for i<0, ints for i>=0.
SSA_HD double ssa_pow10_infl(int t) {  // t = 0..15  <->  i = -6..9
  switch (t) {
    case 0: return 1e-06; case 1: return 1e-05; case 2: return 1e-04; case 3: return 1e-03;
    case 4: return 1e-02; case 5: return 1e-01; case 6: return 1.0;   case 7: return 10.0;
    case 8: return 1e2;   case 9: return 1e3;   case 10: return 1e4;  case 11: return 1e5;
    case 12: return 1e6;  case 13: return 1e7;  case 14: return 1e8;  default: return 1e9;
  }
}

// Upper Cholesky A = U^T U of a packed 6x6 in registers.  Returns 1 on success, 0 if a pivot is <= 0 or NaN (dpotrf
// info > 0 -> scipy LinAlgError) or if any entry is non-finite (scipy check_finite -> ValueError); both are swallowed by
// robust_cholesky's bare except.
// Evaluated as the root-free factorisation A = L D L^T followed by U = sqrt(D) L^T: the pivots d_j are the same
// quantities as LAPACK dpotf2's (a_jj minus the squares above it), so the success / failure decision is the same
// condition, but the dependent chain of a column is ONE division instead of a square root AND a division — the kernels
// that run this are nothing but that chain (k_factor / k_refactor: 6 columns per object at low occupancy), and the six
// square roots at the end are independent of each other.  U agrees with dpotf2's to rounding (U^T U = A to 1e-15).
template <bool INL>
SSA_HD int ssa_chol6_t(double* a /* 21, in: A, out: U */) {
  int ok = 1;
#pragma unroll
  for (int e = 0; e < SSA_NP; ++e) ok &= (ssa_fabs(a[e]) <= 1.79769313486231570815e+308);
  double d[6];
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    d[j] = a[ssa_pidx(j, j)];
    ok &= (d[j] > 0.0);
    const double inv = ssa_div_t<INL>(1.0, d[j]);
#pragma unroll
    for (int r = j + 1; r < 6; ++r) {
      const double l = ssa_mul(a[ssa_pidx(j, r)], inv);   // L[r][j]
#pragma unroll
      for (int c = r; c < 6; ++c) a[ssa_pidx(r, c)] = ssa_fma(-l, a[ssa_pidx(j, c)], a[ssa_pidx(r, c)]);
    }
#pragma unroll
    for (int c = j + 1; c < 6; ++c) a[ssa_pidx(j, c)] = ssa_mul(a[ssa_pidx(j, c)], inv);   // row j of L^T
  }
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    const double sj = ssa_sqrt_t<INL>(d[j]);
    a[ssa_pidx(j, j)] = sj;
#pragma unroll
    for (int c = j + 1; c < 6; ++c) a[ssa_pidx(j, c)] = ssa_mul(a[ssa_pidx(j, c)], sj);
  }
  return ok;
}

SSA_HD int ssa_chol6(double* a) { return ssa_chol6_t<false>(a); }

// robust_cholesky((lambda+n) * P).  P is read through (ptr, stride) so the caller can keep it in
// global SoA memory or in shared memory; it is re-read on the (rare) inflation retries instead of
// being held in registers.  Returns the number of the successful attempt: 0 = plain, t+1 = with
// +10**(t-6) on the diagonal, -1 = all 17 attempts failed (LinAlgError).
template <bool INL>
SSA_HD int ssa_robust_chol6_t(const double* P, long stride, double lam, double* U) {
  for (int t = -1; t < 16; ++t) {  // one copy of the factorisation in the instruction stream
#pragma unroll
    for (int e = 0; e < SSA_NP; ++e) U[e] = ssa_mul(lam, P[e * stride]);
    if (t >= 0) {
      const double eps = ssa_pow10_infl(t);
#pragma unroll
      for (int j = 0; j < 6; ++j) U[ssa_pidx(j, j)] = U[ssa_pidx(j, j)] + eps;
    }
    if (ssa_chol6_t<INL>(U)) return t + 1;
  }
  return -1;
}
SSA_HD int ssa_robust_chol6(const double* P, long stride, double lam, double* U) { return ssa_robust_chol6_t<false>(P, stride, lam, U); }

// Sigma point number `k` (0..12), component j, from x and the packed factor.
// s0 = x ; s_{1+r} = x - (-U[r,:]) = x + U[r,:] ; s_{7+r} = x - U[r,:]
SSA_HD void ssa_sigma_point(const double* x, const double* U, int k, double* s) {
  // branch-free in k so that the 13 lanes of a team stay converged; for k == 0 no row matches and
  // u stays +0.0 (x + 0.0 == x for every x the path produces)
  const int r = (k == 0) ? -1 : (k - 1) % 6;
  const int minus = k > 6;
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    double u = 0.0;
#pragma unroll
    for (int rr = 0; rr < 6; ++rr)
      if (rr <= j) u = (rr == r) ? U[ssa_pidx(rr, j)] : u;
    s[j] = minus ? (x[j] - u) : (x[j] + u);
  }
}

// Weighted mean of one component over the 13 sigma points: np.dot(Wm, sigmas)[i]
SSA_HD double ssa_wmean13(const double* v /* [13][ld] */, int ld, int i, const double* Wm) {
  double acc = ssa_mul(Wm[0], v[i]);
#pragma unroll
  for (int k = 1; k < SSA_NSIG; ++k) acc = ssa_fma(Wm[k], v[k * ld + i], acc);
  return acc;
}

// One element of  Y^T diag(Wc) Y  (filterpy unscented_transform fast path, residual = subtract)
SSA_HD double ssa_wcov13(const double* ya, int lda, int i, const double* yb, int ldb, int j, const double* Wc) {
  double acc = 0.0;
#pragma unroll
  for (int k = 0; k < SSA_NSIG; ++k) acc = ssa_fma(ya[k * lda + i], ssa_mul(Wc[k], yb[k * ldb + j]), acc);
  return acc;
}

// One element of  sum_k Wc[k] * outer(a_k, b_k)  (filterpy loop form: S with residual_fn, Pxz)
SSA_HD double ssa_wouter13(const double* ya, int lda, int i, const double* yb, int ldb, int j, const double* Wc) {
  double acc = 0.0;
#pragma unroll
  for (int k = 0; k < SSA_NSIG; ++k) acc = ssa_fma(Wc[k], ssa_mul(ya[k * lda + i], yb[k * ldb + j]), acc);
  return acc;
}

// inverse of a general 3x3 by LU with partial pivoting, the way numpy.linalg.inv does it
// (LAPACK dgesv on the identity: dgetrf column scaling by the reciprocal pivot, dgetrs solves).
// Returns 0 if a pivot is exactly zero (numpy raises LinAlgError "Singular matrix").
template <bool INL>
SSA_HD int ssa_inv3_t(const double* S /* row-major 3x3 */, double* SI) {
  double a[3][3], b[3][3];
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) { a[i][j] = S[3 * i + j]; b[i][j] = (i == j) ? 1.0 : 0.0; }
  int ok = 1;
  double rpiv[3];  // reciprocals of the three pivots: the back substitutions multiply by them (3 divisions instead of 12)
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    // pivot search (first maximum of |a[i][c]|, i >= c) and row swap, written with selects so the
    // register arrays keep static indices
#pragma unroll
    for (int i = c + 1; i < 3; ++i) {
      const int sw = ssa_fabs(a[i][c]) > ssa_fabs(a[c][c]);
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        const double ta = a[c][j], tb = a[i][j];
        a[c][j] = sw ? tb : ta; a[i][j] = sw ? ta : tb;
        const double ua = b[c][j], ub = b[i][j];
        b[c][j] = sw ? ub : ua; b[i][j] = sw ? ua : ub;
      }
    }
    ok &= (a[c][c] != 0.0);
    const double rp = ssa_div_t<INL>(1.0, a[c][c]);
    rpiv[c] = rp;
#pragma unroll
    for (int i = c + 1; i < 3; ++i) {
      a[i][c] = ssa_mul(a[i][c], rp);
#pragma unroll
      for (int j = c + 1; j < 3; ++j) a[i][j] = ssa_fma(-a[i][c], a[c][j], a[i][j]);
    }
  }
  // solve L U X = P I, column by column
#pragma unroll
  for (int col = 0; col < 3; ++col) {
    double y0 = b[0][col];
    double y1 = ssa_fma(-a[1][0], y0, b[1][col]);
    double y2 = ssa_fma(-a[2][1], y1, ssa_fma(-a[2][0], y0, b[2][col]));
    const double x2 = ssa_mul(y2, rpiv[2]);
    const double x1 = ssa_mul(ssa_fma(-a[1][2], x2, y1), rpiv[1]);
    const double x0 = ssa_mul(ssa_fma(-a[0][1], x1, ssa_fma(-a[0][2], x2, y0)), rpiv[0]);
    SI[col] = x0; SI[3 + col] = x1; SI[6 + col] = x2;
  }
  return ok;
}

SSA_HD int ssa_inv3(const double* S, double* SI) { return ssa_inv3_t<false>(S, SI); }

// Consistency diagnostics (SURVEY 8f-3).
// NEES d^T P^-1 d of one object (SS2:436-446 `anees`: delta @ inv(P_filter) @ delta), evaluated through the Cholesky
// factor P = U^T U (w = U^-T d, NEES = w.w) instead of an explicit inverse: same value for a positive definite P,
// better conditioned; NaN when P is not positive definite (numpy's inv would return some number there).
SSA_HD double ssa_nees6(const double* P, long stride, const double* d) {
  double U[SSA_NP];
#pragma unroll
  for (int e = 0; e < SSA_NP; ++e) U[e] = P[e * stride];
  if (!ssa_chol6(U)) return ssa_nan();
  double w[6], acc = 0.0;
#pragma unroll
  for (int i = 0; i < 6; ++i) {  // forward substitution with U^T (lower triangular)
    double t = d[i];
#pragma unroll
    for (int k = 0; k < i; ++k) t = ssa_fma(-U[ssa_pidx(k, i)], w[k], t);
    w[i] = ssa_div(t, U[ssa_pidx(i, i)]);
    acc = ssa_fma(w[i], w[i], acc);
  }
  return acc;
}
// NIS y^T S^-1 y (SS2:564-569 plot_NIS: y @ inv(S) @ y, numpy's order: the row vector y @ inv(S) first) and the
// innovation-bound flags of SS2:598-604: bit a = |y_a| < sqrt(S_aa), bit 3+a = |y_a| < 2 sqrt(S_aa).
SSA_HD double ssa_nis3(const double* S, const double* y, int* flags) {
  double SI[9];
  const int ok = ssa_inv3(S, SI);
  int f = 0;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const double sd = ssa_sqrt(S[4 * a]);
    f |= ((y[a] < sd) && (y[a] > -sd)) ? (1 << a) : 0;
    f |= ((y[a] < ssa_mul(2.0, sd)) && (y[a] > -ssa_mul(2.0, sd))) ? (8 << a) : 0;
  }
  *flags = f;
  if (!ok) return ssa_nan();
  double acc = 0.0;
#pragma unroll
  for (int b = 0; b < 3; ++b) {
    const double t = ssa_fma(y[2], SI[6 + b], ssa_fma(y[1], SI[3 + b], ssa_mul(y[0], SI[b])));
    acc = (b == 0) ? ssa_mul(t, y[0]) : ssa_fma(t, y[b], acc);
  }
  return acc;
}

// Per-episode statistics of the device-resident episodic mode (ssa_ukf_rollout_episode_stats_*): running sums of the
// diagnostics above over one episode, a few doubles per object and per environment instead of the per-step histories
// of the drop-in env.  Counts are kept as doubles (exact up to 2^53).  Host layouts equal the device ones (AoS).
// Object accumulator [SSA_EPO]: sum and count of the non-NaN NEES of its rows, Durbin-Watson state {num, den, prev} of
// its own innovation series per component, and the number of entries of that series.
#define SSA_EPO_S 0
#define SSA_EPO_C 1
#define SSA_EPO_DW 2
#define SSA_EPO_DWN 11
#define SSA_EPO 12
// Environment accumulator [SSA_EPE]: return, observations, NIS sum / count, the six innovation-bound counters (inside
// 1 sigma per component, then inside 2 sigmas), Durbin-Watson state of the overall innovation series and its entries.
#define SSA_EPE_RET 0
#define SSA_EPE_OBS 1
#define SSA_EPE_NIS 2
#define SSA_EPE_NISN 3
#define SSA_EPE_BND 4
#define SSA_EPE_DW 10
#define SSA_EPE_DWN 19
#define SSA_EPE 20
// Record of a finished episode: SSA_EPISODE_STATS_DOUBLES (include/ssa_ukf.h) doubles, layout documented there.
#define SSA_EPR 23

// one row of an episode for one object: NEES of (x_true - x, P) as ssa_diag_kernel evaluates it, NaN left out
SSA_HD void ssa_ep_nees_row(double* o, const double* xt, const double* x, long xs, const double* P, long ps) {
  double d[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) d[i] = xt[i * xs] - x[i * xs];
  const double v = ssa_nees6(P, ps, d);
  if (v == v) {
    o[SSA_EPO_S] = o[SSA_EPO_S] + v;
    o[SSA_EPO_C] = o[SSA_EPO_C] + 1.0;
  }
}
// one entry of a Durbin-Watson series per component, in the order of ssa_innov_stats_kernel; dw = {num, den, prev} x 3,
// n = entries before this one
SSA_HD void ssa_dw_push(double* dw, double n, const double* y) {
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const double e = y[c];
    dw[3 * c + 1] = ssa_fma(e, e, dw[3 * c + 1]);
    if (n > 0.0) {
      const double d = e - dw[3 * c + 2];
      dw[3 * c] = ssa_fma(d, d, dw[3 * c]);
    }
    dw[3 * c + 2] = e;
  }
}
// an update of the tasked object: its innovation y and innovation covariance S (SSA_STEP_RECORD)
SSA_HD void ssa_ep_observe(double* env, double* obj, const double* y, const double* S) {
  env[SSA_EPE_OBS] = env[SSA_EPE_OBS] + 1.0;
  int f = 0;
  const double nis = ssa_nis3(S, y, &f);
  if (nis == nis) {
    env[SSA_EPE_NIS] = env[SSA_EPE_NIS] + nis;
    env[SSA_EPE_NISN] = env[SSA_EPE_NISN] + 1.0;
  }
#pragma unroll
  for (int b = 0; b < 6; ++b) env[SSA_EPE_BND + b] = env[SSA_EPE_BND + b] + (double)((f >> b) & 1);
  ssa_dw_push(env + SSA_EPE_DW, env[SSA_EPE_DWN], y);
  env[SSA_EPE_DWN] = env[SSA_EPE_DWN] + 1.0;
  ssa_dw_push(obj + SSA_EPO_DW, obj[SSA_EPO_DWN], y);
  obj[SSA_EPO_DWN] = obj[SSA_EPO_DWN] + 1.0;
}
// The record of an episode that ended at step L: env accumulator, the m object accumulators [m][SSA_EPO] and the m
// status words of the environment.  Per-object Durbin-Watson min / max over the objects with >= 2 entries, NaN
// propagating as in np.min / np.max, NaN when no object qualifies.
SSA_HD void ssa_ep_finalise(const double* env, const double* obj, const int32_t* status, int m, double L, double* rec) {
  rec[0] = L;
  rec[1] = env[SSA_EPE_RET];
  double s = 0.0, c = 0.0, failed = 0.0;
  for (int j = 0; j < m; ++j) {
    s = s + obj[j * SSA_EPO + SSA_EPO_S];
    c = c + obj[j * SSA_EPO + SSA_EPO_C];
    failed = failed + ((status[j] & SSA_ST_FAILED) ? 1.0 : 0.0);
  }
  rec[2] = s;
  rec[3] = c;
  rec[4] = env[SSA_EPE_NIS];
  rec[5] = env[SSA_EPE_NISN];
  rec[6] = env[SSA_EPE_OBS];
#pragma unroll
  for (int b = 0; b < 6; ++b) rec[7 + b] = env[SSA_EPE_BND + b];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    rec[13 + k] = env[SSA_EPE_DWN] > 0.0 ? ssa_div(env[SSA_EPE_DW + 3 * k], env[SSA_EPE_DW + 3 * k + 1]) : ssa_nan();
    double lo = ssa_nan(), hi = ssa_nan();
    int any = 0, nan = 0;
    for (int j = 0; j < m; ++j) {
      const double* o = obj + j * SSA_EPO;
      if (!(o[SSA_EPO_DWN] >= 2.0)) continue;
      const double v = ssa_div(o[SSA_EPO_DW + 3 * k], o[SSA_EPO_DW + 3 * k + 1]);
      nan |= (v != v);
      lo = (!any || v < lo) ? v : lo;
      hi = (!any || v > hi) ? v : hi;
      any = 1;
    }
    rec[16 + k] = nan ? ssa_nan() : lo;
    rec[19 + k] = nan ? ssa_nan() : hi;
  }
  rec[22] = failed;
}
SSA_HD void ssa_ep_clear(double* env, double* obj, int m) {
  for (int q = 0; q < SSA_EPE; ++q) env[q] = 0.0;
  for (int q = 0; q < m * SSA_EPO; ++q) obj[q] = 0.0;
}

// Determinant of a packed symmetric 6x6 (agent_shannon, agents.py:24: np.linalg.det(P)).  numpy factors with a pivoted
// LU; for the symmetric (normally positive definite) covariances of the path the unpivoted symmetric elimination
// P = L D L^T is just as stable, needs half the arithmetic and keeps its 21 entries in registers with static indices:
// det = prod d_j.  Against exact rational determinants it is as close as LAPACK's (tests/test_det_exact.py).  A zero
// pivot returns 0.
SSA_HD double ssa_det6_sym(const double* P, long stride) {
  double a[SSA_NP];
#pragma unroll
  for (int e = 0; e < SSA_NP; ++e) a[e] = P[e * stride];
  double det = 1.0;
  int zero = 0;
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    const double d = a[ssa_pidx(j, j)];
    det = ssa_mul(det, d);
    zero |= (d == 0.0);
    const double inv = ssa_div(1.0, d);
#pragma unroll
    for (int r = j + 1; r < 6; ++r) {
      const double l = ssa_mul(a[ssa_pidx(j, r)], inv);
#pragma unroll
      for (int c = r; c < 6; ++c) a[ssa_pidx(r, c)] = ssa_fma(-l, a[ssa_pidx(j, c)], a[ssa_pidx(r, c)]);
    }
  }
  return zero ? 0.0 : det;
}

// np.sum of a[0 .. n) (contiguous float64) in numpy's order: the 'shaped' reward's 1 - np.sum(rewards[:i]) (SS2:345),
// where a sequential sum differs in the last bits for most prefix lengths.  numpy's pairwise_sum: a block of n < 8 is
// summed sequentially from 0.0; a block of 8 <= n <= 128 in eight accumulators seeded with a[0..7] and advanced in
// strides of 8, combined ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)), its remainder added in order; a longer block is split at
// n2 = n/2 - (n/2) % 8 and its two halves summed the same way and added.  The reduction adds the result to its 0.0
// identity.  The recursion is walked with an explicit stack (no device recursion): a block of n <= 2^31 elements is
// split at most 24 times before its halves reach 128.
SSA_HD double ssa_pairwise_block(const double* a, long n) {
  if (n < 8) {
    double s = 0.0;
    for (long i = 0; i < n; ++i) s = s + a[i];
    return s;
  }
  double r[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) r[j] = a[j];
  long i = 8;
  for (; i < n - (n % 8); i += 8) {
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = r[j] + a[i + j];
  }
  double s = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
  for (; i < n; ++i) s = s + a[i];
  return s;
}
SSA_HD double ssa_pairwise_sum(const double* a, long n) {
  double left[32];   // sum of the left half of each open split whose right half is being summed
  long right[32];    // length of the right half of each open split (0 once it is being summed)
  int top = 0;
  long off = 0, len = n;
  for (;;) {
    while (len > 128) {  // descend into left halves
      long n2 = len / 2;
      n2 -= n2 % 8;
      right[top] = len - n2;
      ++top;
      len = n2;
    }
    double s = ssa_pairwise_block(a + off, len);
    off += len;
    while (top > 0 && right[top - 1] == 0) {  // both halves of the innermost split are done
      --top;
      s = left[top] + s;
    }
    if (top == 0) return 0.0 + s;
    left[top - 1] = s;  // a left half is done: sum the right one
    len = right[top - 1];
    right[top - 1] = 0;
  }
}

// np.trace(P) over the packed diagonal, numpy's left-to-right order (agents.py:8,40)
SSA_HD double ssa_trace6(const double* P, long stride) {
  double t = P[0];
  t = t + P[6 * stride];
  t = t + P[11 * stride];
  t = t + P[15 * stride];
  t = t + P[18 * stride];
  t = t + P[20 * stride];
  return t;
}

// ---- running normalization of observations and returns (episodic mode, k_normalize; ssa_ukf_rollout_normalize) -------
// Stable-Baselines3's VecNormalize over RunningMeanStd, restated expression by expression so that a learner gets the
// statistics it already uses.  Two deviations.  With obs_dtype float32 the batch moments are summed in float64 over the
// float32-rounded rows, where np.mean / np.var of a float32 array would accumulate in float32.  And the order of the
// batch sums over the E environments: numpy adds the
// rows of a column in sequence, which a CTA cannot do quickly.  The sums here use ONE order that depends on E only (not
// on the column, the layout, the launch path or the block shape): leaves of ssa_norm_leaf(E) consecutive rows, each
// summed in row order from its first element, then the leaf sums combined by the fixed tree of ssa_norm_tree.
// ssa_norm_leaf keeps the tree at most 1024 leaves wide (8 KB of shared memory per column).
SSA_HD int ssa_norm_leaf(int E) { return E <= 32768 ? 32 : (E + 1023) / 1024; }
SSA_HD int ssa_norm_leaves(int E) { return (E + ssa_norm_leaf(E) - 1) / ssa_norm_leaf(E); }
// an observation value as the caller would see it un-normalized: float32-rounded for obs_dtype float32 (decltype(1.0)
// names the built-in double also where the operation-counting build, oracle/opcount_twin.cpp, redefines `double`)
SSA_HD double ssa_norm_in(double v, int f32) { return f32 ? (double)(float)(decltype(1.0))v : v; }
// the reward that enters the returns: _format_reward's nan_to_num(nan = +-inf = 0.5) for the layouts other than 'flatten'
SSA_HD double ssa_norm_reward_in(double r, int nan_to_num) { return (nan_to_num && !(r - r == 0.0)) ? 0.5 : r; }
// one leaf: rows r0 .. r1 - 1 of the column x[r * stride]; sq: the squared deviations from `mean` instead of the values.
// The rows are loaded 16 at a time before they are added in order: on the device a leaf's strided loads are then in
// flight together instead of one L2 round trip per row.
SSA_HD double ssa_norm_leaf_sum(const double* x, long stride, int r0, int r1, int f32, int sq, double mean) {
  double s = 0.0;
  for (int b = r0; b < r1; b += 16) {
    double v[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] = b + j < r1 ? x[(long)(b + j) * stride] : 0.0;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      if (b + j >= r1) break;
      double w = ssa_norm_in(v[j], f32);
      if (sq) {
        const double d = w - mean;
        w = d * d;
      }
      s = b + j == r0 ? w : s + w;
    }
  }
  return s;
}
// the leaf sums v[0 .. n) combined in place, level by level: at level s = 1, 2, 4, ... v[i] += v[i + s] for i = 0, 2s,
// 4s, ... with i + s < n.  The sum ends in v[0].  (k_normalize runs each level's additions in parallel.)
SSA_HD double ssa_norm_tree(double* v, int n) {
  for (int s = 1; s < n; s <<= 1)
    for (int i = 0; i + s < n; i += 2 * s) v[i] = v[i] + v[i + s];
  return v[0];
}
// np.mean and np.var of a column of E rows (the sum over E, then that of the squared deviations from the mean over E),
// in the fixed order; buf holds ssa_norm_leaves(E) doubles
SSA_HD void ssa_norm_moments(const double* x, long stride, int E, int f32, double* buf, double* mean, double* var) {
  const int L = ssa_norm_leaf(E), n = ssa_norm_leaves(E);
  for (int k = 0; k < n; ++k) buf[k] = ssa_norm_leaf_sum(x, stride, k * L, k * L + L < E ? k * L + L : E, f32, 0, 0.0);
  const double mu = ssa_div(ssa_norm_tree(buf, n), (double)E);
  for (int k = 0; k < n; ++k) buf[k] = ssa_norm_leaf_sum(x, stride, k * L, k * L + L < E ? k * L + L : E, f32, 1, mu);
  *mean = mu;
  *var = ssa_div(ssa_norm_tree(buf, n), (double)E);
}
// RunningMeanStd.update_from_moments, in its expression order
SSA_HD void ssa_norm_merge(double* mean, double* var, double* count, double bmean, double bvar, double bcount) {
  const double delta = bmean - *mean;
  const double tot = *count + bcount;
  const double new_mean = *mean + ssa_div(delta * bcount, tot);
  const double m_a = *var * *count, m_b = bvar * bcount;
  const double m_2 = m_a + m_b + ssa_div(delta * delta * *count * bcount, tot);
  *mean = new_mean;
  *var = ssa_div(m_2, tot);
  *count = bcount + *count;
}
// np.clip(v, -c, c): NaN stays NaN
SSA_HD double ssa_norm_clip(double v, double c) { return v < -c ? -c : (v > c ? c : v); }
// VecNormalize.normalize_obs / normalize_reward of one value, with sd = ssa_norm_sd(var, epsilon) of the statistic
// (the division inlined: it runs once per element)
SSA_HD double ssa_norm_sd(double var, double eps) { return ssa_sqrt(var + eps); }
SSA_HD double ssa_norm_obs(double v, double mean, double sd, double clip) { return ssa_norm_clip(ssa_div_i(v - mean, sd), clip); }
SSA_HD double ssa_norm_reward(double r, double sd, double clip) { return ssa_norm_clip(ssa_div_i(r, sd), clip); }
// VecNormalize._update_reward: returns * gamma + reward
SSA_HD double ssa_norm_return(double ret, double gamma, double r) { return ret * gamma + r; }
