// twin.cpp — HOST build of the product's device arithmetic (ssa_gym_b200/csrc/*.h), for tests only.
//
// The sm_100a kernels and this file include the same __host__ __device__ headers, which are built
// from correctly rounded primitives with explicit FMAs and compiled with contraction disabled on
// both sides.  The tests therefore demand BIT-EXACT agreement between the GPU and this twin at any
// problem size, and compare the twin against the independent oracle (oracle/, libm + reference
// operation order, pinned to golden vectors generated from the reference's own functions) at
// tolerance.  This file is test infrastructure: the product never links or loads it, there is no
// CPU fallback behind the C ABI.
//
// The per-object flow below is the single-threaded statement of what one 16-lane team of
// ssa_ukf_kernels.cu does; every arithmetic step is a call into the shared headers.
#include <stdint.h>
#include <string.h>

#include "../../include/ssa_ukf.h"
#include "../../ssa_gym_b200/csrc/ssa_math.h"
#include "../../ssa_gym_b200/csrc/ssa_meas.h"
#include "../../ssa_gym_b200/csrc/ssa_orbit.h"
#include "../../ssa_gym_b200/csrc/ssa_rng.h"
#include "../../ssa_gym_b200/csrc/ssa_ukf_core.h"

namespace {

struct ObjIO {
  double* x_true;   // [6]
  double* x;        // [6]
  double* P;        // [21] packed upper
  int32_t* status;
  int32_t* infl;
  const double* z_noise;  // [3] or null
  double* obs;      // [12]
  double* dpos; double* dvel; double* spos; double* svel; double* trace;
  double* z_true;   // [3]
  double* y;        // [3]
  double* S;        // [9]
  double* sigmas_h; // [39]
  uint8_t* visible; uint8_t* updated;
};

void fail_object(ObjIO& o, int code) {
  o.x[0] = o.x[1] = o.x[2] = SSA_XFAIL_POS;
  o.x[3] = o.x[4] = o.x[5] = SSA_XFAIL_VEL;
  for (int e = 0; e < SSA_NP; ++e) o.P[e] = 0.0;
  for (int i = 0; i < 6; ++i) o.P[ssa_pidx(i, i)] = i < 3 ? SSA_XFAIL_POS : SSA_XFAIL_VEL;
  *o.status |= SSA_ST_FAILED | code;
}

void object_step(const ssa_ukf_cfg& cfg, const ssa_obs& ob, int flags, bool tasked, ObjIO& o) {
  double sig[SSA_NSIG][6];  // sigmas_f
  bool have_sig = false;
  double U[SSA_NP];

  if (flags & SSA_STEP_TRUTH) {
    double xt[6];
    const int exc = ssa_fx(o.x_true, cfg.dt, xt);
    for (int i = 0; i < 6; ++i) o.x_true[i] = xt[i];
    if (exc) *o.status |= SSA_ST_TRUTHEXC;
  }

  if ((flags & SSA_STEP_PREDICT) && !(*o.status & SSA_ST_FAILED)) {
    const int infl = ssa_robust_chol6(o.P, 1, cfg.lam_plus_n, U);
    if (infl < 0) {
      fail_object(o, SSA_ST_LINALG);
    } else {
      if (infl > 0) *o.infl += 1;
      double f[SSA_NSIG][6];
      int exc = 0;
      for (int k = 0; k < SSA_NSIG; ++k) {
        double s[6];
        ssa_sigma_point(o.x, U, k, s);
        exc |= ssa_fx(s, cfg.dt, f[k]);
      }
      if (exc) {
        fail_object(o, SSA_ST_FXEXC);
      } else {
        double xb[6], yv[SSA_NSIG][6], Pn[SSA_NP];
        for (int i = 0; i < 6; ++i) xb[i] = ssa_wmean13(&f[0][0], 6, i, cfg.Wm);
        for (int k = 0; k < SSA_NSIG; ++k)
          for (int i = 0; i < 6; ++i) yv[k][i] = f[k][i] - xb[i];
        for (int i = 0; i < 6; ++i)
          for (int j = i; j < 6; ++j)
            Pn[ssa_pidx(i, j)] = ssa_wcov13(&yv[0][0], 6, i, &yv[0][0], 6, j, cfg.Wc) + cfg.Q[6 * i + j];
        int nan = 0;
        for (int i = 0; i < 6; ++i) { o.x[i] = xb[i]; nan |= ssa_isnan(xb[i]); }
        for (int e = 0; e < SSA_NP; ++e) o.P[e] = Pn[e];
        int code = nan ? SSA_ST_NAN : 0;
        if (cfg.resample_after_predict) {
          const int infl2 = ssa_robust_chol6(o.P, 1, cfg.lam_plus_n, U);
          if (infl2 < 0) code |= SSA_ST_LINALG;
          else if (infl2 > 0) *o.infl += 1;
        }
        if (code) {
          fail_object(o, code);
        } else {
          for (int k = 0; k < SSA_NSIG; ++k) {
            if (cfg.resample_after_predict) ssa_sigma_point(o.x, U, k, sig[k]);
            else for (int i = 0; i < 6; ++i) sig[k][i] = f[k][i];
          }
          have_sig = true;
        }
      }
    }
  }

  const bool want_upd = (flags & SSA_STEP_UPDATE_ALL) || ((flags & SSA_STEP_UPDATE_ACT) && tasked);
  const bool want_meas = want_upd || (flags & SSA_STEP_EPILOGUE);
  double zt_aer[3] = {0, 0, 0};
  int visible = 0;
  if (want_meas) {
    ssa_hx_aer(o.x_true, &ob, zt_aer);
    visible = zt_aer[1] >= cfg.obs_limit;  // SS2:424
    if (o.visible) *o.visible = (uint8_t)visible;
  }
  if (o.updated) *o.updated = 0;

  if (want_upd && !(*o.status & SSA_ST_FAILED)) {
    double zt[3];
    for (int a = 0; a < 3; ++a) zt[a] = (cfg.obs_type == SSA_OBS_AER) ? zt_aer[a] : o.x_true[a];
    if (o.z_true) for (int a = 0; a < 3; ++a) o.z_true[a] = zt[a];  // SS2:298 (written even if not visible)
    if (visible) {
      if (!have_sig) {
        // stand-alone update: filterpy's sigmas_f after predict() are exactly sigma_points(x, P)
        const int infl = ssa_robust_chol6(o.P, 1, cfg.lam_plus_n, U);
        if (infl < 0) { fail_object(o, SSA_ST_LINALG | SSA_ST_IN_UPDATE); goto epilogue; }
        for (int k = 0; k < SSA_NSIG; ++k) ssa_sigma_point(o.x, U, k, sig[k]);
      }
      double z[3];
      for (int a = 0; a < 3; ++a) z[a] = zt[a] + (o.z_noise ? o.z_noise[a] : 0.0);
      double zs[SSA_NSIG][3], rz[SSA_NSIG][3], dx[SSA_NSIG][6], zp[3], Sm[9];
      if (cfg.obs_type == SSA_OBS_AER) {
        double uvw[SSA_NSIG][3], zm[3];
        for (int k = 0; k < SSA_NSIG; ++k) ssa_hx_aer(sig[k], &ob, zs[k], uvw[k]);  // uvw = the topocentric vector (ssa_meas.h)
        for (int a = 0; a < 3; ++a) zm[a] = ssa_wmean13(&uvw[0][0], 3, a, cfg.Wm);
        ssa_uvw2aer(zm, zp);
        for (int k = 0; k < SSA_NSIG; ++k) ssa_residual_aer(zs[k], zp, rz[k]);
        for (int a = 0; a < 3; ++a)
          for (int b = a; b < 3; ++b) {
            const double s = ssa_wouter13(&rz[0][0], 3, a, &rz[0][0], 3, b, cfg.Wc);
            Sm[3 * a + b] = s + cfg.R[3 * a + b];
            Sm[3 * b + a] = s + cfg.R[3 * b + a];
          }
      } else {
        for (int k = 0; k < SSA_NSIG; ++k) for (int a = 0; a < 3; ++a) zs[k][a] = sig[k][a];
        for (int a = 0; a < 3; ++a) zp[a] = ssa_wmean13(&zs[0][0], 3, a, cfg.Wm);
        for (int k = 0; k < SSA_NSIG; ++k) for (int a = 0; a < 3; ++a) rz[k][a] = zs[k][a] - zp[a];
        for (int a = 0; a < 3; ++a)
          for (int b = 0; b < 3; ++b)
            Sm[3 * a + b] = ssa_wcov13(&rz[0][0], 3, a, &rz[0][0], 3, b, cfg.Wc) + cfg.R[3 * a + b];
      }
      for (int k = 0; k < SSA_NSIG; ++k) for (int i = 0; i < 6; ++i) dx[k][i] = sig[k][i] - o.x[i];
      double Pxz[6][3], SI[9], K[6][3], T[3][6], yr[3];
      for (int i = 0; i < 6; ++i)
        for (int a = 0; a < 3; ++a) Pxz[i][a] = ssa_wouter13(&dx[0][0], 6, i, &rz[0][0], 3, a, cfg.Wc);
      const int ok = ssa_inv3(Sm, SI);
      if (cfg.obs_type == SSA_OBS_AER) ssa_residual_aer(z, zp, yr);
      else for (int a = 0; a < 3; ++a) yr[a] = z[a] - zp[a];
      double xn[6];
      int nan = 0;
      for (int i = 0; i < 6; ++i) {
        for (int a = 0; a < 3; ++a)
          K[i][a] = ssa_fma(Pxz[i][2], SI[6 + a], ssa_fma(Pxz[i][1], SI[3 + a], ssa_mul(Pxz[i][0], SI[a])));
        for (int a = 0; a < 3; ++a)
          T[a][i] = ssa_fma(Sm[3 * a + 2], K[i][2], ssa_fma(Sm[3 * a + 1], K[i][1], ssa_mul(Sm[3 * a], K[i][0])));
        xn[i] = o.x[i] + ssa_fma(K[i][2], yr[2], ssa_fma(K[i][1], yr[1], ssa_mul(K[i][0], yr[0])));
        nan |= ssa_isnan(xn[i]);
      }
      for (int i = 0; i < 6; ++i)
        for (int j = i; j < 6; ++j) {
          const int e = ssa_pidx(i, j);
          o.P[e] = o.P[e] - ssa_fma(K[i][2], T[2][j], ssa_fma(K[i][1], T[1][j], ssa_mul(K[i][0], T[0][j])));
        }
      for (int i = 0; i < 6; ++i) o.x[i] = xn[i];
      if (o.y) for (int a = 0; a < 3; ++a) o.y[a] = yr[a];
      if (o.S) for (int e = 0; e < 9; ++e) o.S[e] = Sm[e];
      if (o.sigmas_h) for (int k = 0; k < SSA_NSIG; ++k) for (int a = 0; a < 3; ++a) o.sigmas_h[3 * k + a] = zs[k][a];
      if (o.updated) *o.updated = 1;
      if (!ok) fail_object(o, SSA_ST_LINALG | SSA_ST_IN_UPDATE);
      else if (nan) fail_object(o, SSA_ST_NAN | SSA_ST_IN_UPDATE);
    }
  }

epilogue:
  if (flags & SSA_STEP_EPILOGUE) {
    for (int i = 0; i < 6; ++i) { o.obs[i] = o.x[i]; o.obs[6 + i] = o.P[ssa_pidx(i, i)]; }
    double d[6];
    for (int i = 0; i < 6; ++i) d[i] = o.x[i] - o.x_true[i];
    *o.dpos = ssa_sqrt(ssa_fma(d[2], d[2], ssa_fma(d[1], d[1], ssa_mul(d[0], d[0]))));
    *o.dvel = ssa_sqrt(ssa_fma(d[5], d[5], ssa_fma(d[4], d[4], ssa_mul(d[3], d[3]))));
    *o.spos = ssa_sqrt((o.P[0] + o.P[6]) + o.P[11]);
    *o.svel = ssa_sqrt((o.P[15] + o.P[18]) + o.P[20]);
    *o.trace = ssa_trace6(o.P, 1);
  }
}

}  // namespace

extern "C" {

// Batch step over N objects (arrays in host AoS layout; P packed [N][21]).
int twin_step(const ssa_ukf_cfg* cfg, const double* M, int flags, double* x_true, double* x, double* P,
              int32_t* status, int32_t* infl, const int32_t* actions, const double* z_noise, double* obs,
              double* dpos, double* dvel, double* spos, double* svel, double* trace, double* z_true, double* y,
              double* S, double* sigmas_h, uint8_t* visible, uint8_t* updated) {
  ssa_obs ob0;
  for (int i = 0; i < 9; ++i) { ob0.M[i] = M[i]; ob0.T[i] = cfg->T[i]; }
  for (int i = 0; i < 3; ++i) ob0.obs_itrs[i] = cfg->obs_itrs[i];
  const int N = cfg->n_objects, m = cfg->m;
#pragma omp parallel for schedule(dynamic, 64)
  for (int n = 0; n < N; ++n) {
    ssa_obs ob = ob0;
    if (flags & SSA_STEP_M_PER_ENV) for (int i = 0; i < 9; ++i) ob.M[i] = M[(size_t)(n / m) * 9 + i];  // M is [E][9]
    ObjIO o;
    o.x_true = x_true + 6 * (size_t)n; o.x = x + 6 * (size_t)n; o.P = P + SSA_NP * (size_t)n;
    o.status = status + n; o.infl = infl + n;
    o.z_noise = z_noise ? z_noise + 3 * (size_t)n : nullptr;
    o.obs = obs + 12 * (size_t)n;
    o.dpos = dpos + n; o.dvel = dvel + n; o.spos = spos + n; o.svel = svel + n; o.trace = trace + n;
    o.z_true = z_true ? z_true + 3 * (size_t)n : nullptr;
    o.y = y ? y + 3 * (size_t)n : nullptr;
    o.S = S ? S + 9 * (size_t)n : nullptr;
    o.sigmas_h = sigmas_h ? sigmas_h + 39 * (size_t)n : nullptr;
    o.visible = visible ? visible + n : nullptr;
    o.updated = updated ? updated + n : nullptr;
    const bool tasked = actions && (actions[n / m] == (n % m));
    object_step(*cfg, ob, flags, tasked, o);
  }
  return 0;
}

// ---- unit entry points for component tests ----------------------------------------------------
void twin_fx(const double* x, double dt, double* out, int32_t* exc, int n) {
  for (int i = 0; i < n; ++i) exc[i] = ssa_fx(x + 6 * i, dt, out + 6 * i);
}
void twin_rv2coe(const double* x, double* coe, int32_t* exc, int n) {
  for (int i = 0; i < n; ++i) exc[i] = ssa_rv2coe(x + 6 * i, coe + 6 * i);
}
void twin_coe2rv(const double* coe, double* x, int n) {
  for (int i = 0; i < n; ++i) ssa_coe2rv(coe + 6 * i, x + 6 * i);
}
void twin_hx_aer(const double* x, const double* M, const double* obs_itrs, const double* T, double* out, int n) {
  ssa_obs ob;
  for (int i = 0; i < 9; ++i) { ob.M[i] = M[i]; ob.T[i] = T[i]; }
  for (int i = 0; i < 3; ++i) ob.obs_itrs[i] = obs_itrs[i];
  for (int i = 0; i < n; ++i) ssa_hx_aer(x + 6 * i, &ob, out + 3 * i);
}
void twin_aer2uvw(const double* a, double* u, int n) { for (int i = 0; i < n; ++i) ssa_aer2uvw(a + 3 * i, u + 3 * i); }
void twin_uvw2aer(const double* u, double* a, int n) { for (int i = 0; i < n; ++i) ssa_uvw2aer(u + 3 * i, a + 3 * i); }
void twin_residual_aer(const double* a, const double* b, double* c, int n) {
  for (int i = 0; i < n; ++i) ssa_residual_aer(a + 3 * i, b + 3 * i, c + 3 * i);
}
// P packed [n][21] -> U packed [n][21]; ret[n] = inflation attempt (-1 failed)
void twin_robust_chol(const double* P, double lam, double* U, int32_t* ret, int n) {
  for (int i = 0; i < n; ++i) ret[i] = ssa_robust_chol6(P + 21 * i, 1, lam, U + 21 * i);
}
void twin_inv3(const double* S, double* SI, int32_t* ok, int n) {
  for (int i = 0; i < n; ++i) ok[i] = ssa_inv3(S + 9 * i, SI + 9 * i);
}
// determinants of packed symmetric 6x6 matrices [n][21] (agent_shannon: ssa_env_reduce_kernel / ssa_det_kernel)
void twin_det6_sym(const double* P, double* out, int n) {
  for (int i = 0; i < n; ++i) out[i] = ssa_det6_sym(P + 21 * (size_t)i, 1);
}
// agent_shannon's score log(det / prev) in the device's arithmetic
void twin_log_ratio(const double* det, const double* prev, double* out, int n) {
  for (int i = 0; i < n; ++i) out[i] = ssa_log(ssa_div(det[i], prev[i]));
}
#define TW1(name, fn) \
  void name(const double* x, double* y, int n) { for (int i = 0; i < n; ++i) y[i] = fn(x[i]); }
TW1(twin_sin, ssa_sin) TW1(twin_cos, ssa_cos) TW1(twin_tan, ssa_tan) TW1(twin_atan, ssa_atan)
TW1(twin_asin, ssa_asin) TW1(twin_acos, ssa_acos) TW1(twin_exp, ssa_exp) TW1(twin_log, ssa_log)
TW1(twin_sinh, ssa_sinh) TW1(twin_cosh, ssa_cosh) TW1(twin_tanh, ssa_tanh) TW1(twin_atanh, ssa_atanh)
TW1(twin_asinh, ssa_asinh) TW1(twin_acosh, ssa_acosh) TW1(twin_pow23, ssa_pow23)
void twin_atan2(const double* y, const double* x, double* z, int n) { for (int i = 0; i < n; ++i) z[i] = ssa_atan2(y[i], x[i]); }
void twin_pymod(const double* y, const double* x, double* z, int n) { for (int i = 0; i < n; ++i) z[i] = ssa_pymod(y[i], x[i]); }

// acceptance rule of the catalog generator (ssa_orbit_eval_kernel + ssa_orbit_accept_kernel)
void twin_orbit_gen_eval(const double* cand, int K, const double* table, int n, double step_s, const double* obs_itrs,
                         const double* T, double obs_limit, double min_alt, int first_window, int max_gap, uint8_t* accept,
                         double* elev, double* alt) {
#pragma omp parallel for
  for (int c = 0; c < K; ++c) {
    int all_alt = 1, all_vis = 1, any_gap = 0, first = 0, run = 0, longest = 0, bad = 0;
    for (int i = 0; i < n; ++i) {
      ssa_obs ob;
      memcpy(ob.obs_itrs, obs_itrs, 24); memcpy(ob.T, T, 72); memcpy(ob.M, table + (size_t)i * 9, 72);
      double x[6], xi[3], z[3];
      const int exc = ssa_fx(cand + (size_t)c * 6, ssa_mul(step_s, (double)i), x);
      for (int j = 0; j < 3; ++j) xi[j] = ssa_fma(x[2], ob.M[6 + j], ssa_fma(x[1], ob.M[3 + j], ssa_mul(x[0], ob.M[j])));
      const double h = ssa_ecef_altitude(xi);
      ssa_hx_aer(x, &ob, z);
      const int vis = z[1] >= obs_limit;
      if (elev) elev[(size_t)c * n + i] = z[1];
      if (alt) alt[(size_t)c * n + i] = h;
      all_alt &= (h > min_alt); bad |= exc; all_vis &= vis;
      if (i < first_window) first += vis;
      if (!vis) { any_gap = 1; run += 1; longest = run > longest ? run : longest; } else run = 0;
    }
    int ok = 0;
    if (all_alt && !bad) ok = any_gap ? (first > 0 && longest < max_gap) : all_vis;
    accept[c] = (uint8_t)ok;
  }
}

// diagnostics of ssa_diag_kernel on host-layout arrays (P packed [N][21])
void twin_diagnostics(int N, const double* x_true, const double* x, const double* P, const double* y, const double* S,
                      const uint8_t* updated, double* nees, double* nis, uint8_t* flags) {
  for (int n = 0; n < N; ++n) {
    double d[6];
    for (int i = 0; i < 6; ++i) d[i] = x_true[n * 6 + i] - x[n * 6 + i];
    nees[n] = ssa_nees6(P + (size_t)n * SSA_NP, 1, d);
    double v = ssa_nan();
    int f = 0;
    if (updated[n]) {
      v = ssa_nis3(S + (size_t)n * 9, y + (size_t)n * 3, &f);
      f |= 0x80;
    }
    nis[n] = v;
    flags[n] = (uint8_t)f;
  }
}

// ---- episodic device mode: the draws of k_env_reset / k_env_begin (ssa_rng.h) -------------------------------------
// (re)draw the environments with done[e] != 0 (all when done is null); host layout: x_true / x_filter [N][6],
// P packed [N][21]; sig = x_sigma[6], z_sigma[3], packed P0[21]
void twin_env_reset(int E, int m, const uint64_t* seeds, uint32_t* episode, int32_t* step_idx, const uint8_t* done,
                    const double* orbits, int n_orbits, const double* sig, double* x_true, double* x_filter, double* P,
                    int32_t* status, int32_t* infl) {
  for (int e = 0; e < E; ++e) {
    if (done && !done[e]) continue;
    const uint32_t k0 = (uint32_t)(seeds[e] & 0xffffffffu), k1 = (uint32_t)(seeds[e] >> 32), ep = episode[e];
    for (int j = 0; j < m; ++j) {
      const size_t obj = (size_t)e * m + j;
      const uint32_t row = ssa_draw_orbit(k0, k1, ep, (uint32_t)j, (uint32_t)n_orbits);
      double n6[6];
      ssa_draw_x(k0, k1, ep, (uint32_t)j, n6);
      for (int i = 0; i < 6; ++i) {
        const double xt = orbits[(size_t)row * 6 + i];
        x_true[obj * 6 + i] = xt;
        x_filter[obj * 6 + i] = xt + ssa_mul(n6[i], sig[i]);
      }
      for (int q = 0; q < SSA_NP; ++q) P[obj * SSA_NP + q] = sig[9 + q];
      status[obj] = 0;
      infl[obj] = 0;
    }
    episode[e] = ep + 1u;
    step_idx[e] = 0;
  }
}
// measurement noise of step step_idx[e] + 1, [N][3]
void twin_env_noise(int E, int m, const uint64_t* seeds, const uint32_t* episode, const int32_t* step_idx, const double* sig,
                    double* z_noise) {
  for (int e = 0; e < E; ++e)
    for (int j = 0; j < m; ++j) {
      double n3[3];
      ssa_draw_z((uint32_t)(seeds[e] & 0xffffffffu), (uint32_t)(seeds[e] >> 32), episode[e] - 1u, (uint32_t)j,
                 (uint32_t)(step_idx[e] + 1), n3);
      for (int a = 0; a < 3; ++a) z_noise[((size_t)e * m + j) * 3 + a] = ssa_mul(n3[a], sig[6 + a]);
    }
}
// n standard normals of stream (key, ep = 0, STREAM_Z, j = i, step = 0): for the statistical tests
void twin_normals(uint64_t seed, double* out, int n) {
  for (int i = 0; i + 2 < n + 3; i += 3) {
    double n3[3];
    ssa_draw_z((uint32_t)(seed & 0xffffffffu), (uint32_t)(seed >> 32), 0u, (uint32_t)(i / 3), 0u, n3);
    for (int a = 0; a < 3 && i + a < n; ++a) out[i + a] = n3[a];
  }
}
void twin_philox(const uint32_t* ctr, const uint32_t* key, uint32_t* out) {
  const ssa_u4 r = ssa_philox4x32(ctr[0], ctr[1], ctr[2], ctr[3], key[0], key[1]);
  for (int i = 0; i < 4; ++i) out[i] = r.v[i];
}

}  // extern "C"
