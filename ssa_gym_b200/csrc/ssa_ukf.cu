// ssa_ukf.cu — sm_100a kernels and the C ABI (include/ssa_ukf.h) of the UKF hot path.
//
// Three device implementations of the step live here (DESIGN.md §3), all bit-identical to the host twin
// (tests/twin/twin.cpp):
//  * the TILE PIPELINE (default; ssa_tile.cuh): k_factor -> k_predict_tile -> k_refactor -> k_update_tile.  A CTA owns 32
//    consecutive objects; the propagated sigma set and the measurement sigma set live in its shared memory only, the
//    state tile arrives by one 2-D TMA load (cp.async.bulk.tensor + mbarrier), propagation / measurement tasks are mapped
//    (object, sigma index) so that a warp holds the sigma points of at most four objects, the per-object linear algebra
//    is spread over the tile's threads with every sum over the 13 sigma points in a fixed sequential order.  Two measured
//    alternates of the same arithmetic (both slower, DESIGN.md §3): SSA_UKF_KERNEL=tile2 folds the two factorisations
//    into the tile kernels (two launches, the factor never in HBM), SSA_UKF_KERNEL=fused runs the whole catalog step as
//    ONE launch (k_step_tile: 0.73 KB of DRAM traffic per object-step);
//  * the SPLIT PIPELINE (SSA_UKF_KERNEL=split, and always for the RL-mode update of one tasked object per environment and
//    for the book-version filter): k_factor, k_fx, k_ut, k_hx, k_update(_staged) — one thread per object for the small
//    linear algebra, one thread per (sigma point, object) for fx / hx, intermediates in global scratch;
//  * the TEAM KERNEL ssa_step_kernel (SSA_UKF_KERNEL=team): one launch, one object per 16-lane team.
// The chain of a step is linked by programmatic dependent launch (griddepcontrol) and replayed as a CUDA graph
// (ssa_ukf_step, _step_pinned, _rollout_step).
//
// HBM layout: struct-of-arrays fp64, leading dimension ld = N rounded up to 32:
//   xt[6][ld]  x[6][ld]  P[21][ld] (packed upper triangle; one [33][ld] tensor)  + per-object scalars [ld]
// AoS only where the reference's own array layout is the interface (obs[N][12], z_noise[N][3], ...).
//
// Also here: the device-resident episodic mode (k_env_reset / k_env_begin: vectorised reset and on-the-fly noise with
// the counter-based generator of ssa_rng.h), the per-env and per-shard reward reductions and heuristic taskers,
// consistency diagnostics (NEES / NIS / innovation bounds, Durbin-Watson / autocorrelation), the single-copy snapshot of
// the drop-in env's histories and the catalog generator's acceptance kernels.
//
// No tensor cores: nothing here is a dense contraction (13-term sums of 6x6 outer products).
// No libdevice transcendental, no implicit FMA contraction (compiled with -fmad=false, every FMA is explicit in the
// shared headers).
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <new>
#include <numeric>
#include <vector>

#include <cuda.h>
#include <utility>
#include <cudaTypedefs.h>

#include "../../include/ssa_ukf.h"
#include "ssa_math.h"
#include "ssa_frames.h"
#include "ssa_meas.h"
#include "ssa_orbit.h"
#include "ssa_rng.h"
#include "ssa_ukf_core.h"

namespace {

constexpr int kTeam = 16;
constexpr int kTeamsPerCta = 8;
constexpr int kCtaThreads = kTeam * kTeamsPerCta;  // 128
// Per-team shared workspace, in doubles.  The stride is 16 (mod 32) 4-byte banks so that the two
// teams of a warp touch disjoint bank halves when they read the same logical element.
constexpr int WS_SG = 0;     // [13][6] propagated sigmas -> deviations -> dx
constexpr int WS_ZZ = 78;    // [13][3] uvw -> measurement residuals
constexpr int WS_XB = 117;   // [6] current filter mean
constexpr int WS_PN = 123;   // [21] current packed covariance
constexpr int WS_XT = 144;   // [6] current true state
constexpr int WS_ZM = 150;   // [3] uvw mean
constexpr int WS_SS = 153;   // [9] innovation covariance
constexpr int WS_PX = 162;   // [18] cross covariance
constexpr int WS_KK = 180;   // [18] gain
constexpr int WS_TT = 198;   // [18] S K^T
constexpr int kWsStride = 216;  // 432 words == 16 (mod 32)
static_assert(WS_TT + 18 <= kWsStride, "workspace overflow");
static_assert((kWsStride * 2) % 32 == 16, "team stride must be 16 banks (mod 32)");

__constant__ unsigned char c_pi[21] = {0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 4, 4, 5};
__constant__ unsigned char c_pj[21] = {0, 1, 2, 3, 4, 5, 1, 2, 3, 4, 5, 2, 3, 4, 5, 3, 4, 5, 4, 5, 5};
__constant__ unsigned char c_sa[6] = {0, 0, 0, 1, 1, 2};
__constant__ unsigned char c_sb[6] = {0, 1, 2, 1, 2, 2};

struct KParams {
  // state (SoA, leading dimension ld)
  double* xt; double* x; double* P;
  int32_t* status; int32_t* infl;
  // inputs
  const int32_t* actions;  // [E]
  const double* z_noise;   // [N][3] AoS
  const double* Menv;      // device-resident trans_matrix: [E][9] per env (Mstride 9) or one for all (Mstride 0); null = p.ob.M
  int Mstride;
  const int32_t* Mstep;    // episodic mode: Menv is the whole trans_matrix table [n][9], env e uses row Mstep[e] + Mbias
  int Mbias, Mrows;
  // outputs
  double* obs;             // [N][12] AoS
  double* dpos; double* dvel; double* spos; double* svel; double* trace;  // [ld]
  double* z_true;          // [N][3]
  double* y;               // [N][3]
  double* S;               // [N][9]
  double* sigmas_h;        // [N][39]
  uint8_t* visible; uint8_t* updated;
  int32_t* status_out;     // optional copy of the status word in the double-buffered output block (step_host)
  // scratch of the split pipeline (SoA, leading dimension ld)
  double* U;      // [21][ld] packed Cholesky factor of (lambda+n) P
  double* F;      // [13][6][ld] propagated sigma points
  double* ZS;     // [13][3][ld] measurement sigma points
  double* UVW;    // [13][3][ld] their Cartesian images
  double* ZT;     // [3][ld] az/el/range of the TRUE state
  int32_t* code;  // [ld] failure code raised in this step
  int32_t* exc;   // [ld] OR of the fx exception flags of the 13 sigma points
  long ld;
  long lds;   // leading dimension of the scratch arrays (= chunk capacity)
  long obj0;  // first object of the chunk this launch works on
  int Nc;     // objects in the chunk
  int N, E, m, flags, obs_type, resample;
  double dt, lam, obs_limit;
  double Wm[13], Wc[13];
  const double* qr;  // device constants: packed Q (21, upper triangle) then R (9, row-major)
  const uint8_t* env_gate;  // episodic refresh after an auto-reset: [E] mask, only the objects of these environments are touched
  ssa_obs ob;
};

__device__ __forceinline__ void team_sync(unsigned mask) { __syncwarp(mask); }

// trans_matrix of environment e when it is device-resident (p.Menv != null)
__device__ __forceinline__ const double* env_M(const KParams& p, long e) {
  if (p.Mstep) {
    int row = p.Mstep[e] + p.Mbias;
    row = row < p.Mrows ? row : p.Mrows - 1;
    return p.Menv + 9L * row;
  }
  return p.Menv + e * p.Mstride;
}

// The fused step.  Stage selection by p.flags (uniform across the grid).
__global__ void __launch_bounds__(kCtaThreads) ssa_step_kernel(const KParams p) {
  __shared__ double ws_all[kTeamsPerCta * kWsStride];
  const int lane32 = threadIdx.x & 31;
  const int lane = threadIdx.x & 15;
  const unsigned tmask = 0xFFFFu << (lane32 & 16);
  const int team = threadIdx.x >> 4;
  const long obj = (long)blockIdx.x * kTeamsPerCta + team;
  if (obj >= p.N) return;  // a team leaves together
  if (p.env_gate && !p.env_gate[obj / p.m]) return;  // (one object per team: the team leaves together)
  double* ws = ws_all + team * kWsStride;
  const int flags = p.flags;
  const long ld = p.ld;
  const int truth_lane = (lane32 & 16) + 13;

  // ---- stage the object's state into the team workspace ---------------------------------------
  if (lane < 6) {
    ws[WS_XB + lane] = p.x[lane * ld + obj];
    ws[WS_XT + lane] = p.xt[lane * ld + obj];
  }
  ws[WS_PN + lane] = p.P[lane * ld + obj];
  if (lane < 5) ws[WS_PN + 16 + lane] = p.P[(16 + lane) * ld + obj];
  int status = p.status[obj];
  int infl_count = 0;
  int code = 0;
  team_sync(tmask);

  double x[6], xt[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) { x[i] = ws[WS_XB + i]; xt[i] = ws[WS_XT + i]; }

  double sg[6];   // this lane's sigma point for the update (sigmas_f[lane])
  double U[SSA_NP];
  bool have_sig = false;

  // ---- truth propagation + predict ----------------------------------------------------------------
  if (flags & (SSA_STEP_TRUTH | SSA_STEP_PREDICT)) {
    bool live = (flags & SSA_STEP_PREDICT) && !(status & SSA_ST_FAILED);
    if (live) {
      const int infl = ssa_robust_chol6(ws + WS_PN, 1, p.lam, U);
      if (infl < 0) { live = false; code |= SSA_ST_LINALG; }
      else if (infl > 0) infl_count += 1;
    }
    double s[6], f[6];
    if (live && lane < 13) {
      ssa_sigma_point(x, U, lane, s);
    } else {
#pragma unroll
      for (int i = 0; i < 6; ++i) s[i] = xt[i];
    }
    const int exc = ssa_fx(s, p.dt, f);
    if (flags & SSA_STEP_TRUTH) {
      if (lane == 13) {
#pragma unroll
        for (int i = 0; i < 6; ++i) ws[WS_XT + i] = f[i];
        if (exc) status |= SSA_ST_TRUTHEXC;
      }
      status = __shfl_sync(tmask, status, truth_lane);
    }
    if (live) {
      if (lane < 13) {
#pragma unroll
        for (int i = 0; i < 6; ++i) ws[WS_SG + lane * 6 + i] = f[i];
      }
      if (__any_sync(tmask, (lane < 13) && exc)) { live = false; code |= SSA_ST_FXEXC; }
    }
    team_sync(tmask);
    if (live) {
      // unscented transform: mean (lanes 0..5), deviations (lanes 0..12), covariance (21 elements)
      if (lane < 6) ws[WS_XB + lane] = ssa_wmean13(ws + WS_SG, 6, lane, p.Wm);
      team_sync(tmask);
      int nan = 0;
#pragma unroll
      for (int i = 0; i < 6; ++i) { x[i] = ws[WS_XB + i]; nan |= ssa_isnan(x[i]); }
      if (lane < 13) {
#pragma unroll
        for (int i = 0; i < 6; ++i) ws[WS_SG + lane * 6 + i] = f[i] - x[i];
      }
      team_sync(tmask);
      {
        const int i = c_pi[lane], j = c_pj[lane];
        ws[WS_PN + lane] = ssa_wcov13(ws + WS_SG, 6, i, ws + WS_SG, 6, j, p.Wc) + __ldg(p.qr + lane);
        if (lane < 5) {
          const int i2 = c_pi[16 + lane], j2 = c_pj[16 + lane];
          ws[WS_PN + 16 + lane] = ssa_wcov13(ws + WS_SG, 6, i2, ws + WS_SG, 6, j2, p.Wc) + __ldg(p.qr + 16 + lane);
        }
      }
      team_sync(tmask);
      if (nan) code |= SSA_ST_NAN;
      if (p.resample) {
        const int infl2 = ssa_robust_chol6(ws + WS_PN, 1, p.lam, U);
        if (infl2 < 0) code |= SSA_ST_LINALG;
        else if (infl2 > 0) infl_count += 1;
      }
      if (!code) {
        if (p.resample) {
          ssa_sigma_point(x, U, lane < 13 ? lane : 0, sg);
        } else {
#pragma unroll
          for (int i = 0; i < 6; ++i) sg[i] = f[i];
        }
        have_sig = true;
      }
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) xt[i] = ws[WS_XT + i];
  }

  if (code) {  // filter_error(): sentinels (SS2:369-382)
    status |= SSA_ST_FAILED | code;
    if (lane < 6) ws[WS_XB + lane] = lane < 3 ? SSA_XFAIL_POS : SSA_XFAIL_VEL;
    {
      const int i = c_pi[lane], j = c_pj[lane];
      ws[WS_PN + lane] = (i == j) ? (i < 3 ? SSA_XFAIL_POS : SSA_XFAIL_VEL) : 0.0;
      if (lane < 5) {
        const int i2 = c_pi[16 + lane], j2 = c_pj[16 + lane];
        ws[WS_PN + 16 + lane] = (i2 == j2) ? (i2 < 3 ? SSA_XFAIL_POS : SSA_XFAIL_VEL) : 0.0;
      }
    }
    team_sync(tmask);
#pragma unroll
    for (int i = 0; i < 6; ++i) x[i] = ws[WS_XB + i];
    code = 0;
  }

  // ---- measurement: truth elevation (visibility) on lane 13, sigma measurements on lanes 0..12 ----
  bool want_upd = (flags & SSA_STEP_UPDATE_ALL) != 0;
  if (flags & SSA_STEP_UPDATE_ACT) want_upd = want_upd || (p.actions[obj / p.m] == (int)(obj % p.m));
  const bool want_meas = want_upd || (flags & SSA_STEP_EPILOGUE);
  int updated = 0;
  if (want_meas) {
    bool do_upd = want_upd && !(status & SSA_ST_FAILED);
    if (do_upd && !have_sig) {
      // stand-alone update: sigmas_f of filterpy after predict() are exactly sigma_points(x, P)
      const int infl = ssa_robust_chol6(ws + WS_PN, 1, p.lam, U);
      if (infl < 0) { do_upd = false; code |= SSA_ST_LINALG | SSA_ST_IN_UPDATE; }
      else ssa_sigma_point(x, U, lane < 13 ? lane : 0, sg);
    }
    double hin[6], zk[3];
    const bool sigma_lane = do_upd && lane < 13;
#pragma unroll
    for (int i = 0; i < 6; ++i) hin[i] = sigma_lane ? sg[i] : xt[i];
    ssa_obs ob = p.ob;
    if (p.Menv) {
#pragma unroll
      for (int i = 0; i < 9; ++i) ob.M[i] = env_M(p, obj / p.m)[i];
    }
    double enz[3];
    ssa_hx_aer(hin, &ob, zk, enz);
    // broadcast the truth measurement of lane 13
    double zt[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) zt[a] = __shfl_sync(tmask, zk[a], truth_lane);
    const int visible = zt[1] >= p.obs_limit;  // SS2:424
    if (lane == 13) p.visible[obj] = (uint8_t)visible;
    if (p.obs_type == SSA_OBS_XYZ) {
#pragma unroll
      for (int a = 0; a < 3; ++a) { zt[a] = xt[a]; zk[a] = hin[a]; }
    }
    if (do_upd) {
      if (p.z_true && lane < 3) p.z_true[obj * 3 + lane] = zt[lane];  // SS2:298
      if (visible) {
        double z[3], zp[3], rz[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) z[a] = zt[a] + (p.z_noise ? p.z_noise[obj * 3 + a] : 0.0);
        if (p.obs_type == SSA_OBS_AER) {
          if (lane < 13) {
#pragma unroll
            for (int a = 0; a < 3; ++a) ws[WS_ZZ + lane * 3 + a] = enz[a];
          }
          team_sync(tmask);
          if (lane < 3) ws[WS_ZM + lane] = ssa_wmean13(ws + WS_ZZ, 3, lane, p.Wm);
          team_sync(tmask);
          double zm[3];
#pragma unroll
          for (int a = 0; a < 3; ++a) zm[a] = ws[WS_ZM + a];
          ssa_uvw2aer(zm, zp);
          ssa_residual_aer(zk, zp, rz);
        } else {
          if (lane < 13) {
#pragma unroll
            for (int a = 0; a < 3; ++a) ws[WS_ZZ + lane * 3 + a] = zk[a];
          }
          team_sync(tmask);
          if (lane < 3) ws[WS_ZM + lane] = ssa_wmean13(ws + WS_ZZ, 3, lane, p.Wm);
          team_sync(tmask);
#pragma unroll
          for (int a = 0; a < 3; ++a) { zp[a] = ws[WS_ZM + a]; rz[a] = zk[a] - zp[a]; }
        }
        if (lane < 13) {
#pragma unroll
          for (int a = 0; a < 3; ++a) ws[WS_ZZ + lane * 3 + a] = rz[a];
#pragma unroll
          for (int i = 0; i < 6; ++i) ws[WS_SG + lane * 6 + i] = sg[i] - x[i];
        }
        team_sync(tmask);
        // 6 unique elements of S and 18 of Pxz over 16 lanes (two rounds)
#pragma unroll
        for (int round = 0; round < 2; ++round) {
          const int e = lane + 16 * round;
          if (e < 6) {
            const int a = c_sa[e], b = c_sb[e];
            double s;
            if (p.obs_type == SSA_OBS_AER) s = ssa_wouter13(ws + WS_ZZ, 3, a, ws + WS_ZZ, 3, b, p.Wc);
            else s = ssa_wcov13(ws + WS_ZZ, 3, a, ws + WS_ZZ, 3, b, p.Wc);
            ws[WS_SS + 3 * a + b] = s + __ldg(p.qr + 21 + 3 * a + b);
            if (a != b) {
              double s2 = s;
              if (p.obs_type != SSA_OBS_AER) s2 = ssa_wcov13(ws + WS_ZZ, 3, b, ws + WS_ZZ, 3, a, p.Wc);
              ws[WS_SS + 3 * b + a] = s2 + __ldg(p.qr + 21 + 3 * b + a);
            }
          } else if (e < 24) {
            const int i = (e - 6) / 3, a = (e - 6) % 3;
            ws[WS_PX + (e - 6)] = ssa_wouter13(ws + WS_SG, 6, i, ws + WS_ZZ, 3, a, p.Wc);
          }
        }
        team_sync(tmask);
        double Sm[9], SI[9], yr[3];
#pragma unroll
        for (int e = 0; e < 9; ++e) Sm[e] = ws[WS_SS + e];
        const int ok = ssa_inv3(Sm, SI);
        if (p.obs_type == SSA_OBS_AER) ssa_residual_aer(z, zp, yr);
        else {
#pragma unroll
          for (int a = 0; a < 3; ++a) yr[a] = z[a] - zp[a];
        }
        if (lane < 6) {
          double K[3];
          const double px0 = ws[WS_PX + lane * 3], px1 = ws[WS_PX + lane * 3 + 1], px2 = ws[WS_PX + lane * 3 + 2];
#pragma unroll
          for (int a = 0; a < 3; ++a) {
            K[a] = ssa_fma(px2, SI[6 + a], ssa_fma(px1, SI[3 + a], ssa_mul(px0, SI[a])));
            ws[WS_KK + lane * 3 + a] = K[a];
          }
#pragma unroll
          for (int a = 0; a < 3; ++a)
            ws[WS_TT + a * 6 + lane] =
                ssa_fma(Sm[3 * a + 2], K[2], ssa_fma(Sm[3 * a + 1], K[1], ssa_mul(Sm[3 * a], K[0])));
          ws[WS_XB + lane] = x[lane < 6 ? lane : 0] + ssa_fma(K[2], yr[2], ssa_fma(K[1], yr[1], ssa_mul(K[0], yr[0])));
        }
        team_sync(tmask);
#pragma unroll
        for (int round = 0; round < 2; ++round) {
          const int e = lane + 16 * round;
          if (e < 21) {
            const int i = c_pi[e], j = c_pj[e];
            const double kt = ssa_fma(ws[WS_KK + i * 3 + 2], ws[WS_TT + 12 + j],
                                      ssa_fma(ws[WS_KK + i * 3 + 1], ws[WS_TT + 6 + j],
                                              ssa_mul(ws[WS_KK + i * 3], ws[WS_TT + j])));
            ws[WS_PN + e] = ws[WS_PN + e] - kt;
          }
        }
        int nan = 0;
#pragma unroll
        for (int i = 0; i < 6; ++i) { x[i] = ws[WS_XB + i]; nan |= ssa_isnan(x[i]); }
        if (p.y && lane < 3) p.y[obj * 3 + lane] = yr[lane];
        if (p.S && lane < 9) p.S[obj * 9 + lane] = Sm[lane];
        if (p.sigmas_h && lane < 13) {
#pragma unroll
          for (int a = 0; a < 3; ++a) p.sigmas_h[obj * 39 + lane * 3 + a] = zk[a];
        }
        updated = 1;
        if (!ok) code |= SSA_ST_LINALG | SSA_ST_IN_UPDATE;
        else if (nan) code |= SSA_ST_NAN | SSA_ST_IN_UPDATE;
        team_sync(tmask);
      }
    }
    if (code) {
      status |= SSA_ST_FAILED | code;
      if (lane < 6) ws[WS_XB + lane] = lane < 3 ? SSA_XFAIL_POS : SSA_XFAIL_VEL;
      {
        const int i = c_pi[lane], j = c_pj[lane];
        ws[WS_PN + lane] = (i == j) ? (i < 3 ? SSA_XFAIL_POS : SSA_XFAIL_VEL) : 0.0;
        if (lane < 5) {
          const int i2 = c_pi[16 + lane], j2 = c_pj[16 + lane];
          ws[WS_PN + 16 + lane] = (i2 == j2) ? (i2 < 3 ? SSA_XFAIL_POS : SSA_XFAIL_VEL) : 0.0;
        }
      }
      team_sync(tmask);
#pragma unroll
      for (int i = 0; i < 6; ++i) x[i] = ws[WS_XB + i];
    }
  }
  if (lane == 13 && p.updated) p.updated[obj] = (uint8_t)updated;

  // ---- write back state ----------------------------------------------------------------------------
  team_sync(tmask);
  if (lane < 6) {
    p.x[lane * ld + obj] = ws[WS_XB + lane];
    if (flags & SSA_STEP_TRUTH) p.xt[lane * ld + obj] = ws[WS_XT + lane];
  }
  p.P[lane * ld + obj] = ws[WS_PN + lane];
  if (lane < 5) p.P[(16 + lane) * ld + obj] = ws[WS_PN + 16 + lane];
  if (lane == 0) {
    p.status[obj] = status;
    if (p.status_out) p.status_out[obj] = status;
    if (infl_count) p.infl[obj] += infl_count;
  }

  // ---- epilogue: observation row, errors, trace (results.py:36-72) -------------------------------
  if (flags & SSA_STEP_EPILOGUE) {
    if (lane < 12) {
      const int d = lane < 6 ? 0 : lane - 6;
      p.obs[obj * 12 + lane] = lane < 6 ? ws[WS_XB + lane] : ws[WS_PN + ssa_pidx(d, d)];
    }
    if (lane == 12 || lane == 13) {
      const int o = (lane == 12) ? 0 : 3;
      const double d0 = x[o] - xt[o], d1 = x[o + 1] - xt[o + 1], d2 = x[o + 2] - xt[o + 2];
      const double dd = ssa_sqrt(ssa_fma(d2, d2, ssa_fma(d1, d1, ssa_mul(d0, d0))));
      const double sp = (lane == 12) ? ssa_sqrt((ws[WS_PN + 0] + ws[WS_PN + 6]) + ws[WS_PN + 11])
                                     : ssa_sqrt((ws[WS_PN + 15] + ws[WS_PN + 18]) + ws[WS_PN + 20]);
      if (lane == 12) { p.dpos[obj] = dd; p.spos[obj] = sp; }
      else { p.dvel[obj] = dd; p.svel[obj] = sp; }
    }
    if (lane == 14) p.trace[obj] = ssa_trace6(ws + WS_PN, 1);
  }
}


// =====================================================================================================
// Split pipeline (default): five launches per step, each with the thread mapping that suits its stage.
//   k_factor   one thread per object      robust Cholesky of (lambda+n) P                  -> U
//   k_fx       one thread per (k, object) fx of sigma point k (k = 13: the TRUE state)     -> F, xt
//   k_ut       one thread per object      unscented transform, +Q, re-factorisation        -> x, P, U
//   k_hx       one thread per (k, object) hx of re-drawn sigma point k (k = 13: truth)     -> ZS, UVW, ZT
//   k_update   one thread per object      S, Pxz, K, state/covariance update, epilogue     -> x, P, obs...
// Objects are the fastest-varying thread index everywhere, so every load/store of the SoA arrays is a
// fully coalesced 256-byte warp access; a block of k_fx / k_hx works on ONE sigma index k, so the
// row-of-U selection is uniform.  All lanes do distinct useful work (no redundant factorisation, no idle
// lanes), intermediates stay in L2 for C2-sized batches.  The arithmetic of every output element is the
// same sequence of rounded operations as in the team kernel and the host twin.
// =====================================================================================================
#ifndef SSA_CHOL_INLINE
#define SSA_CHOL_INLINE true
#endif
constexpr int kSplitThreads = 128;
#ifndef SSA_FX_THREADS
#define SSA_FX_THREADS 128
#endif
#ifndef SSA_OBJ_THREADS
#define SSA_OBJ_THREADS 128
#endif
constexpr int kFxThreads = SSA_FX_THREADS;    // block size of the per-sigma-point kernels k_fx / k_hx
constexpr int kObjThreads = SSA_OBJ_THREADS;  // block size of the per-object kernels k_factor / k_ut
#ifndef SSA_LB_FX
#define SSA_LB_FX 8
#endif
#ifndef SSA_LB_UT
#define SSA_LB_UT 2
#endif
#ifndef SSA_LB_UPD
#define SSA_LB_UPD 4
#endif
#ifndef SSA_LB_FAC
#define SSA_LB_FAC 4
#endif
#ifndef SSA_LB_HX
#define SSA_LB_HX 10
#endif

// Programmatic dependent launch: the five kernels of a step form a chain on one stream.  Each kernel lets its
// successor be scheduled as soon as all of its own blocks are resident (launch_dependents) and waits for the
// complete, flushed results of its predecessor before touching memory (wait) — so the successor's launch latency
// and block ramp-up overlap the predecessor's tail.  Both instructions are no-ops for a normal launch.
__device__ __forceinline__ void pdl_prologue() {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
}

// (Measured and not kept: the factor in a per-thread row of shared memory instead of registers / local memory, to run
// 6-10 blocks per SM instead of 4: ptxas keeps the unrolled factorisation in registers either way and spills under the
// tighter cap; k_factor 0.082 -> 0.095 .. 0.161 ms at 1 M objects.)
__global__ void __launch_bounds__(kObjThreads, SSA_LB_FAC * 128 / kObjThreads) k_factor(const KParams p) {
  pdl_prologue();
  const long loc = (long)blockIdx.x * blockDim.x + threadIdx.x;  // index inside the chunk
  if (loc >= p.Nc) return;
  const long obj = p.obj0 + loc;
  const long lds = p.lds;
  const long ld = p.ld;
  const int st = p.status[obj];
  int code = 0;
  p.exc[obj] = 0;
  const bool predict = (p.flags & SSA_STEP_PREDICT) != 0;
  const bool update = (p.flags & (SSA_STEP_UPDATE_ALL | SSA_STEP_UPDATE_ACT)) != 0;
  if ((predict || update) && !(st & SSA_ST_FAILED)) {
    double U[SSA_NP];
    const int r = ssa_robust_chol6_t<SSA_CHOL_INLINE>(p.P + obj, ld, p.lam, U);
    if (r < 0) {
      code = SSA_ST_LINALG | (predict ? 0 : SSA_ST_IN_UPDATE);
    } else {
      if (r > 0 && predict) p.infl[obj] += 1;
#pragma unroll
      for (int e = 0; e < SSA_NP; ++e) p.U[e * lds + loc] = U[e];
    }
  }
  p.code[obj] = code;
}

// sigma point k of object obj from x and the stored factor: s = x +- U[r, :]
__device__ __forceinline__ void load_sigma(const KParams& p, long loc, int k, const double* x, double* s) {
  const long lds = p.lds;
  const int r = (k == 0) ? -1 : (k - 1) % 6;
  const bool minus = k > 6;
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    double u = 0.0;
    if (r >= 0 && r <= j) u = p.U[ssa_pidx(r, j) * lds + loc];
    s[j] = minus ? (x[j] - u) : (x[j] + u);
  }
}

__global__ void __launch_bounds__(kFxThreads, SSA_LB_FX * 128 / kFxThreads) k_fx(const KParams p) {
  pdl_prologue();
  const long loc = (long)blockIdx.x * blockDim.x + threadIdx.x;  // index inside the chunk
  if (loc >= p.Nc) return;
  const long obj = p.obj0 + loc;
  const long lds = p.lds;
  const int k = blockIdx.y;  // uniform per block
  const long ld = p.ld;
  double s[6], f[6];
  if (k == 13) {
    if (!(p.flags & SSA_STEP_TRUTH)) return;
#pragma unroll
    for (int i = 0; i < 6; ++i) s[i] = p.xt[i * ld + obj];
    const int exc = ssa_fx(s, p.dt, f);
#pragma unroll
    for (int i = 0; i < 6; ++i) p.xt[i * ld + obj] = f[i];
    if (exc) atomicOr(p.status + obj, SSA_ST_TRUTHEXC);
    return;
  }
  if (!(p.flags & SSA_STEP_PREDICT)) return;
  if ((p.status[obj] & SSA_ST_FAILED) || p.code[obj]) return;
  double x[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) x[i] = p.x[i * ld + obj];
  load_sigma(p, loc, k, x, s);
  const int exc = ssa_fx(s, p.dt, f);
#pragma unroll
  for (int i = 0; i < 6; ++i) p.F[(k * 6 + i) * lds + loc] = f[i];
  if (exc) atomicOr(p.exc + obj, 1);
}

__device__ __forceinline__ void store_sentinel(const KParams& p, long obj) {
  const long ld = p.ld;
#pragma unroll
  for (int i = 0; i < 6; ++i) p.x[i * ld + obj] = i < 3 ? SSA_XFAIL_POS : SSA_XFAIL_VEL;
#pragma unroll
  for (int i = 0; i < 6; ++i)
#pragma unroll
    for (int j = i; j < 6; ++j)
      p.P[ssa_pidx(i, j) * ld + obj] = (i == j) ? (i < 3 ? SSA_XFAIL_POS : SSA_XFAIL_VEL) : 0.0;
}

// ---- bulk-async staging (TMA engine, 1-D cp.async.bulk) of the per-object columns ---------------------------------
// A thread-per-object kernel on a C2-sized batch has ~1 warp per SM sub-partition: nothing hides a load, and the
// ~100 L2 round trips that k_update makes one after the other (the compiler cannot hoist 135 loads into 128
// registers) were 70 % of its run time (ncu: long_scoreboard 13.8 of 19 cycles per issue).  The staged variants
// fetch every row tile the block will read with a few 2-D TMA tile loads (box = 32 objects x up to 81 rows of the
// [rows][ld] SoA arrays; the scratch arrays and the state arrays are each ONE tensor, so k_update needs three
// loads), all in flight together, completion counted by one mbarrier; every thread then reads only
// its own column of the tile, so no further synchronisation is needed.  The arithmetic is the same template body.
// MEASURED on B200 (k_update -> k_update_staged): 24.3 -> 16.4 us at C2, 75 -> 66 us at 125 k objects, 0.493 ->
// 0.433 ms at 1 M.  The same treatment of k_ut (78 rows of F) did not pay (12.3 -> 12.3 us at C2, 0.221 -> 0.248 ms
// at 1 M: that kernel already front-loads its loads with 246 registers and is bounded by the Cholesky chain), so
// k_ut stays a plain global-load kernel.
// (A first version issued one 1-D bulk copy per row from different lanes: UBLKCP is a uniform-datapath
// instruction, so the compiler serialised the 135 copies through an ELECT loop, ~1000 extra instructions.)
__device__ __forceinline__ uint32_t smem_u32(const void* q) { return (uint32_t)__cvta_generic_to_shared(q); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// one TMA tile load: box (32 columns x the map's row count) at column c0, row c1 of a [rows][ld] fp64 array
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* tm, int c0, int c1, uint64_t* bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
                   smem_u32(dst)),
               "l"((uint64_t)tm), "r"(c0), "r"(c1), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok)
                 : "r"(smem_u32(bar)), "r"(parity)
                 : "memory");
  } while (!ok);
}

// The unscented transform of the propagated points (UKF.predict, then the fork's re-draw).  F = the thread's column of
// the propagated sigma set, fs = its row stride.
__device__ __forceinline__ void ut_body(const KParams& p, long loc, long obj, const double* F, long fs) {
  const long lds = p.lds;
  const long ld = p.ld;
  int st = p.status[obj];
  if (st & SSA_ST_FAILED) return;
  int code = p.code[obj];
  if (!code && p.exc[obj]) code = SSA_ST_FXEXC;
  if (!code) {
    double xb[6];
    int nan = 0;
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      double acc = ssa_mul(p.Wm[0], F[i * fs]);
#pragma unroll
      for (int k = 1; k < SSA_NSIG; ++k) acc = ssa_fma(p.Wm[k], F[(k * 6 + i) * fs], acc);
      xb[i] = acc;
      nan |= ssa_isnan(acc);
    }
    double Pn[SSA_NP];
#pragma unroll
    for (int e = 0; e < SSA_NP; ++e) Pn[e] = 0.0;
#pragma unroll
    for (int k = 0; k < SSA_NSIG; ++k) {
      double y[6];
#pragma unroll
      for (int i = 0; i < 6; ++i) y[i] = F[(k * 6 + i) * fs] - xb[i];
#pragma unroll
      for (int i = 0; i < 6; ++i)
#pragma unroll
        for (int j = i; j < 6; ++j) Pn[ssa_pidx(i, j)] = ssa_fma(y[i], ssa_mul(p.Wc[k], y[j]), Pn[ssa_pidx(i, j)]);
    }
#pragma unroll
    for (int e = 0; e < SSA_NP; ++e) Pn[e] = Pn[e] + __ldg(p.qr + e);
#pragma unroll
    for (int i = 0; i < 6; ++i) p.x[i * ld + obj] = xb[i];
#pragma unroll
    for (int e = 0; e < SSA_NP; ++e) p.P[e * ld + obj] = Pn[e];
    if (nan) code |= SSA_ST_NAN;
    if (p.resample) {
      double U[SSA_NP];
      const int r2 = ssa_robust_chol6_t<SSA_CHOL_INLINE>(Pn, 1, p.lam, U);
      if (r2 < 0) code |= SSA_ST_LINALG;
      else {
        if (r2 > 0) p.infl[obj] += 1;
#pragma unroll
        for (int e = 0; e < SSA_NP; ++e) p.U[e * lds + loc] = U[e];
      }
    }
  }
  if (code) {
    store_sentinel(p, obj);
    p.status[obj] = st | SSA_ST_FAILED | code;
  }
  p.code[obj] = code;
}

__global__ void __launch_bounds__(kObjThreads, SSA_LB_UT * 128 / kObjThreads) k_ut(const KParams p) {
  pdl_prologue();
  const long loc = (long)blockIdx.x * blockDim.x + threadIdx.x;  // index inside the chunk
  if (loc >= p.Nc) return;
  if (!(p.flags & SSA_STEP_PREDICT)) return;
  ut_body(p, loc, p.obj0 + loc, p.F + loc, p.lds);
}

// Rows of the scratch tensor [U 21][F 78][ZS 39][UVW 39][ZT 3] and of the state tensor [xt 6][x 6][P 21]
constexpr int SC_U = 0, SC_ZS = 99, SC_ROWS = 180;
constexpr int ST_ROWS = 33;

// object index of update slot `idx` (ALL: identity; ACT: the tasked object of env idx), -1 if none
__device__ __forceinline__ long upd_object(const KParams& p, long lidx) {
  if (p.flags & SSA_STEP_UPDATE_ALL) return lidx < p.Nc ? p.obj0 + lidx : -1;
  if (p.flags & SSA_STEP_UPDATE_ACT) {  // one slot per environment that intersects the chunk
    const long e = p.obj0 / p.m + lidx;
    if (e > (p.obj0 + p.Nc - 1) / p.m || e >= p.E) return -1;
    const int a = p.actions[e];
    if (a < 0 || a >= p.m) return -1;
    const long obj = e * (long)p.m + a;
    return (obj >= p.obj0 && obj < p.obj0 + p.Nc) ? obj : -1;  // the tasked object may live in another chunk
  }
  return -1;
}

#ifndef SSA_HX_INLINE
#define SSA_HX_INLINE true
#endif
// measurement of the TRUE state of object idx (scratch column loc): visibility (SS2:418-425), z_true into the scratch row ZT
__device__ __forceinline__ void hx_truth(const KParams& p, const long idx, const long loc, const bool store_zt) {
  double xt[3], zt[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) xt[i] = p.xt[i * p.ld + idx];
  ssa_obs ob = p.ob;
  if (p.Menv) {
#pragma unroll
    for (int i = 0; i < 9; ++i) ob.M[i] = env_M(p, idx / p.m)[i];
  }
  ssa_hx_aer_t<SSA_HX_INLINE>(xt, &ob, zt);
  if (store_zt) {
#pragma unroll
    for (int a = 0; a < 3; ++a) p.ZT[a * p.lds + loc] = zt[a];
  }
  p.visible[idx] = (uint8_t)(zt[1] >= p.obs_limit);
}

__global__ void __launch_bounds__(kFxThreads, SSA_LB_HX * 128 / kFxThreads) k_hx(const KParams p) {
  pdl_prologue();
  const long lidx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  const int k = blockIdx.y;
  const long ld = p.ld;
  const long lds = p.lds;
  if (k == 13) {  // truth measurement of every object: visibility (SS2:418-425) and z_true
    if (lidx >= p.Nc) return;
    const long idx = p.obj0 + lidx;
    if (p.env_gate && !p.env_gate[idx / p.m]) return;
    hx_truth(p, idx, lidx, true);
    return;
  }
  const long obj = upd_object(p, lidx);
  if (obj < 0) return;
  const long loc = obj - p.obj0;
  if ((p.status[obj] & SSA_ST_FAILED) || p.code[obj]) return;
  double s[6];
  if (p.resample) {  // sigmas_f = points re-drawn around the prior; book version: the propagated points
    double x[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) x[i] = p.x[i * ld + obj];
    load_sigma(p, loc, k, x, s);
  } else {
#pragma unroll
    for (int i = 0; i < 6; ++i) s[i] = p.F[(k * 6 + i) * lds + loc];
  }
  double z[3];
  if (p.obs_type == SSA_OBS_AER) {
    double uvw[3];
    ssa_obs ob = p.ob;
    if (p.Menv) {
#pragma unroll
      for (int i = 0; i < 9; ++i) ob.M[i] = env_M(p, obj / p.m)[i];
    }
    ssa_hx_aer_t<SSA_HX_INLINE>(s, &ob, z, uvw);
#pragma unroll
    for (int a = 0; a < 3; ++a) p.UVW[(k * 3 + a) * lds + loc] = uvw[a];
  } else {
#pragma unroll
    for (int a = 0; a < 3; ++a) z[a] = s[a];
  }
#pragma unroll
  for (int a = 0; a < 3; ++a) p.ZS[(k * 3 + a) * lds + loc] = z[a];
}

// Row offsets of the staged tile of k_update_staged
constexpr int UR_ZS = 0, UR_UVW = 39, UR_ZT = 78, UR_U = 81, UR_XT = 102, UR_X = 108, UR_P = 114, UR_ROWS = 135;

// UKF.update + epilogue of one object.  STAGED = false: every operand is read from global memory (k_update);
// STAGED = true: from the block's shared tile `sm` (already offset by the thread's column, row stride ss).
#ifndef SSA_UPD_INLINE
#define SSA_UPD_INLINE true
#endif
template <bool STAGED>
__device__ __forceinline__ void update_body(const KParams& p, long loc, long obj, const double* sm, int ss) {
  const long lds = p.lds;
  const long ld = p.ld;
  const int flags = p.flags;
#define V_ZS(e) (STAGED ? sm[(UR_ZS + (e)) * ss] : p.ZS[(e) * lds + loc])
#define V_UVW(e) (STAGED ? sm[(UR_UVW + (e)) * ss] : p.UVW[(e) * lds + loc])
#define V_U(e) (STAGED ? sm[(UR_U + (e)) * ss] : p.U[(e) * lds + loc])
#define V_P(e) (STAGED ? sm[(UR_P + (e)) * ss] : p.P[(e) * ld + obj])
#define V_X(e) (STAGED ? sm[(UR_X + (e)) * ss] : p.x[(e) * ld + obj])
#define V_XT(e) (STAGED ? sm[(UR_XT + (e)) * ss] : p.xt[(e) * ld + obj])
#define V_ZT(e) (STAGED ? sm[(UR_ZT + (e)) * ss] : p.ZT[(e) * lds + loc])
  int st = p.status[obj];
  bool want_upd = (flags & SSA_STEP_UPDATE_ALL) != 0;
  if (flags & SSA_STEP_UPDATE_ACT) want_upd = want_upd || (p.actions[obj / p.m] == (int)(obj % p.m));
  int updated = 0;
  int code = 0;
  // the state as the epilogue will see it: the prior, overwritten below by the update (or by the failure sentinel)
  double xe[6], dg[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) { xe[i] = V_X(i); dg[i] = V_P(ssa_pidx(i, i)); }
  if (want_upd && !(st & SSA_ST_FAILED)) {
    double zt[3];
    const int visible = p.visible[obj];
#pragma unroll
    for (int a = 0; a < 3; ++a) zt[a] = (p.obs_type == SSA_OBS_AER) ? V_ZT(a) : V_XT(a);
    if (p.z_true) {
#pragma unroll
      for (int a = 0; a < 3; ++a) p.z_true[obj * 3 + a] = zt[a];
    }
    if (p.code[obj]) {
      code = p.code[obj];  // stand-alone update whose factorisation failed
    } else if (visible) {
      double x[6], z[3], zp[3];
#pragma unroll
      for (int i = 0; i < 6; ++i) x[i] = xe[i];
#pragma unroll
      for (int a = 0; a < 3; ++a) z[a] = zt[a] + (p.z_noise ? p.z_noise[obj * 3 + a] : 0.0);
      if (p.obs_type == SSA_OBS_AER) {
        double zm[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) {
          double acc = ssa_mul(p.Wm[0], V_UVW(a));
#pragma unroll
          for (int k = 1; k < SSA_NSIG; ++k) acc = ssa_fma(p.Wm[k], V_UVW(k * 3 + a), acc);
          zm[a] = acc;
        }
        ssa_uvw2aer_t<SSA_UPD_INLINE>(zm, zp);
      } else {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
          double acc = ssa_mul(p.Wm[0], V_ZS(a));
#pragma unroll
          for (int k = 1; k < SSA_NSIG; ++k) acc = ssa_fma(p.Wm[k], V_ZS(k * 3 + a), acc);
          zp[a] = acc;
        }
      }
      double Ss[9], Pxz[18];
#pragma unroll
      for (int e = 0; e < 9; ++e) Ss[e] = 0.0;
#pragma unroll
      for (int e = 0; e < 18; ++e) Pxz[e] = 0.0;
      const bool from_f = !p.resample;
#ifndef SSA_UPD_UNROLL
#define SSA_UPD_UNROLL 13
#endif
#define SSA_STR_(x) #x
#define SSA_UNROLL_(n) _Pragma(SSA_STR_(unroll n))
      SSA_UNROLL_(SSA_UPD_UNROLL)
      for (int k = 0; k < SSA_NSIG; ++k) {
        double zk[3], rz[3], sk[6];
#pragma unroll
        for (int a = 0; a < 3; ++a) zk[a] = V_ZS(k * 3 + a);
        if (p.obs_type == SSA_OBS_AER) ssa_residual_aer(zk, zp, rz);
        else {
#pragma unroll
          for (int a = 0; a < 3; ++a) rz[a] = zk[a] - zp[a];
        }
        if (from_f) {
#pragma unroll
          for (int i = 0; i < 6; ++i) sk[i] = p.F[(k * 6 + i) * lds + loc];
        } else {  // sigma point k re-drawn around the prior: x +- U[r, :]
          const int r = (k == 0) ? -1 : (k - 1) % 6;
          const bool minus = k > 6;
#pragma unroll
          for (int j = 0; j < 6; ++j) {
            double u = 0.0;
            if (r >= 0 && r <= j) u = V_U(ssa_pidx(r, j));
            sk[j] = minus ? (x[j] - u) : (x[j] + u);
          }
        }
        if (p.obs_type == SSA_OBS_AER) {
#pragma unroll
          for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int b = a; b < 3; ++b) Ss[3 * a + b] = ssa_fma(p.Wc[k], ssa_mul(rz[a], rz[b]), Ss[3 * a + b]);
        } else {
#pragma unroll
          for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int b = 0; b < 3; ++b) Ss[3 * a + b] = ssa_fma(rz[a], ssa_mul(p.Wc[k], rz[b]), Ss[3 * a + b]);
        }
#pragma unroll
        for (int i = 0; i < 6; ++i) {
          const double dx = sk[i] - x[i];
#pragma unroll
          for (int a = 0; a < 3; ++a) Pxz[3 * i + a] = ssa_fma(p.Wc[k], ssa_mul(dx, rz[a]), Pxz[3 * i + a]);
        }
      }
      double Sm[9], SI[9], yr[3];
      if (p.obs_type == SSA_OBS_AER) {
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
          for (int b = a; b < 3; ++b) {
            Sm[3 * a + b] = Ss[3 * a + b] + __ldg(p.qr + 21 + 3 * a + b);
            Sm[3 * b + a] = Ss[3 * a + b] + __ldg(p.qr + 21 + 3 * b + a);
          }
      } else {
#pragma unroll
        for (int e = 0; e < 9; ++e) Sm[e] = Ss[e] + __ldg(p.qr + 21 + e);
      }
      const int ok = ssa_inv3_t<SSA_UPD_INLINE>(Sm, SI);
      if (p.obs_type == SSA_OBS_AER) ssa_residual_aer(z, zp, yr);
      else {
#pragma unroll
        for (int a = 0; a < 3; ++a) yr[a] = z[a] - zp[a];
      }
      double K[18], T[18];
      int nan = 0;
#pragma unroll
      for (int i = 0; i < 6; ++i) {
#pragma unroll
        for (int a = 0; a < 3; ++a)
          K[3 * i + a] = ssa_fma(Pxz[3 * i + 2], SI[6 + a], ssa_fma(Pxz[3 * i + 1], SI[3 + a], ssa_mul(Pxz[3 * i], SI[a])));
#pragma unroll
        for (int a = 0; a < 3; ++a)
          T[a * 6 + i] = ssa_fma(Sm[3 * a + 2], K[3 * i + 2], ssa_fma(Sm[3 * a + 1], K[3 * i + 1], ssa_mul(Sm[3 * a], K[3 * i])));
        const double xn = x[i] + ssa_fma(K[3 * i + 2], yr[2], ssa_fma(K[3 * i + 1], yr[1], ssa_mul(K[3 * i], yr[0])));
        nan |= ssa_isnan(xn);
        p.x[i * ld + obj] = xn;
        xe[i] = xn;
      }
#pragma unroll
      for (int i = 0; i < 6; ++i)
#pragma unroll
        for (int j = i; j < 6; ++j) {
          const int e = ssa_pidx(i, j);
          const double kt = ssa_fma(K[3 * i + 2], T[12 + j], ssa_fma(K[3 * i + 1], T[6 + j], ssa_mul(K[3 * i], T[j])));
          const double pn = V_P(e) - kt;
          p.P[e * ld + obj] = pn;
          if (i == j) dg[i] = pn;
        }
      if (p.y) {
#pragma unroll
        for (int a = 0; a < 3; ++a) p.y[obj * 3 + a] = yr[a];
      }
      if (p.S) {
#pragma unroll
        for (int e = 0; e < 9; ++e) p.S[obj * 9 + e] = Sm[e];
      }
      if (p.sigmas_h) {
#pragma unroll 1
        for (int e = 0; e < 39; ++e) p.sigmas_h[obj * 39 + e] = V_ZS(e);
      }
      updated = 1;
      if (!ok) code = SSA_ST_LINALG | SSA_ST_IN_UPDATE;
      else if (nan) code = SSA_ST_NAN | SSA_ST_IN_UPDATE;
    }
    if (code) {
      store_sentinel(p, obj);
#pragma unroll
      for (int i = 0; i < 6; ++i) xe[i] = dg[i] = (i < 3 ? SSA_XFAIL_POS : SSA_XFAIL_VEL);
      st |= SSA_ST_FAILED | code;
      p.status[obj] = st;
    }
  }
  if (p.updated) p.updated[obj] = (uint8_t)updated;
  if (p.status_out) p.status_out[obj] = st;
  if (flags & SSA_STEP_EPILOGUE) {
    double xt[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) xt[i] = V_XT(i);
#pragma unroll
    for (int i = 0; i < 6; ++i) { p.obs[obj * 12 + i] = xe[i]; p.obs[obj * 12 + 6 + i] = dg[i]; }
    const double d0 = xe[0] - xt[0], d1 = xe[1] - xt[1], d2 = xe[2] - xt[2];
    const double d3 = xe[3] - xt[3], d4 = xe[4] - xt[4], d5 = xe[5] - xt[5];
    p.dpos[obj] = ssa_sqrt_t<SSA_UPD_INLINE>(ssa_fma(d2, d2, ssa_fma(d1, d1, ssa_mul(d0, d0))));
    p.dvel[obj] = ssa_sqrt_t<SSA_UPD_INLINE>(ssa_fma(d5, d5, ssa_fma(d4, d4, ssa_mul(d3, d3))));
    p.spos[obj] = ssa_sqrt_t<SSA_UPD_INLINE>((dg[0] + dg[1]) + dg[2]);
    p.svel[obj] = ssa_sqrt_t<SSA_UPD_INLINE>((dg[3] + dg[4]) + dg[5]);
    p.trace[obj] = ((((dg[0] + dg[1]) + dg[2]) + dg[3]) + dg[4]) + dg[5];
  }
#undef V_ZS
#undef V_UVW
#undef V_U
#undef V_P
#undef V_X
#undef V_XT
#undef V_ZT
}

__global__ void __launch_bounds__(kSplitThreads, SSA_LB_UPD) k_update(const KParams p) {
  pdl_prologue();
  const long loc = (long)blockIdx.x * blockDim.x + threadIdx.x;  // index inside the chunk
  if (loc >= p.Nc) return;
  if (p.env_gate && !p.env_gate[(p.obj0 + loc) / p.m]) return;
  update_body<false>(p, loc, p.obj0 + loc, nullptr, 0);
}

// Launched instead of k_update for an update of EVERY object (SSA_STEP_UPDATE_ALL, resampled sigma points).
__global__ void __launch_bounds__(32) k_update_staged(const KParams p, const __grid_constant__ CUtensorMap tm_z,
                                                       const __grid_constant__ CUtensorMap tm_u,
                                                       const __grid_constant__ CUtensorMap tm_s) {
  extern __shared__ __align__(128) double tile[];  // [UR_ROWS][32], then the mbarrier
  pdl_prologue();
  uint64_t* bar = (uint64_t*)(tile + UR_ROWS * 32);
  const int col0 = blockIdx.x * 32;
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    mbar_expect_tx(bar, UR_ROWS * 256);
    tma_load_2d(tile + UR_ZS * 32, &tm_z, col0, SC_ZS, bar);               // ZS, UVW, ZT: 81 rows
    tma_load_2d(tile + UR_U * 32, &tm_u, col0, SC_U, bar);                 // U: 21 rows
    tma_load_2d(tile + UR_XT * 32, &tm_s, (int)p.obj0 + col0, 0, bar);     // xt, x, P: 33 rows
  }
  __syncwarp();
  const long loc = col0 + threadIdx.x;
  mbar_wait(bar, 0);
  if (loc >= p.Nc) return;
  update_body<true>(p, loc, p.obj0 + loc, tile + threadIdx.x, 32);
}

constexpr int kUpdStagedSmem = UR_ROWS * 32 * 8 + 16;
constexpr long kStagedMaxDefault = 1L << 40;

#include "ssa_tile.cuh"

// ---- per-environment reductions: reward/done and greedy taskers ------------------------------------
struct EnvParams {
  const double* dpos; const double* dvel; const double* spos; const double* trace;
  const uint8_t* visible;
  double* reward; uint8_t* done; int32_t* greedy; double* env_stats;  // env_stats[E][4]: max dpos, trinary, argmax spos, n_visible
  int32_t* step_idx;  // per-env step counters (used when step_index < 0)
  int E, m, reward_type, n_steps, step_index;
  int increment;    // episodic mode: step_idx[e] += 1 before it is used (the device owns the counters)
  int greedy_only;  // refresh greedy / env_stats only (after an auto-reset); reward and done stay
  const double* P; long ld;   // packed covariances (agent_shannon: determinants)
  const double* det_cur;      // [N] det P of the current covariances (ssa_det_kernel, thread per object)
  // agent_shannon's determinant history, keyed to the step index (see SSA_TASKER_SHANNON in ssa_ukf.h): det_last holds
  // det P of step det_step[e], det_prev the denominator of that step's ratio (det P of the step before it)
  double* det_prev;           // [N]
  double* det_last;           // [N]
  int32_t* det_step;          // [E] step index det_last belongs to (< 0: no history, ssa_ukf_reset)
  const uint8_t* reset_mask;  // episodic refresh after an auto-reset: only these environments are re-evaluated
  // episodic mode with the 'shaped' reward (null otherwise: the host finishes that reward from env_stats)
  double* rew_hist;           // [E][n_steps] rewards of the running episode, entry 0 = 0 (np.sum(rewards[:i]), SS2:345)
  int32_t* spos_prev;         // [E] argmax sigma_pos of the environment's previous step (SS2:348)
  const int32_t* act_in;      // [E] REQUESTED actions (SS2:348 compares them also on steps update_interval skips)
  uint8_t* truncated;         // [E] episodic mode: done raised by the step limit alone (null outside that mode)
};


struct ArgMax { double v; int i; };
__device__ __forceinline__ ArgMax am_better(ArgMax a, ArgMax b) {
  // np.argmax semantics: first maximum wins (lowest index among equal values)
  if (b.i < 0) return a;
  if (a.i < 0) return b;
  if (b.v > a.v || (b.v == a.v && b.i < a.i)) return b;
  return a;
}
__device__ __forceinline__ ArgMax am_warp(ArgMax a) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ArgMax b;
    b.v = __shfl_xor_sync(0xffffffffu, a.v, o);
    b.i = __shfl_xor_sync(0xffffffffu, a.i, o);
    a = am_better(a, b);
  }
  return a;
}

// det P of every object (agent_shannon), one thread per object: a chain of 6 divisions that would hold the per-environment
// reduction below at 4 CTAs per SM if it ran there on m of 128 threads (measured: 50 us per launch at E = 4096)
__global__ void __launch_bounds__(128) ssa_det_kernel(const double* __restrict__ P, long ld, int N, double* __restrict__ det_cur,
                                                      const uint8_t* __restrict__ env_gate, int m) {
  const long n = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N || (env_gate && !env_gate[n / m])) return;
  det_cur[n] = ssa_det6_sym(P + n, ld);
}

// WARP = false: one CTA per environment, threads stride over the m objects of the env (catalog-sized environments).
// WARP = true (m <= 64, the RL configurations: m = 10 .. 40): one WARP per environment, four environments per CTA, no
// shared memory and no barrier — with one CTA per 10-object environment 118 of 128 threads only took part in the
// shuffles (measured at E = 4096: 30 us per launch, two launches per episodic step).
template <bool WARP>
__device__ __forceinline__ void env_reduce_body(const EnvParams& p, const int e);
template <bool WARP>
__global__ void __launch_bounds__(128, 5) ssa_env_reduce_kernel(const EnvParams p) {
  const int e = WARP ? (int)(blockIdx.x * 4 + (threadIdx.x >> 5)) : (int)blockIdx.x;
  if (WARP && e >= p.E) return;
  // the refresh after an auto-reset concerns the re-drawn environments only: the others keep this step's results
  if (p.greedy_only && p.reset_mask && !p.reset_mask[e]) return;
  env_reduce_body<WARP>(p, e);
}
// WARP: the calling warp reduces environment e (its results go through slot threadIdx.x >> 5 of the shared scratch);
// else the whole CTA does.
template <bool WARP>
__device__ __forceinline__ void env_reduce_body(const EnvParams& p, const int e) {
  const int j0 = WARP ? (int)(threadIdx.x & 31) : (int)threadIdx.x, jstep = WARP ? 32 : (int)blockDim.x;
  const long base = (long)e * p.m;
  ArgMax a_trace{0.0, -1}, a_vtrace{0.0, -1}, a_vdpos{0.0, -1}, a_vdvel{0.0, -1}, a_spos{0.0, -1}, a_dpos{0.0, -1};
  ArgMax a_vaer{0.0, -1}, a_vshan{0.0, -1};
  int tri = 0, nvis = 0, vis_nonzero = 0;
  int step_i = p.step_index >= 0 ? p.step_index : p.step_idx[e];
  if (p.increment) step_i += 1;
  // agent_shannon's history: a later step than the stored one shifts it, the same step re-reads it (so that calling
  // the reduction again at one step gives the same picks), and step 0, an earlier step or no history restart it
  const int hist = p.det_step[e];
  const bool restart = step_i <= 0 || hist < 0 || step_i < hist, shift = !restart && step_i > hist;
  for (int j = j0; j < p.m; j += jstep) {
    const double dp = p.dpos[base + j], dv = p.dvel[base + j], sp = p.spos[base + j], tr = p.trace[base + j];
    const int vis = p.visible[base + j];
    // agent_shannon (agents.py:15-26): log(det P_i / det P_{i-1}); the first step of an episode has no P_{i-1} (the
    // reference reads row -1 of its history array there): the ratio is taken as 1
    // (det_cur null: the determinant is evaluated here — the RL-sized environments, one lane per object — instead of
    // by ssa_det_kernel: one launch fewer per episodic step)
    const double det = p.det_cur ? p.det_cur[base + j] : ssa_det6_sym(p.P + base + j, p.ld);
    double prev;
    if (restart) {
      prev = det;
      p.det_prev[base + j] = det;
      p.det_last[base + j] = det;
    } else if (shift) {
      prev = p.det_last[base + j];
      p.det_prev[base + j] = prev;
      p.det_last[base + j] = det;
    } else {
      prev = p.det_prev[base + j];
    }
    const double shan = ssa_log(ssa_div(det, prev));
    if (vis) {
      // agent_visible_greedy_aer (agents.py:57-63): the 'aer' observation's trace column after nan_to_num (SS2:839)
      const double tr_aer = (tr - tr == 0.0) ? tr : 0.001;
      a_vaer = am_better(a_vaer, ArgMax{tr_aer, j});
      // np.argmax treats NaN as the maximum (first NaN wins): a NaN score is ordered above everything
      const double sh = (shan == shan) ? shan : ssa_from_hilo(0x7ff00000, 0);
      a_vshan = am_better(a_vshan, ArgMax{sh, j});
    }
    a_trace = am_better(a_trace, ArgMax{tr, j});
    // sigma_pos = sqrt of a sum of covariance diagonal entries: NaN if update() left a negative one (only x is checked
    // for NaN there); np.argmax (the 'shaped' reward, SS2:348) orders a NaN first, as the Shannon column does
    a_spos = am_better(a_spos, ArgMax{(sp == sp) ? sp : ssa_from_hilo(0x7ff00000, 0), j});
    a_dpos = am_better(a_dpos, ArgMax{dp, j});
    if (vis) {
      a_vtrace = am_better(a_vtrace, ArgMax{tr, j});
      a_vdpos = am_better(a_vdpos, ArgMax{dp, j});
      a_vdvel = am_better(a_vdvel, ArgMax{dv, j});
      nvis += 1;
      vis_nonzero |= (j != 0);
    }
    tri += (dp < 1e4) + (dp < 1e7);  // results.py:431-433
  }
  __shared__ ArgMax sm[8][4];
  __shared__ int si[3][4];
  ArgMax r[8] = {am_warp(a_trace), am_warp(a_vtrace), am_warp(a_vdpos), am_warp(a_vdvel), am_warp(a_spos), am_warp(a_dpos),
                 am_warp(a_vaer), am_warp(a_vshan)};
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    tri += __shfl_xor_sync(0xffffffffu, tri, o);
    nvis += __shfl_xor_sync(0xffffffffu, nvis, o);
    vis_nonzero |= __shfl_xor_sync(0xffffffffu, vis_nonzero, o);
  }
  const int w = WARP ? 0 : (int)(threadIdx.x >> 5);
  if (!WARP) {
    if ((threadIdx.x & 31) == 0) {
      for (int q = 0; q < 8; ++q) sm[q][w] = r[q];
      si[0][w] = tri; si[1][w] = nvis; si[2][w] = vis_nonzero;
    }
    __syncthreads();
  } else if ((threadIdx.x & 31) == 0) {  // the warp's own results, slot of this warp (no other warp reads it)
    const int ww = threadIdx.x >> 5;
    for (int q = 0; q < 8; ++q) sm[q][ww] = r[q];
    si[0][ww] = tri; si[1][ww] = nvis; si[2][ww] = vis_nonzero;
  }
  if (WARP ? ((threadIdx.x & 31) == 0) : (threadIdx.x == 0)) {
    const int nw = blockDim.x >> 5;
    if (!WARP) {
      for (int q = 0; q < 8; ++q) for (int k = 1; k < nw; ++k) sm[q][0] = am_better(sm[q][0], sm[q][k]);
      for (int k = 1; k < nw; ++k) { si[0][0] += si[0][k]; si[1][0] += si[1][k]; si[2][0] |= si[2][k]; }
    }
    const int c0 = WARP ? (int)(threadIdx.x >> 5) : 0;  // column of the per-environment results
    const double max_dpos = sm[5][c0].v;
    if (p.increment) p.step_idx[e] = step_i;
    p.det_step[e] = step_i;
    // `if not np.any(visible)` tests the INDEX array: it is also false-y when the only visible
    // object is index 0 (agents.py:37) -> the reference samples a random action; we return -1.
    const int any_vis = si[2][c0];
    p.greedy[e * SSA_N_TASKERS + SSA_TASKER_NAIVE_GREEDY] = sm[0][c0].i;
    p.greedy[e * SSA_N_TASKERS + SSA_TASKER_VISIBLE_GREEDY] = any_vis ? sm[1][c0].i : -1;
    p.greedy[e * SSA_N_TASKERS + SSA_TASKER_POS_ERROR_GREEDY] = any_vis ? sm[2][c0].i : -1;
    p.greedy[e * SSA_N_TASKERS + SSA_TASKER_VEL_ERROR_GREEDY] = any_vis ? sm[3][c0].i : -1;
    p.greedy[e * SSA_N_TASKERS + SSA_TASKER_VISIBLE_GREEDY_AER] = any_vis ? sm[6][c0].i : -1;
    p.greedy[e * SSA_N_TASKERS + SSA_TASKER_SHANNON] = any_vis ? sm[7][c0].i : -1;
    const double trinary = ((double)si[0][c0] / (double)p.m) / 2.0;
    p.env_stats[e * 4 + 0] = max_dpos;
    p.env_stats[e * 4 + 1] = trinary;
    p.env_stats[e * 4 + 2] = (double)sm[4][c0].i;
    p.env_stats[e * 4 + 3] = (double)si[1][c0];
    if (p.greedy_only) return;
    double reward = 0.0;
    int done = 0;
    if (p.reward_type == SSA_REWARD_JONES) {  // SS2:324-336
      if (max_dpos > 5e6) { done = 1; reward = 0.0; }
      else if (max_dpos < 3e4) { done = 1; reward = 1.0; }
      else if (step_i + 1 >= p.n_steps) { done = 1; reward = 0.0; }
    } else if (p.reward_type == SSA_REWARD_TRINARY) {  // SS2:337-338
      reward = trinary;
    } else if (p.rew_hist) {  // 'shaped' in the episodic mode (SS2:339-351, episode.py step_reward)
      double* hist = p.rew_hist + (long)e * p.n_steps;
      if (max_dpos > 5e6) { done = 1; reward = 0.0; }
      else if (max_dpos < 3e4) { done = 1; reward = 1.0 - ssa_pairwise_sum(hist, step_i < p.n_steps ? step_i : p.n_steps); }
      else {
        const double r = ssa_div(1.0, (double)p.n_steps);
        reward = (p.act_in[e] == p.spos_prev[e]) ? r : -r;
      }
      if (step_i < p.n_steps) hist[step_i] = reward;  // (without auto-reset an episode may run past its last step)
      p.spos_prev[e] = sm[4][c0].i;
    } else {  // 'shaped' needs the reward history: finished on the host from env_stats (SS2:339-351)
      if (max_dpos > 5e6) { done = 1; reward = 0.0; }
      else if (max_dpos < 3e4) { done = 1; reward = 1.0; }
    }
    if (step_i + 1 >= p.n_steps) done = 1;  // SS2:353-354
    p.reward[e] = reward;
    p.done[e] = (uint8_t)done;
    // gym's TimeLimit rule: a lost or successful last step is a termination; 'trinary' ends at the step limit only
    if (p.truncated)
      p.truncated[e] = (uint8_t)(done && (p.reward_type == SSA_REWARD_TRINARY || !(max_dpos > 5e6 || max_dpos < 3e4)));
  }
}

// ---- device-resident episodic mode (SURVEY 8f-2): vectorised reset and on-the-fly noise, see ssa_rng.h -----------
struct RolloutParams {
  double* xt; double* x; double* P; long ld;   // state (SoA)
  int32_t* status; int32_t* infl;
  double* z_noise;                            // [N][3]
  const double* orbits; int n_orbits;         // catalog [n_orbits][6]
  const uint32_t* key;                        // [E][2] Philox key of each environment (from its seed)
  uint32_t* episode;                          // [E] resets performed so far
  int32_t* step_idx;                          // [E]
  int32_t* actions; int32_t* act_eff;         // [E] requested / effective (update_interval) actions
  const uint8_t* done;                        // [E] reset mask (null: every environment)
  const double* sig;                          // x_sigma[6], z_sigma[3], packed P0[21]
  double* rew_hist; int32_t* spos_prev;       // 'shaped' reward state (EnvParams), null for the other rewards
  const int32_t* greedy; const uint8_t* visible;  // greedy block [E][SSA_N_TASKERS], visibility [N] (device taskers)
  int tasker; double spoil_p;                 // ssa_ukf_rollout_tasker (SSA_TASKER_EXTERNAL: the caller's actions)
  int E, m, update_interval, n_steps;
  // final observations of the environments an auto-reset re-draws (env_terminal_rows); term null: not recorded
  const double* obs;                          // [N][12] observation rows of the output block
  double* term;                               // [E][m][12], or [E][m][4] with term_aer
  int term_aer;
  const double* table; int n_table;           // trans_matrix table (the 'aer' rows)
  ssa_obs ob;                                 // observer constants (M unused)
};

// the 'aer' observation of one object (SS2:834-840, vec_env.py _format_obs) from its [12] observation row: az / el /
// range of the filter mean x[0..2] through the trans_matrix M, np.trace's left-to-right sum of the diag P columns, and
// nan_to_num(nan = +-inf = 0.001) of the four values
__device__ __forceinline__ void obs_aer_row(const double* o, const double* M, const ssa_obs& ob, double* out) {
  double x[3], v[4];
#pragma unroll
  for (int k = 0; k < 3; ++k) x[k] = o[k];
  ssa_hx_aer_m<false>(x, M, ob.obs_itrs, ob.T, v);
  v[3] = ((((o[6] + o[7]) + o[8]) + o[9]) + o[10]) + o[11];
#pragma unroll
  for (int k = 0; k < 4; ++k) out[k] = (v[k] - v[k] == 0.0) ? v[k] : 0.001;
}

// the final observation of finished environment e, in the layout of the step, before env_reset_body re-draws it: its
// obs rows, or their 'aer' rows at the step index the episode ended on (read before env_reset_body zeroes it)
__device__ __forceinline__ void env_terminal_rows(const RolloutParams& p, const int e) {
  const int i = p.step_idx[e];
  const double* M = p.table + (long)(i < p.n_table - 1 ? i : p.n_table - 1) * 9;
  for (int j = threadIdx.x; j < p.m; j += blockDim.x) {
    const long obj = (long)e * p.m + j;
    if (p.term_aer) {
      obs_aer_row(p.obs + obj * 12, M, p.ob, p.term + obj * 4);
    } else {
#pragma unroll
      for (int k = 0; k < 12; ++k) p.term[obj * 12 + k] = p.obs[obj * 12 + k];
    }
  }
}

// start of a step: measurement noise of step i+1 for every object, the device tasker's pick (which replaces the
// requested action) and the effective action of every environment
__global__ void __launch_bounds__(128) k_env_begin(const RolloutParams p) {
  const long obj = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (obj >= (long)p.E * p.m) return;
  const int e = (int)(obj / p.m), j = (int)(obj % p.m);
  const int step = p.step_idx[e] + 1;
  double n3[3];
  ssa_draw_z(p.key[2 * e], p.key[2 * e + 1], p.episode[e] - 1u, (uint32_t)j, (uint32_t)step, n3);
#pragma unroll
  for (int a = 0; a < 3; ++a) p.z_noise[obj * 3 + a] = ssa_mul(n3[a], p.sig[6 + a]);
  if (j != 0) return;
  int a;
  if (p.tasker != SSA_TASKER_EXTERNAL) {
    a = ssa_tasker_pick(p.key[2 * e], p.key[2 * e + 1], p.episode[e] - 1u, (uint32_t)step, p.m, p.tasker,
                        p.greedy + (long)e * SSA_N_TASKERS, p.visible + obj, p.spoil_p);
    p.actions[e] = a;
  } else {
    a = p.actions[e];
  }
  p.act_eff[e] = (step % p.update_interval == 0) ? a : -1;  // SS2:292
}

// (re)draw the environments whose done flag is set (all of them when p.done is null): SS2:193-221
__device__ __forceinline__ void env_reset_body(const RolloutParams& p, const int e);
__global__ void __launch_bounds__(128) k_env_reset(const RolloutParams p) {
  const int e = blockIdx.x;
  if (p.done && !p.done[e]) return;
  if (p.term) env_terminal_rows(p, e);
  env_reset_body(p, e);
}
__device__ __forceinline__ void env_reset_body(const RolloutParams& p, const int e) {
  const uint32_t k0 = p.key[2 * e], k1 = p.key[2 * e + 1], ep = p.episode[e];
  for (int j = threadIdx.x; j < p.m; j += blockDim.x) {
    const long obj = (long)e * p.m + j;
    const uint32_t row = ssa_draw_orbit(k0, k1, ep, (uint32_t)j, (uint32_t)p.n_orbits);
    double n6[6];
    ssa_draw_x(k0, k1, ep, (uint32_t)j, n6);
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      const double xt = p.orbits[(long)row * 6 + i];
      p.xt[i * p.ld + obj] = xt;
      p.x[i * p.ld + obj] = xt + ssa_mul(n6[i], p.sig[i]);
    }
#pragma unroll
    for (int q = 0; q < SSA_NP; ++q) p.P[q * p.ld + obj] = p.sig[9 + q];
    p.status[obj] = 0;
    p.infl[obj] = 0;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    p.episode[e] = ep + 1u;
    p.step_idx[e] = 0;
    if (p.rew_hist) {  // a new episode: rewards[0] = 0 (entries 1 .. i-1 are written by its steps before any read) and
      p.rew_hist[(long)e * p.n_steps] = 0.0;  // the argmax of its all-equal sigma_pos[0] (vec_env.py host mode: 0)
      p.spos_prev[e] = 0;
    }
  }
}

// consistency diagnostics of the current step, one thread per object (ssa_ukf_core.h: ssa_nees6 / ssa_nis3)
__global__ void ssa_diag_kernel(const double* __restrict__ xt, const double* __restrict__ x, const double* __restrict__ P,
                                const double* __restrict__ y, const double* __restrict__ S, const uint8_t* __restrict__ updated,
                                double* diag, uint8_t* flags, long ld, int N) {
  const long n = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  double d[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) d[i] = xt[i * ld + n] - x[i * ld + n];
  diag[2 * n] = ssa_nees6(P + n, ld, d);
  double nis = ssa_nan();
  int f = 0;
  if (updated[n]) {  // y / S of this step were recorded (SSA_STEP_RECORD) for the objects that were updated
    double Sm[9], yy[3];
#pragma unroll
    for (int e = 0; e < 9; ++e) Sm[e] = S[n * 9 + e];
#pragma unroll
    for (int a = 0; a < 3; ++a) yy[a] = y[n * 3 + a];
    nis = ssa_nis3(Sm, yy, &f);
    f |= 0x80;
  }
  diag[2 * n + 1] = nis;
  flags[n] = (uint8_t)f;
}

// ---- innovation whiteness statistics (SURVEY 8f-3; SS2:655-698 autocorrelation, SS2:782-832 innovation_dw_test) ---------
// One block per (series, component) of B innovation series y[b][t][3], t < n, with a validity mask (an observation was
// taken / the object was the tasked one).  Durbin-Watson: sum_t (e_t - e_{t-1})^2 / sum_t e_t^2 over the VALID entries in
// order (the reference forms the series of the tasked steps first).  Autocorrelation: statsmodels acf(x, missing=
// 'conservative', fft=False): the series is demeaned by the mean of its valid entries, the invalid entries count as zero,
// acf[k] = sum_t x_t x_{t+k} / sum_t x_t^2 for k = 0..nlags.  All sums run in increasing t (deterministic).
__global__ void __launch_bounds__(64) ssa_innov_stats_kernel(const double* __restrict__ y, const uint8_t* __restrict__ valid, int n, int nlags,
                                                             double* __restrict__ dw, double* __restrict__ acf, double* __restrict__ work) {
  const int b = blockIdx.x / 3, c = blockIdx.x % 3;
  const double* yy = y + (long)b * n * 3 + c;
  const uint8_t* vv = valid + (long)b * n;
  double* xo = work + (long)blockIdx.x * n;   // demeaned series, zeros at the invalid entries
  __shared__ double s_mean, s_acov0;
  if (threadIdx.x == 0) {
    double sum = 0.0, num = 0.0, den = 0.0, prev = 0.0;
    int cnt = 0;
    for (int t = 0; t < n; ++t) {
      if (!vv[t]) continue;
      const double e = yy[3L * t];
      sum += e;
      den = ssa_fma(e, e, den);
      if (cnt) { const double d = e - prev; num = ssa_fma(d, d, num); }
      prev = e;
      ++cnt;
    }
    dw[blockIdx.x] = cnt ? ssa_div(num, den) : ssa_nan();
    s_mean = cnt ? ssa_div(sum, (double)cnt) : 0.0;
  }
  __syncthreads();
  for (int t = threadIdx.x; t < n; t += blockDim.x) xo[t] = vv[t] ? (yy[3L * t] - s_mean) : 0.0;
  __syncthreads();
  for (int k = threadIdx.x; k <= nlags; k += blockDim.x) {
    double acc = 0.0;
    for (int t = 0; t + k < n; ++t) acc = ssa_fma(xo[t], xo[t + k], acc);
    acf[(long)blockIdx.x * (nlags + 1) + k] = acc;
    if (k == 0) s_acov0 = acc;
  }
  __syncthreads();
  for (int k = threadIdx.x; k <= nlags; k += blockDim.x) {
    double* a = acf + (long)blockIdx.x * (nlags + 1) + k;
    *a = ssa_div(*a, s_acov0);
  }
}

// ---- catalog generator (SURVEY 8f-4, envs/orbit_gen.py:47-75): acceptance rule of a batch of candidate orbits ------
// one thread per (candidate, sample time): propagate from the epoch, altitude and elevation at that time
__global__ void __launch_bounds__(128) ssa_orbit_eval_kernel(const double* __restrict__ cand, int K, const double* __restrict__ table,
                                                             int n, double step_s, ssa_obs ob, double obs_limit, double min_alt,
                                                             uint8_t* flags, double* elev, double* alt) {
  const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long)K * n) return;
  const int i = (int)(t / K), c = (int)(t % K);  // candidates fastest: a warp shares the sample time (and its matrix)
  double x0[6], x[6];
#pragma unroll
  for (int q = 0; q < 6; ++q) x0[q] = cand[(long)c * 6 + q];
  const int exc = ssa_fx(x0, ssa_mul(step_s, (double)i), x);
#pragma unroll
  for (int q = 0; q < 9; ++q) ob.M[q] = table[(long)i * 9 + q];
  // orbit_gen.py:57 forms x_gcrs[:3] @ trans_matrix[i] (a row vector times the matrix, i.e. M^T x) for the altitude test
  double xi[3];
#pragma unroll
  for (int j = 0; j < 3; ++j) xi[j] = ssa_fma(x[2], ob.M[6 + j], ssa_fma(x[1], ob.M[3 + j], ssa_mul(x[0], ob.M[j])));
  const double h = ssa_ecef_altitude(xi);
  double z[3];
  ssa_hx_aer(x, &ob, z);
  const long o = (long)c * n + i;
  flags[o] = (uint8_t)((h > min_alt ? 1 : 0) | (z[1] >= obs_limit ? 2 : 0) | (exc ? 4 : 0));
  if (elev) elev[o] = z[1];
  if (alt) alt[o] = h;
}
// one thread per candidate: the visibility-gap rule (orbit_gen.py:60-73)
__global__ void ssa_orbit_accept_kernel(const uint8_t* __restrict__ flags, int K, int n, int first_window, int max_gap, uint8_t* accept) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= K) return;
  int all_alt = 1, all_vis = 1, any_gap = 0, first = 0, run = 0, longest = 0, bad = 0;
  for (int i = 0; i < n; ++i) {
    const int f = flags[(long)c * n + i];
    all_alt &= f & 1;
    const int vis = (f >> 1) & 1;
    bad |= f & 4;
    all_vis &= vis;
    if (i < first_window) first += vis;
    if (!vis) { any_gap = 1; run += 1; longest = run > longest ? run : longest; }
    else run = 0;
  }
  int ok = 0;
  if (all_alt && !bad) ok = any_gap ? (first > 0 && longest < max_gap) : all_vis;
  accept[c] = (uint8_t)ok;
}

// ---- catalog mode (C4): per-shard reward terms over ALL objects of the handle ----------------------------------------
// {max delta_pos, sum of trinary counts (results.py:431-433), number of objects, max trace P, its index (first maximum
// wins, np.argmax)} -> 5 doubles, reduced in two deterministic stages (per-block partials, then one block).
constexpr int kStatBlocks = 296;
struct CatPart { double max_dpos; double max_trace; long arg_trace; long tri; };
__device__ __forceinline__ CatPart cat_merge(CatPart a, CatPart b) {
  CatPart r;
  r.max_dpos = b.max_dpos > a.max_dpos ? b.max_dpos : a.max_dpos;
  const bool takeb = b.arg_trace >= 0 && (a.arg_trace < 0 || b.max_trace > a.max_trace || (b.max_trace == a.max_trace && b.arg_trace < a.arg_trace));
  r.max_trace = takeb ? b.max_trace : a.max_trace;
  r.arg_trace = takeb ? b.arg_trace : a.arg_trace;
  r.tri = a.tri + b.tri;
  return r;
}
__device__ __forceinline__ CatPart cat_block_reduce(CatPart v) {
  __shared__ CatPart sm[8];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    CatPart w;
    w.max_dpos = __shfl_xor_sync(0xffffffffu, v.max_dpos, o);
    w.max_trace = __shfl_xor_sync(0xffffffffu, v.max_trace, o);
    w.arg_trace = __shfl_xor_sync(0xffffffffu, v.arg_trace, o);
    w.tri = __shfl_xor_sync(0xffffffffu, v.tri, o);
    v = cat_merge(v, w);
  }
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x == 0) for (int w = 1; w < (int)(blockDim.x >> 5); ++w) v = cat_merge(v, sm[w]);
  return v;
}
__global__ void __launch_bounds__(256) ssa_cat_stats_stage1(const double* __restrict__ dpos, const double* __restrict__ trace, long N,
                                                            CatPart* part) {
  CatPart v{-1.0, 0.0, -1, 0};
  for (long n = (long)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (long)gridDim.x * blockDim.x) {
    const double d = dpos[n];
    CatPart w{d, trace[n], n, (long)((d < 1e4) + (d < 1e7))};
    v = cat_merge(v, w);
  }
  v = cat_block_reduce(v);
  if (threadIdx.x == 0) part[blockIdx.x] = v;
}
__global__ void __launch_bounds__(256) ssa_cat_stats_stage2(const CatPart* __restrict__ part, int nparts, long N, long index_offset,
                                                            double* out) {
  CatPart v{-1.0, 0.0, -1, 0};
  for (int i = threadIdx.x; i < nparts; i += blockDim.x) v = cat_merge(v, part[i]);
  v = cat_block_reduce(v);
  if (threadIdx.x == 0) {
    out[0] = v.max_dpos; out[1] = (double)v.tri; out[2] = (double)N; out[3] = v.max_trace; out[4] = (double)(v.arg_trace + index_offset);
  }
}

// reward.py:6-50 score terms, one thread per object
__global__ void ssa_scores_kernel(const double* __restrict__ P, const double* __restrict__ dpos, double* out, long ld,
                                  int N, double dt) {
  const long n = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  double a[6][6];
  for (int i = 0; i < 6; ++i)
    for (int j = i; j < 6; ++j) { a[i][j] = P[ssa_pidx(i, j) * ld + n]; a[j][i] = a[i][j]; }
  const double pe = ssa_sqrt((a[0][0] + a[1][1]) + a[2][2]);
  const double ve = ssa_sqrt((a[3][3] + a[4][4]) + a[5][5]);
  out[n * 6 + 0] = ssa_fma(ve, 30.0, pe);  // score_scaled_trace_P
  out[n * 6 + 1] = ((((a[0][0] + a[1][1]) + a[2][2]) + a[3][3]) + a[4][4]) + a[5][5];  // score_trace_P
  // determinants by Gaussian elimination with partial pivoting (np.linalg.det = LU)
  double det3;
  {
    const double m00 = a[0][0], m01 = a[0][1], m02 = a[0][2], m11 = a[1][1], m12 = a[1][2], m22 = a[2][2];
    det3 = m00 * (m11 * m22 - m12 * m12) - m01 * (m01 * m22 - m12 * m02) + m02 * (m01 * m12 - m11 * m02);
  }
  double det = 1.0;
  for (int c = 0; c < 6; ++c) {
    int pv = c;
    for (int i = c + 1; i < 6; ++i) if (fabs(a[i][c]) > fabs(a[pv][c])) pv = i;
    if (pv != c) { for (int j = 0; j < 6; ++j) { const double t = a[c][j]; a[c][j] = a[pv][j]; a[pv][j] = t; } det = -det; }
    det *= a[c][c];
    if (a[c][c] == 0.0) break;
    const double rp = 1.0 / a[c][c];
    for (int i = c + 1; i < 6; ++i) {
      const double l = a[i][c] * rp;
      for (int j = c + 1; j < 6; ++j) a[i][j] -= l * a[c][j];
    }
  }
  const double dt2 = dt * dt, dt6 = dt2 * dt2 * dt2;
  out[n * 6 + 2] = ssa_exp(ssa_div(ssa_log(ssa_mul(det, dt6)), 12.0));  // score_scaled_det_P: (det P dt^6)^(1/12), NaN for det < 0 like np.power
  out[n * 6 + 3] = det;                          // score_det_P
  out[n * 6 + 4] = det3;                         // score_det_pos_P
  out[n * 6 + 5] = dpos[n];                      // |delta pos| (score_neg_max_pos_error = -max over objects)
}

// ---- layout conversion kernels (reference AoS <-> device SoA) ---------------------------------------
__global__ void ssa_aos_to_soa(const double* __restrict__ src, double* __restrict__ dst, int N, int C, long ld) {
  const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long)N * C) return;
  const long n = t / C;
  const int c = (int)(t % C);
  dst[c * ld + n] = src[t];
}
__global__ void ssa_soa_to_aos(const double* __restrict__ src, double* __restrict__ dst, int N, int C, long ld) {
  const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long)N * C) return;
  const long n = t / C;
  const int c = (int)(t % C);
  dst[t] = src[c * ld + n];
}
// full 6x6 AoS [N][36] (or one shared 6x6 when per_object == 0) -> packed SoA (upper triangle)
__global__ void ssa_pfull_to_packed(const double* __restrict__ src, double* __restrict__ dst, int N, long ld,
                                    int per_object) {
  const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long)N * SSA_NP) return;
  const long n = t / SSA_NP;
  const int e = (int)(t % SSA_NP);
  const int i = c_pi[e], j = c_pj[e];
  dst[e * ld + n] = src[(per_object ? n * 36 : 0) + i * 6 + j];
}
__global__ void ssa_packed_to_pfull(const double* __restrict__ src, double* __restrict__ dst, int N, long ld) {
  const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long)N * 36) return;
  const long n = t / 36;
  const int r = (int)(t % 36) / 6, c = (int)(t % 36) % 6;
  const int i = r < c ? r : c, j = r < c ? c : r;
  dst[t] = src[ssa_pidx(i, j) * ld + n];
}
// ssa_ukf_snapshot: every per-step output of the step in the host layout of the reference's history arrays, packed
// into ONE contiguous block (one thread per object):
//   doubles [N][118] = x_true 6 | x_filter 6 | P 36 (full, mirrored) | obs 12 | dpos dvel spos svel | z_true 3 | y 3 |
//                      S 9 | sigmas_h 39          then int32 status [N], uint8 visible [N], uint8 updated [N]
constexpr int kSnapDoubles = 118;
struct SnapParams {
  const double *xt, *x, *P, *obs, *dpos, *dvel, *spos, *svel, *z_true, *y, *S, *sigmas_h;
  const int32_t* status; const uint8_t *visible, *updated;
  long ld; int N;
  double* out;
};
__global__ void ssa_snapshot_kernel(const SnapParams p) {
  const long n = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= p.N) return;
  double* o = p.out + n * kSnapDoubles;
#pragma unroll
  for (int i = 0; i < 6; ++i) { o[i] = p.xt[i * p.ld + n]; o[6 + i] = p.x[i * p.ld + n]; }
#pragma unroll
  for (int r = 0; r < 6; ++r)
#pragma unroll
    for (int c = 0; c < 6; ++c) o[12 + 6 * r + c] = p.P[ssa_pidx(r < c ? r : c, r < c ? c : r) * p.ld + n];
#pragma unroll
  for (int i = 0; i < 12; ++i) o[48 + i] = p.obs[n * 12 + i];
  o[60] = p.dpos[n]; o[61] = p.dvel[n]; o[62] = p.spos[n]; o[63] = p.svel[n];
#pragma unroll
  for (int i = 0; i < 3; ++i) { o[64 + i] = p.z_true[n * 3 + i]; o[67 + i] = p.y[n * 3 + i]; }
#pragma unroll
  for (int i = 0; i < 9; ++i) o[70 + i] = p.S[n * 9 + i];
  for (int i = 0; i < 39; ++i) o[79 + i] = p.sigmas_h[n * 39 + i];
  int32_t* st = (int32_t*)(p.out + (long)p.N * kSnapDoubles);
  st[n] = p.status[n];
  uint8_t* u8 = (uint8_t*)(st + p.N);
  u8[n] = p.visible[n];
  u8[p.N + n] = p.updated[n];
}

// FP64 pipe microbenchmark: 8 independent DFMA chains per thread.
__global__ void __launch_bounds__(256) ssa_dfma_peak_kernel(double* out, int iters, double a, double b) {
  double v0 = threadIdx.x, v1 = v0 + 1, v2 = v0 + 2, v3 = v0 + 3, v4 = v0 + 4, v5 = v0 + 5, v6 = v0 + 6, v7 = v0 + 7;
  for (int i = 0; i < iters; ++i) {
    v0 = __fma_rn(v0, a, b); v1 = __fma_rn(v1, a, b); v2 = __fma_rn(v2, a, b); v3 = __fma_rn(v3, a, b);
    v4 = __fma_rn(v4, a, b); v5 = __fma_rn(v5, a, b); v6 = __fma_rn(v6, a, b); v7 = __fma_rn(v7, a, b);
  }
  const double s = ((v0 + v1) + (v2 + v3)) + ((v4 + v5) + (v6 + v7));
  if (s == 12345.678) out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}


// ---- unit kernels: the device build of single functions, one thread per element.  They exist so that
// the tests can demand bit-equality between sm_100a and the host twin function by function, and so
// that the Python operator callables (fx, hx, ...) evaluate on the device when called directly. ----
__global__ void ssa_unit_math_kernel(int op, const double* a, const double* b, double* out, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double x = a[i], y = b ? b[i] : 0.0;
  double r;
  switch (op) {
    case 0: r = ssa_sin(x); break;      case 1: r = ssa_cos(x); break;     case 2: r = ssa_tan(x); break;
    case 3: r = ssa_atan(x); break;     case 4: r = ssa_asin(x); break;    case 5: r = ssa_acos(x); break;
    case 6: r = ssa_exp(x); break;      case 7: r = ssa_log(x); break;     case 8: r = ssa_sinh(x); break;
    case 9: r = ssa_cosh(x); break;     case 10: r = ssa_tanh(x); break;   case 11: r = ssa_atanh(x); break;
    case 12: r = ssa_asinh(x); break;   case 13: r = ssa_acosh(x); break;  case 14: r = ssa_pow23(x); break;
    case 15: r = ssa_atan2(x, y); break; case 16: r = ssa_pymod(x, y); break;
    case 17: r = ssa_div(x, y); break;  case 18: r = ssa_sqrt(x); break;
    default: r = ssa_nan();
  }
  out[i] = r;
}
__global__ void ssa_unit_fx_kernel(const double* x, double dt, double* out, int32_t* exc, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double s[6], f[6];
  for (int k = 0; k < 6; ++k) s[k] = x[6 * (long)i + k];
  exc[i] = ssa_fx(s, dt, f);
  for (int k = 0; k < 6; ++k) out[6 * (long)i + k] = f[k];
}
__global__ void ssa_unit_hx_kernel(const double* x, ssa_obs ob, double* out, int n, int stride) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double s[3], z[3];
  for (int k = 0; k < 3; ++k) s[k] = x[stride * (long)i + k];
  ssa_hx_aer(s, &ob, z);
  for (int k = 0; k < 3; ++k) out[3 * (long)i + k] = z[k];
}
__global__ void ssa_unit_aer_kernel(int op, const double* a, const double* b, double* out, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double u[3], v[3] = {0, 0, 0}, r[3];
  for (int k = 0; k < 3; ++k) { u[k] = a[3 * (long)i + k]; if (b) v[k] = b[3 * (long)i + k]; }
  if (op == 0) ssa_aer2uvw(u, r);
  else if (op == 1) ssa_uvw2aer(u, r);
  else ssa_residual_aer(u, v, r);
  for (int k = 0; k < 3; ++k) out[3 * (long)i + k] = r[k];
}
__global__ void ssa_unit_chol_kernel(const double* P, double lam, double* U, int32_t* ret, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double u[SSA_NP];
  ret[i] = ssa_robust_chol6(P + (long)i * SSA_NP, 1, lam, u);
  for (int e = 0; e < SSA_NP; ++e) U[(long)i * SSA_NP + e] = u[e];
}
__global__ void ssa_unit_inv3_kernel(const double* S, double* SI, int32_t* ok, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double s[9], si[9];
  for (int e = 0; e < 9; ++e) s[e] = S[(long)i * 9 + e];
  ok[i] = ssa_inv3(s, si);
  for (int e = 0; e < 9; ++e) SI[(long)i * 9 + e] = si[e];
}

thread_local char g_err[512] = "";
// 2-D tensor map over a row-major [rows][ld] fp64 array with a box of 32 columns x box_rows rows (no swizzle: a
// thread reads only its own column of the tile).  cuTensorMapEncodeTiled is resolved through the runtime so that
// the library does not link against libcuda.
int make_tmap(CUtensorMap* tm, const double* base, long ld, int rows, int box_rows) {
  static PFN_cuTensorMapEncodeTiled_v12000 enc = nullptr;
  if (!enc) {
    cudaDriverEntryPointQueryResult q;
    void* fn = nullptr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess || !fn) return 1;
    enc = (PFN_cuTensorMapEncodeTiled_v12000)fn;
  }
  const cuuint64_t gdim[2] = {(cuuint64_t)ld, (cuuint64_t)rows};
  const cuuint64_t gstride[1] = {(cuuint64_t)ld * sizeof(double)};
  const cuuint32_t box[2] = {32u, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1u, 1u};
  const CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, (void*)base, gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : 1;
}

// launch with the programmatic-stream-serialization attribute (see pdl_prologue)
template <typename... KArgs, typename... Args>
void launch_chain(bool pdl, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = pdl ? 1 : 0;
  cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}

int set_err(const char* what, cudaError_t e) {
  snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
  return SSA_ECUDA;
}
#define CK(call)                                         \
  do {                                                   \
    cudaError_t e_ = (call);                             \
    if (e_ != cudaSuccess) return set_err(#call, e_);    \
  } while (0)

}  // namespace

// ---------------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------------
// The output block of the episodic mode (include/ssa_ukf.h), on the device and as its pinned host mirror:
// [obs 12N doubles][reward E doubles][greedy 6E int32][done E bytes, padded to 8][truncated E bytes, padded to 8]
struct RolloutBlock {
  double* obs; double* reward; int32_t* greedy; uint8_t* done; uint8_t* truncated;
  size_t bytes;  // of the whole block
  size_t tail;   // byte offset of reward .. truncated (what follows the observation rows)
};

// the views of the block at base (null: only its sizes)
static RolloutBlock rollout_block(void* base, size_t N, size_t E) {
  RolloutBlock b = {};
  const size_t flags = (E + 7) / 8 * 8;
  b.tail = sizeof(double) * 12 * N;
  b.bytes = sizeof(double) * (12 * N + E) + sizeof(int32_t) * SSA_N_TASKERS * E + 2 * flags;
  if (!base) return b;
  b.obs = (double*)base;
  b.reward = b.obs + 12 * N;
  b.greedy = (int32_t*)(b.reward + E);
  b.done = (uint8_t*)(b.greedy + SSA_N_TASKERS * E);
  b.truncated = b.done + flags;
  return b;
}

// A parity's block of the double-buffered host pipeline (ssa_ukf_step_host, ssa_ukf_step_pinned), in doubles:
//   OUT  [obs 12N][dpos ld][status ld int32]        <- one D2H copy in the pinned mode; pinned mirror hout
//        [dvel ld][spos ld][svel ld][trace ld]      (device only; in hout: the step's reward terms, SSA_F_CATALOG_STATS)
//   IN   [z_noise 3N][M 9][pad 1][actions E int32]  <- one H2D copy in the pinned mode; pinned mirror hin
struct PipeBlock {
  double* obs; double* dpos; int32_t* status; double* dvel; double* spos; double* svel; double* trace;
  double* stats;  // (hout only)
  double* z_noise; double* M; int32_t* actions;
  size_t out, in, dev, hout;  // doubles: the two copies (OUT up to the status words, IN), the device block, hout
};

// the views of the device block dev, or (dev null) of the pinned mirrors hout and hin; all null: only the sizes
static PipeBlock pipe_block(double* dev, double* hout, double* hin, size_t N, size_t E, size_t ld) {
  PipeBlock b = {};
  b.out = 12 * N + ld + ld / 2;
  b.in = 3 * N + 10 + (E + 1) / 2;
  b.dev = b.out + 4 * ld + b.in;
  b.hout = b.out + 8;
  double* out = dev ? dev : hout;
  double* in = dev ? dev + b.out + 4 * ld : hin;
  if (out) { b.obs = out; b.dpos = out + 12 * N; b.status = (int32_t*)(b.dpos + ld); }
  if (dev) { b.dvel = b.dpos + ld + ld / 2; b.spos = b.dvel + ld; b.svel = b.spos + ld; b.trace = b.svel + ld; }
  if (hout) b.stats = hout + b.out;
  if (in) { b.z_noise = in; b.M = in + 3 * N; b.actions = (int32_t*)(b.M + 10); }
  return b;
}

// SSA_UKF_KERNEL, the catalog step's kernels (unset or unknown: tile): tile, the tile kernels; tile2, the two
// factorisations inside the tile kernels instead of k_factor / k_refactor; fused, one launch per full catalog step
// (k_step_tile) instead of the four tile kernels; split, the five-kernel split pipeline; team, the 16-lane team kernel
enum class StepKernel { tile, tile2, fused, split, team };

struct ssa_ukf {
  ssa_ukf_cfg cfg;
  int device;
  long ld;
  long launches;
  // one slab for all fp64 SoA state
  double* slab;
  double *xt, *x, *P, *dpos, *dvel, *spos, *svel, *trace, *det_prev, *det_last, *det_cur;
  double *obs, *z_noise, *z_true, *y, *S, *sigmas_h, *scores, *reward, *env_stats;
  double* stage;  // staging for AoS<->SoA conversion ([N][39] doubles)
  double* qr;     // packed Q (21) + R (9)
  double* scratch;  // U[21] F[78] ZS[39] UVW[39] ZT[3] rows of ld doubles
  double* Menv;     // [E][9]
  int32_t* step_idx;  // [E]
  int32_t* det_step;  // [E] (EnvParams::det_step)
  int32_t *code, *exc;
  long chunk;     // objects per chunk of the split pipeline (scratch capacity); N when everything fits in L2
  long staged_max;  // chunks up to this many objects use the TMA-staged k_update (default: all)
  CUtensorMap tm_z, tm_u, tm_s, tm_x;
  int pdl;  // programmatic dependent launch of the step's kernel chain (SSA_UKF_PDL=0 turns it off)
  StepKernel kernel;  // SSA_UKF_KERNEL
  bool act_split;   // SSA_UKF_ACT=split: the RL-mode update of the tasked objects runs as k_hx + k_update instead of k_update_tile
  int use_graph;    // ssa_ukf_step_pinned / ssa_ukf_rollout_step as captured graphs (SSA_UKF_GRAPH=0: plain launches)
  int det_kernel;   // SSA_UKF_DET_KERNEL set: ssa_det_kernel also for m <= 64, not the determinants inside the reduction
  int refresh_chain;  // SSA_UKF_REFRESH_CHAIN set: an auto-reset step re-draws with k_env_reset + the refresh chain
  int sm_count;
  // double-buffered host pipeline (ssa_ukf_step_host)
  struct {
    int init, parity;
    long calls;
    cudaStream_t up, dn;
    cudaEvent_t e_up[2], e_c[2], e_dn[2];
    PipeBlock dev[2], host[2];  // per parity: the device block and its pinned host mirrors (pipe_block, ssa_ukf_host_io)
    cudaGraphExec_t gexec[2];  // the step's kernel chain captured per parity (ssa_ukf_step_pinned)
    int gflags[2], gkernels[2];
  } hp;
  // ssa_ukf_step as one graph launch (SSA_UKF_STEP_GRAPH=0: five plain launches).  The only launch parameter that
  // changes from step to step is the trans_matrix, which only k_hx reads: its kernel node is re-parameterised
  // before every launch (cudaGraphExecKernelNodeSetParams), the other four nodes stay as captured.
  struct {
    int on, n;
    int flags[4];
    cudaGraph_t graph[4];  // kept alive: the node handles used for the parameter update belong to it
    cudaGraphExec_t gexec[4];
    int gkernels[4];
    cudaGraphNode_t hx_node[4];
    cudaKernelNodeParams hx_params[4];
  } sg;
  // device-resident episodic mode (ssa_ukf_rollout_*)
  struct {
    int init, n_orbits, n_table, update_interval;
    double* dbuf;        // device: orbits [n_orbits][6], table [n_table][9], sig [30]
    double *orbits, *table, *sig;
    uint32_t* ibuf;      // device: key [E][2], episode [E], act_in [E], act_eff [E]
    uint32_t *key, *episode;
    int32_t *act_in, *act_eff;
    RolloutBlock dev, host;  // the output block and its pinned host mirror
    int32_t* hin;        // pinned host actions [E]
    float *dobs32, *hobs32;    // SSA_ROLLOUT_OBS_F32: obs [N][12] as floats (device block, pinned host mirror)
    double *daer, *haer;       // SSA_ROLLOUT_OBS_AER: the 'aer' observation [N][4] (device block, pinned host mirror)
    double* rew_hist;          // 'shaped' only: [E][n_steps] reward history, then spos_prev [E] int32
    int32_t* spos_prev;
    int tasker;                // ssa_ukf_rollout_tasker
    double spoil_p;
    // final observations (ssa_ukf_rollout_terminal_obs_download), ssa_ukf_rollout_reset_envs, and the rows of every
    // gathered download (gather_download: final observations, episode records, normalized final observations)
    double* tbuf;              // device: terminal [12N], gathered rows [max(12N, SSA_EPR E)], then idx [E] int32, mask [E] uint8
    double *term, *gath;
    int32_t* gidx;
    uint8_t* mask;
    double* hgath;             // pinned: gathered rows [max(12N, SSA_EPR E)], then idx [E] int32
    int32_t* hgidx;
    int term_w;                // doubles per object of the terminal rows: 12, 4 after an SSA_ROLLOUT_OBS_AER auto-reset step
    cudaGraphExec_t gexec[6];  // [auto_reset + 2 * (obs_f32 ? 1 : obs_aer ? 2 : 0)]
    int gkernels[6];
  } ro;
  // per-episode statistics of the episodic mode (ssa_ukf_rollout_episode_stats_*)
  struct {
    int on;              // buffers allocated (ssa_ukf_rollout_episode_stats_enable)
    int live;            // accumulating: the step graphs carry k_ep_row0 / k_ep_step (from the next rollout_reset on)
    double* buf;         // device: obj [N][SSA_EPO], env [E][SSA_EPE], rec [E][SSA_EPR]
    double *obj, *env, *rec;
  } es;
  // running normalization of observations and returns in the episodic mode (ssa_ukf_rollout_normalize, k_normalize)
  struct {
    int on;
    int F;               // normalized columns per environment: 12 m, or 4 m for SSA_NORM_OBS_AER
    ssa_norm_cfg cfg;
    double* buf;         // device: state [4 + E + 3F] (SSA_F_ROLLOUT_NORM_STATE), reward_norm [E], then floats obs_norm,
                         // term_norm [E][F] each
    double *state, *reward;
    float *obs, *term;
    double* hbuf;        // pinned: reward_norm [E], obs_norm [E][F] floats (the step copies both at once)
    float* hobs;
  } nm;
  int32_t *status, *infl, *actions, *greedy;
  uint8_t *visible, *updated, *innov_flags, *done;
  double* diag;     // [N][2] NEES, NIS of the last ssa_ukf_diagnostics call
  void* snap;       // device block of ssa_ukf_snapshot (allocated on first use)
  void* cat_part; double* cat_stats;  // ssa_ukf_catalog_stats: per-block partials, result [5]
  long cat_index_offset;
  const double *last_dpos, *last_trace;  // where the most recent step left delta_pos / trace (the handle's arrays, or a
                                         // block of the double-buffered host pipeline)
  size_t stage_bytes;
};

// Captures the kernels that enqueue(stream) launches into *exec: a non-blocking stream in thread-local capture mode,
// instantiated without flags.  *kernels: the launches it made (the handle's counter is left as it was; every launch of
// the graph adds them).  keep: receives the captured graph, which the caller then owns; null: destroyed here.
template <typename Enqueue>
static int capture_chain(ssa_ukf* h, Enqueue&& enqueue, cudaGraph_t* keep, cudaGraphExec_t* exec, int* kernels) {
  cudaStream_t cs;
  CK(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
  const long l0 = h->launches;
  CK(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
  const int rc = enqueue(cs);
  cudaGraph_t g = nullptr;
  const cudaError_t ce = cudaStreamEndCapture(cs, &g);
  *kernels = (int)(h->launches - l0);
  h->launches = l0;
  cudaStreamDestroy(cs);
  if (rc) { if (g) cudaGraphDestroy(g); return rc; }
  if (ce != cudaSuccess) return set_err("cudaStreamEndCapture", ce);
  const cudaError_t ie = cudaGraphInstantiate(exec, g, 0);
  if (ie == cudaSuccess && keep) { *keep = g; return SSA_OK; }
  cudaGraphDestroy(g);
  return ie == cudaSuccess ? SSA_OK : set_err("cudaGraphInstantiate", ie);
}

// the team kernel's rule: never captured into a graph; an auto-reset step re-draws with k_env_reset + the refresh chain
static bool team_kernel(const ssa_ukf* h) { return h->kernel == StepKernel::team; }

// the guard of the ssa_ukf_rollout_* entry points that need ssa_ukf_rollout_config
static bool rollout_ready(const ssa_ukf* h) {
  if (h && h->ro.init) return true;
  snprintf(g_err, sizeof(g_err), "episodic mode not configured");
  return false;
}

// the captured step graphs of the episodic mode (re-captured on the next ssa_ukf_rollout_step)
static void rollout_drop_graphs(ssa_ukf* h) {
  for (int i = 0; i < 6; ++i) if (h->ro.gexec[i]) { cudaGraphExecDestroy(h->ro.gexec[i]); h->ro.gexec[i] = nullptr; }
}

// The only code that frees the buffers of the episodic mode, of its episode statistics and of its normalization; each
// leaves its part of the handle zeroed (not configured / not enabled).
static void rollout_free(ssa_ukf* h) {
  cudaFree(h->ro.dbuf); cudaFree(h->ro.ibuf); cudaFree(h->ro.dev.obs); cudaFree(h->ro.dobs32);
  cudaFree(h->ro.daer); cudaFree(h->ro.rew_hist); cudaFree(h->ro.tbuf);
  cudaFreeHost(h->ro.host.obs); cudaFreeHost(h->ro.hin); cudaFreeHost(h->ro.hobs32); cudaFreeHost(h->ro.haer);
  cudaFreeHost(h->ro.hgath);
  rollout_drop_graphs(h);
  memset(&h->ro, 0, sizeof(h->ro));
}

static void episode_stats_free(ssa_ukf* h) {
  cudaFree(h->es.buf);
  memset(&h->es, 0, sizeof(h->es));
}

static void norm_free(ssa_ukf* h) {
  cudaFree(h->nm.buf); cudaFreeHost(h->nm.hbuf);
  memset(&h->nm, 0, sizeof(h->nm));
}

extern "C" {

int ssa_ukf_abi_version(void) { return SSA_UKF_ABI_VERSION; }
const char* ssa_ukf_last_error(void) { return g_err; }
int ssa_ukf_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}
long ssa_ukf_ld(const ssa_ukf* h) { return h ? h->ld : 0; }
long ssa_ukf_launch_count(const ssa_ukf* h) { return h ? h->launches : 0; }

int ssa_ukf_create(const ssa_ukf_cfg* cfg, int device, ssa_ukf** out) {
  if (!cfg || !out) { snprintf(g_err, sizeof(g_err), "null argument"); return SSA_EINVAL; }
  if (cfg->abi_version != SSA_UKF_ABI_VERSION) { snprintf(g_err, sizeof(g_err), "ABI version mismatch"); return SSA_EINVAL; }
  if (cfg->n_objects <= 0 || cfg->m <= 0 || cfg->n_envs <= 0 || (long)cfg->n_envs * cfg->m != cfg->n_objects) {
    snprintf(g_err, sizeof(g_err), "need n_objects == n_envs * m > 0");
    return SSA_EINVAL;
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    snprintf(g_err, sizeof(g_err), "no CUDA device: libssa_ukf has no CPU fallback");
    return SSA_ENODEV;
  }
  if (device < 0 || device >= ndev) { snprintf(g_err, sizeof(g_err), "bad device index"); return SSA_EINVAL; }
  CK(cudaSetDevice(device));
  ssa_ukf* h = new (std::nothrow) ssa_ukf();
  if (!h) return SSA_ENOMEM;
  memset(h, 0, sizeof(*h));
  h->cfg = *cfg;
  h->device = device;
  const long N = cfg->n_objects, E = cfg->n_envs;
  h->ld = (N + 31) / 32 * 32;
  const long ld = h->ld;
  // fp64 slab: xt 6, x 6, P 21, dpos dvel spos svel trace 5 (SoA rows of ld) + AoS outputs
  const size_t n_soa = (size_t)(6 + 6 + 21 + 5 + 3) * ld;
  const size_t n_aos = (size_t)N * (12 + 3 + 3 + 3 + 9 + 39 + 6 + 2) + (size_t)E * (1 + 4 + 9) + 32;
  cudaError_t e = cudaMalloc(&h->slab, (n_soa + n_aos) * sizeof(double));
  if (e != cudaSuccess) { delete h; return set_err("cudaMalloc(slab)", e); }
  cudaMemset(h->slab, 0, (n_soa + n_aos) * sizeof(double));
  double* q = h->slab;
  h->xt = q; q += 6 * ld;
  h->x = q; q += 6 * ld;
  h->P = q; q += 21 * ld;
  h->dpos = q; q += ld; h->dvel = q; q += ld; h->spos = q; q += ld; h->svel = q; q += ld; h->trace = q; q += ld;
  h->det_prev = q; q += ld;
  h->det_last = q; q += ld;
  h->det_cur = q; q += ld;
  h->obs = q; q += N * 12;
  h->z_noise = q; q += N * 3;
  h->z_true = q; q += N * 3;
  h->y = q; q += N * 3;
  h->S = q; q += N * 9;
  h->sigmas_h = q; q += N * 39;
  h->scores = q; q += N * 6;
  h->diag = q; q += N * 2;
  h->reward = q; q += E;
  h->env_stats = q; q += E * 4;
  h->qr = q; q += 32;
  h->Menv = q; q += E * 9;
  {
    double qr[30];
    int e2 = 0;
    for (int i = 0; i < 6; ++i) for (int j = i; j < 6; ++j) qr[e2++] = cfg->Q[6 * i + j];
    for (int k = 0; k < 9; ++k) qr[21 + k] = cfg->R[k];
    e = cudaMemcpy(h->qr, qr, sizeof(qr), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { cudaFree(h->slab); delete h; return set_err("cudaMemcpy(qr)", e); }
  }
  h->stage_bytes = (size_t)N * 39 * sizeof(double);
  if ((e = cudaMalloc(&h->stage, h->stage_bytes)) != cudaSuccess) { ssa_ukf_destroy(h); return set_err("cudaMalloc(stage)", e); }
  if ((e = cudaMalloc(&h->status, sizeof(int32_t) * (4 * ld + 3 * E + E * SSA_N_TASKERS))) != cudaSuccess) {
    ssa_ukf_destroy(h);
    return set_err("cudaMalloc(int)", e);
  }
  cudaMemset(h->status, 0, sizeof(int32_t) * (4 * ld + 3 * E + E * SSA_N_TASKERS));
  h->infl = h->status + ld;
  h->code = h->infl + ld;
  h->exc = h->code + ld;
  h->actions = h->exc + ld;
  h->greedy = h->actions + E;
  h->step_idx = h->greedy + E * SSA_N_TASKERS;
  h->det_step = h->step_idx + E;
  cudaMemset(h->det_step, 0xFF, sizeof(int32_t) * E);  // -1: no determinant history yet
  // Scratch of the split pipeline is sized for one CHUNK of objects (180 doubles = 1.44 KB per object); batches
  // larger than the chunk run chunk by chunk.  Measured on B200 with 1 M objects: L2-sized chunks (24 k..196 k
  // objects) are SLOWER than one pass (2.4-4.0 ms vs 2.16 ms per step) — the per-launch tails cost more than the
  // HBM round trip of the sigma sets saves — so the default chunk (4 Mi objects, 6 GB of scratch) only bounds
  // memory for very large catalogs.  The book-version filter (resample off) keeps sigmas_f across calls and is
  // not chunked.
  {
    long chunk = 4L << 20;
    const char* cv = getenv("SSA_UKF_CHUNK");
    if (cv && atol(cv) > 0) chunk = atol(cv);
    if (!cfg->resample_after_predict || chunk >= N) chunk = N;
    if (chunk < N) chunk = chunk < 32 ? 32 : chunk / 32 * 32;
    h->chunk = chunk;
  }
  const long lds = (h->chunk + 31) / 32 * 32;
  if ((e = cudaMalloc(&h->scratch, sizeof(double) * (size_t)(21 + 78 + 39 + 39 + 3) * lds)) != cudaSuccess) {
    ssa_ukf_destroy(h);
    return set_err("cudaMalloc(scratch)", e);
  }
  cudaMemset(h->scratch, 0, sizeof(double) * (size_t)(21 + 78 + 39 + 39 + 3) * lds);
  {
    const char *kv = getenv("SSA_UKF_KERNEL"), *av = getenv("SSA_UKF_ACT");
    const auto is = [](const char* v, const char* s) { return v && strcmp(v, s) == 0; };
    h->kernel = is(kv, "team") ? StepKernel::team : is(kv, "split") ? StepKernel::split : is(kv, "fused") ? StepKernel::fused
              : is(kv, "tile2") ? StepKernel::tile2 : StepKernel::tile;
    h->act_split = is(av, "split");
    h->sm_count = 148;
    cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, h->device);
    cudaFuncSetAttribute(k_update_tile<SSA_TILE, kTileThreads, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(UpdateTile<SSA_TILE>));
    cudaFuncSetAttribute(k_update_tile<SSA_TILE, kTileThreads, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(UpdateTile<SSA_TILE>));
    cudaFuncSetAttribute(k_step_tile<SSA_TILE, kTileThreads>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(UpdateTile<SSA_TILE>));
    const char* gv = getenv("SSA_UKF_STEP_GRAPH");
    h->sg.on = (gv && strcmp(gv, "0") == 0) ? 0 : 1;
    const char* cg = getenv("SSA_UKF_GRAPH");
    h->use_graph = (cg && strcmp(cg, "0") == 0) ? 0 : 1;
    h->det_kernel = getenv("SSA_UKF_DET_KERNEL") ? 1 : 0;
    h->refresh_chain = getenv("SSA_UKF_REFRESH_CHAIN") ? 1 : 0;
    const char* pv = getenv("SSA_UKF_PDL");
    h->pdl = (pv && strcmp(pv, "0") == 0) ? 0 : 1;
    h->staged_max = kStagedMaxDefault;
    const char* sv = getenv("SSA_UKF_STAGED_MAX");
    if (sv) h->staged_max = atol(sv);
    cudaFuncSetAttribute(k_update_staged, cudaFuncAttributeMaxDynamicSharedMemorySize, kUpdStagedSmem);
    // tensor maps of the two SoA tensors (scratch [180][lds], state [33][ld]); one map per box height
    const int rc = make_tmap(&h->tm_z, h->scratch, lds, SC_ROWS, 81) |
                   make_tmap(&h->tm_u, h->scratch, lds, SC_ROWS, 21) | make_tmap(&h->tm_s, h->xt, ld, ST_ROWS, ST_ROWS) |
                   make_tmap(&h->tm_x, h->xt, ld, ST_ROWS, 12);
    if (rc) { ssa_ukf_destroy(h); return set_err("cuTensorMapEncodeTiled", cudaErrorUnknown); }
  }
  if ((e = cudaMalloc(&h->visible, 3 * ld + E)) != cudaSuccess) { ssa_ukf_destroy(h); return set_err("cudaMalloc(u8)", e); }
  cudaMemset(h->visible, 0, 3 * ld + E);
  h->updated = h->visible + ld;
  h->innov_flags = h->updated + ld;
  h->done = h->innov_flags + ld;
  *out = h;
  return SSA_OK;
}

int ssa_ukf_destroy(ssa_ukf* h) {
  if (!h) return SSA_OK;
  cudaSetDevice(h->device);
  cudaFree(h->slab);
  if (h->hp.init) {
    cudaStreamSynchronize(h->hp.up); cudaStreamSynchronize(h->hp.dn);
    for (int b = 0; b < 2; ++b) {
      cudaFree(h->hp.dev[b].obs); cudaFreeHost(h->hp.host[b].z_noise); cudaFreeHost(h->hp.host[b].obs);
      if (h->hp.gexec[b]) cudaGraphExecDestroy(h->hp.gexec[b]);
      cudaEventDestroy(h->hp.e_up[b]); cudaEventDestroy(h->hp.e_c[b]); cudaEventDestroy(h->hp.e_dn[b]);
    }
    cudaStreamDestroy(h->hp.up); cudaStreamDestroy(h->hp.dn);
  }
  for (int i = 0; i < h->sg.n; ++i) { cudaGraphExecDestroy(h->sg.gexec[i]); cudaGraphDestroy(h->sg.graph[i]); }
  rollout_free(h);
  episode_stats_free(h);
  norm_free(h);
  cudaFree(h->snap);
  cudaFree(h->cat_part);
  cudaFree(h->stage);
  cudaFree(h->scratch);
  cudaFree(h->status);
  cudaFree(h->visible);
  delete h;
  return SSA_OK;
}

static int upload_soa(ssa_ukf* h, const double* host, double* dst, int C, cudaStream_t st) {
  const long N = h->cfg.n_objects;
  CK(cudaMemcpyAsync(h->stage, host, sizeof(double) * N * C, cudaMemcpyHostToDevice, st));
  const long tot = N * C;
  ssa_aos_to_soa<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(h->stage, dst, (int)N, C, h->ld);
  h->launches++;
  CK(cudaGetLastError());
  return SSA_OK;
}

int ssa_ukf_reset(ssa_ukf* h, const double* x_true, const double* x_filter, const double* P0, int p0_per_object,
                  void* stream) {
  if (!h || !x_true || !x_filter || !P0) { snprintf(g_err, sizeof(g_err), "null argument"); return SSA_EINVAL; }
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(h->device));
  const long N = h->cfg.n_objects;
  int rc;
  if ((rc = upload_soa(h, x_true, h->xt, 6, st))) return rc;
  CK(cudaStreamSynchronize(st));  // the staging buffer is reused
  if ((rc = upload_soa(h, x_filter, h->x, 6, st))) return rc;
  CK(cudaStreamSynchronize(st));
  if (p0_per_object) {
    // chunk through the staging buffer ([N][39] doubles >= [N][36])
    CK(cudaMemcpyAsync(h->stage, P0, sizeof(double) * N * 36, cudaMemcpyHostToDevice, st));
  } else {
    CK(cudaMemcpyAsync(h->stage, P0, sizeof(double) * 36, cudaMemcpyHostToDevice, st));
  }
  ssa_pfull_to_packed<<<(unsigned)((N * SSA_NP + 255) / 256), 256, 0, st>>>(h->stage, h->P, (int)N, h->ld, p0_per_object);
  h->launches++;
  CK(cudaGetLastError());
  CK(cudaMemsetAsync(h->status, 0, sizeof(int32_t) * 2 * h->ld, st));
  CK(cudaMemsetAsync(h->visible, 0, 2 * h->ld, st));
  CK(cudaMemsetAsync(h->det_step, 0xFF, sizeof(int32_t) * h->cfg.n_envs, st));  // -1: no previous covariance yet (agent_shannon)
  CK(cudaStreamSynchronize(st));
  return SSA_OK;
}

static int field_info(ssa_ukf* h, int field, void** p, size_t* bytes, int* soa_cols) {
  const size_t N = h->cfg.n_objects, E = h->cfg.n_envs, ld = h->ld;
  *soa_cols = 0;
  switch (field) {
    case SSA_F_X_TRUE: *p = h->xt; *bytes = 6 * ld * 8; *soa_cols = 6; break;
    case SSA_F_X_FILTER: *p = h->x; *bytes = 6 * ld * 8; *soa_cols = 6; break;
    case SSA_F_P_FILTER: *p = h->P; *bytes = 21 * ld * 8; *soa_cols = 21; break;
    case SSA_F_OBS: *p = h->obs; *bytes = N * 12 * 8; break;
    case SSA_F_DELTA_POS: *p = h->dpos; *bytes = N * 8; break;
    case SSA_F_DELTA_VEL: *p = h->dvel; *bytes = N * 8; break;
    case SSA_F_SIGMA_POS: *p = h->spos; *bytes = N * 8; break;
    case SSA_F_SIGMA_VEL: *p = h->svel; *bytes = N * 8; break;
    case SSA_F_TRACE: *p = h->trace; *bytes = N * 8; break;
    case SSA_F_Z_TRUE: *p = h->z_true; *bytes = N * 3 * 8; break;
    case SSA_F_Y: *p = h->y; *bytes = N * 3 * 8; break;
    case SSA_F_S: *p = h->S; *bytes = N * 9 * 8; break;
    case SSA_F_SIGMAS_H: *p = h->sigmas_h; *bytes = N * 39 * 8; break;
    case SSA_F_Z_NOISE: *p = h->z_noise; *bytes = N * 3 * 8; break;
    case SSA_F_VISIBLE: *p = h->visible; *bytes = N; break;
    case SSA_F_UPDATED: *p = h->updated; *bytes = N; break;
    case SSA_F_STATUS: *p = h->status; *bytes = N * 4; break;
    case SSA_F_INFLATIONS: *p = h->infl; *bytes = N * 4; break;
    case SSA_F_ACTIONS: *p = h->actions; *bytes = E * 4; break;
    case SSA_F_REWARD: *p = h->reward; *bytes = E * 8; break;
    case SSA_F_DONE: *p = h->done; *bytes = E; break;
    case SSA_F_GREEDY: *p = h->greedy; *bytes = E * SSA_N_TASKERS * 4; break;
    case SSA_F_SCORES: *p = h->scores; *bytes = N * 6 * 8; break;
    case SSA_F_TRANS_ENV: *p = h->Menv; *bytes = E * 9 * 8; break;
    case SSA_F_STEP_INDEX: *p = h->step_idx; *bytes = E * 4; break;
    case SSA_F_ENV_STATS: *p = h->env_stats; *bytes = E * 4 * 8; break;
    case SSA_F_DIAG: *p = h->diag; *bytes = N * 2 * 8; break;
    case SSA_F_CATALOG_STATS:
      if (!h->cat_stats) { snprintf(g_err, sizeof(g_err), "call ssa_ukf_catalog_stats first"); return SSA_EINVAL; }
      *p = h->cat_stats; *bytes = 5 * 8; break;
    case SSA_F_INNOV_FLAGS: *p = h->innov_flags; *bytes = N; break;
    case SSA_F_ROLLOUT_OBS: case SSA_F_ROLLOUT_REWARD: case SSA_F_ROLLOUT_ACTIONS: case SSA_F_ROLLOUT_GREEDY:
    case SSA_F_ROLLOUT_DONE: case SSA_F_ROLLOUT_OBS_AER: case SSA_F_ROLLOUT_TERMINAL_OBS: case SSA_F_ROLLOUT_TRUNCATED: {
      if (!rollout_ready(h)) return SSA_EINVAL;
      const RolloutBlock& b = h->ro.dev;
      switch (field) {
        case SSA_F_ROLLOUT_OBS: *p = b.obs; *bytes = N * 12 * 8; break;
        case SSA_F_ROLLOUT_REWARD: *p = b.reward; *bytes = E * 8; break;
        case SSA_F_ROLLOUT_ACTIONS: *p = h->ro.act_in; *bytes = E * 4; break;
        case SSA_F_ROLLOUT_GREEDY: *p = b.greedy; *bytes = E * SSA_N_TASKERS * 4; break;
        case SSA_F_ROLLOUT_DONE: *p = b.done; *bytes = E; break;
        case SSA_F_ROLLOUT_OBS_AER: *p = h->ro.daer; *bytes = N * 4 * 8; break;
        case SSA_F_ROLLOUT_TERMINAL_OBS: *p = h->ro.term; *bytes = N * 12 * 8; break;
        case SSA_F_ROLLOUT_TRUNCATED: *p = b.truncated; *bytes = E; break;
      }
      break;
    }
    case SSA_F_ROLLOUT_EPISODE_STATS:
      if (!h->es.on) { snprintf(g_err, sizeof(g_err), "episode statistics not enabled"); return SSA_EINVAL; }
      *p = h->es.rec; *bytes = E * SSA_EPR * 8; break;
    case SSA_F_ROLLOUT_OBS_NORM: case SSA_F_ROLLOUT_REWARD_NORM: case SSA_F_ROLLOUT_TERMINAL_OBS_NORM:
    case SSA_F_ROLLOUT_NORM_STATE: {
      if (!h->nm.on) { snprintf(g_err, sizeof(g_err), "normalization not enabled"); return SSA_EINVAL; }
      const size_t F = h->nm.F;
      if (field == SSA_F_ROLLOUT_OBS_NORM) { *p = h->nm.obs; *bytes = E * F * 4; }
      else if (field == SSA_F_ROLLOUT_REWARD_NORM) { *p = h->nm.reward; *bytes = E * 8; }
      else if (field == SSA_F_ROLLOUT_TERMINAL_OBS_NORM) { *p = h->nm.term; *bytes = E * F * 4; }
      else { *p = h->nm.state; *bytes = (4 + E + 3 * F) * 8; }
      break;
    }
    default: snprintf(g_err, sizeof(g_err), "unknown field %d", field); return SSA_EINVAL;
  }
  return SSA_OK;
}

int ssa_ukf_device_ptr(ssa_ukf* h, int field, void** dptr, size_t* bytes) {
  if (!h || !dptr) return SSA_EINVAL;
  int cols;
  size_t b;
  int rc = field_info(h, field, dptr, &b, &cols);
  if (bytes) *bytes = b;
  return rc;
}

int ssa_ukf_upload(ssa_ukf* h, int field, const void* host, size_t bytes, void* stream) {
  if (!h || !host) return SSA_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(h->device));
  void* p; size_t b; int cols;
  int rc = field_info(h, field, &p, &b, &cols);
  if (rc) return rc;
  const size_t N = h->cfg.n_objects;
  if (field == SSA_F_X_TRUE || field == SSA_F_X_FILTER) {
    if (bytes != N * 6 * 8) { snprintf(g_err, sizeof(g_err), "size mismatch"); return SSA_EINVAL; }
    rc = upload_soa(h, (const double*)host, (double*)p, 6, st);
    if (rc) return rc;
    CK(cudaStreamSynchronize(st));
    return SSA_OK;
  }
  if (field == SSA_F_P_FILTER) {
    if (bytes != N * 36 * 8) { snprintf(g_err, sizeof(g_err), "size mismatch"); return SSA_EINVAL; }
    CK(cudaMemcpyAsync(h->stage, host, bytes, cudaMemcpyHostToDevice, st));
    ssa_pfull_to_packed<<<(unsigned)((N * SSA_NP + 255) / 256), 256, 0, st>>>(h->stage, h->P, (int)N, h->ld, 1);
    h->launches++;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(st));
    return SSA_OK;
  }
  if (bytes != b) { snprintf(g_err, sizeof(g_err), "size mismatch for field %d: got %zu want %zu", field, bytes, b); return SSA_EINVAL; }
  CK(cudaMemcpyAsync(p, host, bytes, cudaMemcpyHostToDevice, st));
  return SSA_OK;
}

int ssa_ukf_download(ssa_ukf* h, int field, void* host, size_t bytes, void* stream) {
  if (!h || !host) return SSA_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(h->device));
  void* p; size_t b; int cols;
  int rc = field_info(h, field, &p, &b, &cols);
  if (rc) return rc;
  const size_t N = h->cfg.n_objects;
  if (field == SSA_F_X_TRUE || field == SSA_F_X_FILTER) {
    if (bytes != N * 6 * 8) { snprintf(g_err, sizeof(g_err), "size mismatch"); return SSA_EINVAL; }
    ssa_soa_to_aos<<<(unsigned)((N * 6 + 255) / 256), 256, 0, st>>>((const double*)p, h->stage, (int)N, 6, h->ld);
    h->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(host, h->stage, bytes, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return SSA_OK;
  }
  if (field == SSA_F_P_FILTER) {
    if (bytes != N * 36 * 8) { snprintf(g_err, sizeof(g_err), "size mismatch"); return SSA_EINVAL; }
    ssa_packed_to_pfull<<<(unsigned)((N * 36 + 255) / 256), 256, 0, st>>>(h->P, h->stage, (int)N, h->ld);
    h->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(host, h->stage, bytes, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return SSA_OK;
  }
  if (bytes != b) { snprintf(g_err, sizeof(g_err), "size mismatch for field %d: got %zu want %zu", field, bytes, b); return SSA_EINVAL; }
  CK(cudaMemcpyAsync(host, p, bytes, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return SSA_OK;
}

struct StepOverride {  // episodic mode: redirect the step's inputs / outputs
  double* obs; const int32_t* actions; const double* table; const int32_t* step_idx; int bias, rows;
  const uint8_t* env_gate;  // refresh of the re-drawn environments only (null: every environment)
};

// the episodic step's: observations in the output block, effective actions, env e's trans_matrix table row step_idx[e] + bias
static StepOverride rollout_override(const ssa_ukf* h, int bias, const uint8_t* env_gate) {
  return StepOverride{h->ro.dev.obs, h->ro.act_eff, h->ro.table, h->step_idx, bias, h->ro.n_table, env_gate};
}

static int cat_stats_launch(ssa_ukf* h, const double* dpos, const double* trace, long index_offset, cudaStream_t st, double* out);

// The parameters of the step's kernels over the whole batch (obj0 = 0, Nc = N): inputs and outputs in the handle's
// arrays, in the block of host-pipeline parity hostbuf (>= 0), or redirected by ov (episodic mode).
static KParams step_params(const ssa_ukf* h, const double M[9], int flags, int hostbuf, const StepOverride* ov) {
  KParams p;
  memset(&p, 0, sizeof(p));
  const ssa_ukf_cfg& c = h->cfg;
  p.xt = h->xt; p.x = h->x; p.P = h->P; p.status = h->status; p.infl = h->infl;
  p.actions = h->actions; p.z_noise = h->z_noise;
  p.Menv = (flags & SSA_STEP_M_PER_ENV) ? h->Menv : nullptr;
  p.Mstride = 9;
  p.obs = h->obs; p.dpos = h->dpos; p.dvel = h->dvel; p.spos = h->spos; p.svel = h->svel; p.trace = h->trace;
  if (flags & SSA_STEP_RECORD) { p.z_true = h->z_true; p.y = h->y; p.S = h->S; p.sigmas_h = h->sigmas_h; }
  p.visible = h->visible; p.updated = h->updated;
  p.lds = (h->chunk + 31) / 32 * 32;
  p.obj0 = 0; p.Nc = c.n_objects;
  p.U = h->scratch; p.F = p.U + 21 * p.lds; p.ZS = p.F + 78 * p.lds; p.UVW = p.ZS + 39 * p.lds; p.ZT = p.UVW + 39 * p.lds;
  p.code = h->code; p.exc = h->exc; p.E = c.n_envs;
  p.ld = h->ld; p.N = c.n_objects; p.m = c.m; p.flags = flags; p.obs_type = c.obs_type; p.resample = c.resample_after_predict;
  p.dt = c.dt; p.lam = c.lam_plus_n; p.obs_limit = c.obs_limit;
  memcpy(p.Wm, c.Wm, sizeof(p.Wm)); memcpy(p.Wc, c.Wc, sizeof(p.Wc));
  p.qr = h->qr;
  if (hostbuf >= 0) {  // outputs / inputs of the double-buffered host pipeline
    const PipeBlock& b = h->hp.dev[hostbuf];
    p.obs = b.obs; p.dpos = b.dpos; p.status_out = b.status; p.dvel = b.dvel; p.spos = b.spos; p.svel = b.svel; p.trace = b.trace;
    p.z_noise = b.z_noise; p.actions = b.actions;
    if (!M && !(flags & SSA_STEP_M_PER_ENV)) {  // pinned mode: the trans_matrix arrives with the input block
      p.Menv = b.M;
      p.Mstride = 0;
    }
  }
  if (ov) {
    p.obs = ov->obs; p.actions = ov->actions;
    p.Menv = ov->table; p.Mstep = ov->step_idx; p.Mbias = ov->bias; p.Mrows = ov->rows;
    p.env_gate = ov->env_gate;
  }
  if (M) memcpy(p.ob.M, M, sizeof(p.ob.M));
  memcpy(p.ob.obs_itrs, c.obs_itrs, sizeof(p.ob.obs_itrs));
  memcpy(p.ob.T, c.T, sizeof(p.ob.T));
  return p;
}

static int step_impl(ssa_ukf* h, const double M[9], int flags, void* stream, cudaEvent_t* ev, int hostbuf = -1,
                     const StepOverride* ov = nullptr) {
  if (!h) return SSA_EINVAL;
  if ((flags & (SSA_STEP_UPDATE_ALL | SSA_STEP_UPDATE_ACT | SSA_STEP_EPILOGUE)) && !M && !(flags & SSA_STEP_M_PER_ENV) &&
      hostbuf < 0 && !ov) {
    snprintf(g_err, sizeof(g_err), "trans_matrix required for update/epilogue");
    return SSA_EINVAL;
  }
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(h->device));
  KParams p = step_params(h, M, flags, hostbuf, ov);
  const ssa_ukf_cfg& c = h->cfg;
  if (ev) CK(cudaEventRecord(ev[0], st));
  if (h->kernel == StepKernel::team) {
    const unsigned grid = (unsigned)((c.n_objects + kTeamsPerCta - 1) / kTeamsPerCta);
    ssa_step_kernel<<<grid, kCtaThreads, 0, st>>>(p);
    h->launches++;
    if (ev) for (int i = 1; i <= 5; ++i) CK(cudaEventRecord(ev[i], st));
    CK(cudaGetLastError());
    return SSA_OK;
  }
  const bool predict = flags & SSA_STEP_PREDICT, truth = flags & SSA_STEP_TRUTH;
  const bool update = flags & (SSA_STEP_UPDATE_ALL | SSA_STEP_UPDATE_ACT), epi = flags & SSA_STEP_EPILOGUE;
  // per-kernel profiling (ev) runs the kernels un-chunked over the whole batch when the scratch allows it, else
  // it brackets the kernels of the first chunk only
  for (long o0 = 0; o0 < c.n_objects; o0 += h->chunk) {
    p.obj0 = o0;
    p.Nc = (int)((c.n_objects - o0) < h->chunk ? (c.n_objects - o0) : h->chunk);
    const unsigned gobj = (unsigned)((p.Nc + kSplitThreads - 1) / kSplitThreads);
    const unsigned gobj2 = (unsigned)((p.Nc + kObjThreads - 1) / kObjThreads);
    const unsigned gfx = (unsigned)((p.Nc + kFxThreads - 1) / kFxThreads);
    const unsigned gtile = (unsigned)((p.Nc + SSA_TILE - 1) / SSA_TILE);
    cudaEvent_t* evc = (ev && o0 == 0) ? ev : nullptr;
    const bool pdl = h->pdl && !ev;
    // the tile kernels keep the sigma sets in shared memory; the book-version filter (sigmas_f kept across calls)
    // and the RL-mode update of one tasked object per environment use the split kernels
    const bool tile = h->kernel != StepKernel::split && p.resample;
    if (tile && h->kernel == StepKernel::fused && predict && (flags & SSA_STEP_UPDATE_ALL)) {  // the whole step of the chunk in one launch
      launch_chain(pdl, k_step_tile<SSA_TILE, kTileThreads>, gtile, kTileThreads, sizeof(UpdateTile<SSA_TILE>), st, p, h->tm_s, h->tm_u);
      h->launches++;
      if (evc) for (int i = 1; i <= 5; ++i) CK(cudaEventRecord(evc[i], st));
      continue;
    }
    // SSA_UKF_KERNEL=tile2: the factorisations ride inside the tile kernels (two launches per catalog step, the factor
    // never in HBM) instead of running as k_factor / k_refactor (default: four launches, measured faster — DESIGN.md)
    const bool fold = tile && h->kernel == StepKernel::tile2 && predict;
    // (RL mode: the same kernel, only the tasked object of an environment takes the update — the others get the truth
    // measurement and the epilogue; the refresh after an auto-reset, gated per environment, keeps the split kernels)
    const bool tile_upd = tile && ((flags & SSA_STEP_UPDATE_ALL) || ((flags & SSA_STEP_UPDATE_ACT) && !p.env_gate && !h->act_split));
    if ((predict || update) && !fold) { launch_chain(pdl, k_factor, gobj2, kObjThreads, 0, st, p); h->launches++; }
    if (evc) CK(cudaEventRecord(evc[1], st));
    if (predict || truth) {
      // (one wave of tiles only at 5 CTAs per SM: the 56-register build of the kernel)
      const bool one_wave5 = gtile > (unsigned)h->sm_count * SSA_LB_PT && gtile <= (unsigned)h->sm_count * 5;
      if (fold) launch_chain(pdl, k_predict_tile<SSA_TILE, kTileThreads, true, SSA_LB_PT>, gtile, kTileThreads, 0, st, p, h->tm_s, h->tm_u);
      else if (tile && one_wave5) launch_chain(pdl, k_predict_tile<SSA_TILE, kTileThreads, false, 5>, gtile, kTileThreads, 0, st, p, h->tm_x, h->tm_u);
      else if (tile) launch_chain(pdl, k_predict_tile<SSA_TILE, kTileThreads, false, SSA_LB_PT>, gtile, kTileThreads, 0, st, p, h->tm_x, h->tm_u);
      else launch_chain(pdl, k_fx, dim3(gfx, 14), kFxThreads, 0, st, p);
      h->launches++;
    }
    if (evc) CK(cudaEventRecord(evc[2], st));
    const bool staged = p.Nc <= h->staged_max;
    if (predict && !(fold && tile_upd)) {
      if (tile) launch_chain(pdl, k_refactor, gobj2, kObjThreads, 0, st, p);
      else launch_chain(pdl, k_ut, gobj2, kObjThreads, 0, st, p);
      h->launches++;
    }
    if (evc) CK(cudaEventRecord(evc[3], st));
    if ((update || epi) && !tile_upd) { launch_chain(pdl, k_hx, dim3(gfx, 14), kFxThreads, 0, st, p); h->launches++; }
    if (evc) CK(cudaEventRecord(evc[4], st));
    if (update || epi) {
      if (tile_upd && fold) launch_chain(pdl, k_update_tile<SSA_TILE, kTileThreads, true>, gtile, kTileThreads, sizeof(UpdateTile<SSA_TILE>), st, p, h->tm_s, h->tm_u);
      else if (tile_upd) launch_chain(pdl, k_update_tile<SSA_TILE, kTileThreads, false>, gtile, kTileThreads, sizeof(UpdateTile<SSA_TILE>), st, p, h->tm_s, h->tm_u);
      else if (staged && p.resample && (flags & SSA_STEP_UPDATE_ALL))
        launch_chain(pdl, k_update_staged, (unsigned)((p.Nc + 31) / 32), 32, kUpdStagedSmem, st, p, h->tm_z, h->tm_u, h->tm_s);
      else launch_chain(pdl, k_update, gobj, kSplitThreads, 0, st, p);
      h->launches++;
    }
    if (evc) CK(cudaEventRecord(evc[5], st));
  }
  if (flags & SSA_STEP_CATALOG_STATS) {  // the shard's reward terms of THIS step, same chain / same graph
    // (a pinned step writes the slot of its parity: the consumer of step i may still be reading while step i + 1 runs)
    const int rc = cat_stats_launch(h, p.dpos, p.trace, h->cat_index_offset, st, hostbuf >= 0 ? h->cat_stats + 5 * (1 + hostbuf) : h->cat_stats);
    if (rc) return rc;
  }
  CK(cudaGetLastError());
  return SSA_OK;
}

int ssa_ukf_step(ssa_ukf* h, const double M[9], int flags, void* stream) {
  if (!h) return SSA_EINVAL;
  h->last_dpos = h->dpos; h->last_trace = h->trace;
  if (!h->sg.on || team_kernel(h) || (flags & SSA_STEP_M_PER_ENV) || !M || h->chunk < h->cfg.n_objects)
    return step_impl(h, M, flags, stream, nullptr);
  CK(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  int gi = -1;
  for (int i = 0; i < h->sg.n; ++i) if (h->sg.flags[i] == flags) gi = i;
  if (gi < 0) {  // capture the chain for this flag combination (at most 4 are cached)
    if (h->sg.n == 4) { cudaGraphExecDestroy(h->sg.gexec[3]); cudaGraphDestroy(h->sg.graph[3]); h->sg.n = 3; }
    gi = h->sg.n;
    const int rc = capture_chain(h, [&](cudaStream_t cs) { return step_impl(h, M, flags, cs, nullptr); },
                                 &h->sg.graph[gi], &h->sg.gexec[gi], &h->sg.gkernels[gi]);
    if (rc) return rc;
    h->sg.hx_node[gi] = nullptr;
    size_t nn = 0;
    cudaGraphGetNodes(h->sg.graph[gi], nullptr, &nn);
    cudaGraphNode_t nodes[16];
    if (nn > 16) nn = 16;
    cudaGraphGetNodes(h->sg.graph[gi], nodes, &nn);
    for (size_t i = 0; i < nn; ++i) {
      cudaGraphNodeType ty;
      cudaKernelNodeParams kp;
      if (cudaGraphNodeGetType(nodes[i], &ty) == cudaSuccess && ty == cudaGraphNodeTypeKernel &&
          cudaGraphKernelNodeGetParams(nodes[i], &kp) == cudaSuccess &&
          (kp.func == (void*)k_hx || kp.func == (void*)k_update_tile<SSA_TILE, kTileThreads, false> ||
           kp.func == (void*)k_update_tile<SSA_TILE, kTileThreads, true> ||
           kp.func == (void*)k_step_tile<SSA_TILE, kTileThreads>)) {
        h->sg.hx_node[gi] = nodes[i];
        h->sg.hx_params[gi] = kp;
      }
    }
    h->sg.flags[gi] = flags;
    h->sg.n = gi + 1;
  }
  if (h->sg.hx_node[gi]) {  // this step's trans_matrix
    KParams p = step_params(h, M, flags, -1, nullptr);  // (one chunk: the parameters of every launch of the graph)
    void* args[3] = {&p, &h->tm_s, &h->tm_u};  // k_hx takes the first, k_update_tile / k_step_tile all three
    cudaKernelNodeParams kp = h->sg.hx_params[gi];
    kp.kernelParams = args;
    kp.extra = nullptr;
    CK(cudaGraphExecKernelNodeSetParams(h->sg.gexec[gi], h->sg.hx_node[gi], &kp));
  }
  CK(cudaGraphLaunch(h->sg.gexec[gi], st));
  h->launches += h->sg.gkernels[gi];
  return SSA_OK;
}

// the handle's device current, and the double-buffered host pipeline allocated on first use
static int hostpipe_init(ssa_ukf* h) {
  CK(cudaSetDevice(h->device));
  if (h->hp.init) return SSA_OK;
  const size_t N = h->cfg.n_objects, E = h->cfg.n_envs, ld = h->ld;
  CK(cudaStreamCreateWithFlags(&h->hp.up, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&h->hp.dn, cudaStreamNonBlocking));
  const PipeBlock size = pipe_block(nullptr, nullptr, nullptr, N, E, ld);
  for (int b = 0; b < 2; ++b) {
    double *dev, *hout, *hin;
    CK(cudaMalloc(&dev, sizeof(double) * size.dev));
    CK(cudaMemset(dev, 0, sizeof(double) * size.dev));
    h->hp.dev[b] = pipe_block(dev, nullptr, nullptr, N, E, ld);
    CK(cudaHostAlloc(&hin, sizeof(double) * size.in, cudaHostAllocDefault));
    CK(cudaHostAlloc(&hout, sizeof(double) * size.hout, cudaHostAllocDefault));
    memset(hin, 0, sizeof(double) * size.in);
    memset(hout, 0, sizeof(double) * size.hout);
    h->hp.host[b] = pipe_block(nullptr, hout, hin, N, E, ld);
    CK(cudaEventCreateWithFlags(&h->hp.e_up[b], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&h->hp.e_c[b], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&h->hp.e_dn[b], cudaEventDisableTiming));
  }
  h->hp.init = 1;
  return SSA_OK;
}

int ssa_ukf_step_host(ssa_ukf* h, const double M[9], int flags, const int32_t* actions_host, const double* z_noise_host,
                      double* obs_host, double* delta_pos_host, int32_t* status_host, void* stream) {
  if (!h) return SSA_EINVAL;
  int rc = hostpipe_init(h);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t N = h->cfg.n_objects, E = h->cfg.n_envs;
  const int b = h->hp.parity;
  const PipeBlock& blk = h->hp.dev[b];
  if (!M) { snprintf(g_err, sizeof(g_err), "ssa_ukf_step_host: trans_matrix required"); return SSA_EINVAL; }
  // upload stream: buffer b is free once the compute of two calls ago has consumed it
  if (h->hp.calls >= 2) CK(cudaStreamWaitEvent(h->hp.up, h->hp.e_c[b], 0));
  if (z_noise_host) CK(cudaMemcpyAsync(blk.z_noise, z_noise_host, sizeof(double) * 3 * N, cudaMemcpyHostToDevice, h->hp.up));
  if (actions_host) CK(cudaMemcpyAsync(blk.actions, actions_host, sizeof(int32_t) * E, cudaMemcpyHostToDevice, h->hp.up));
  CK(cudaEventRecord(h->hp.e_up[b], h->hp.up));
  // compute on the caller's stream: needs this step's inputs and a drained output buffer
  CK(cudaStreamWaitEvent(st, h->hp.e_up[b], 0));
  if (h->hp.calls >= 2) CK(cudaStreamWaitEvent(st, h->hp.e_dn[b], 0));
  rc = step_impl(h, M, flags, stream, nullptr, b);
  if (rc) return rc;
  h->last_dpos = blk.dpos; h->last_trace = blk.trace;
  CK(cudaEventRecord(h->hp.e_c[b], st));
  // download stream
  CK(cudaStreamWaitEvent(h->hp.dn, h->hp.e_c[b], 0));
  if (obs_host) CK(cudaMemcpyAsync(obs_host, blk.obs, sizeof(double) * 12 * N, cudaMemcpyDeviceToHost, h->hp.dn));
  if (delta_pos_host) CK(cudaMemcpyAsync(delta_pos_host, blk.dpos, sizeof(double) * N, cudaMemcpyDeviceToHost, h->hp.dn));
  if (status_host) CK(cudaMemcpyAsync(status_host, blk.status, sizeof(int32_t) * N, cudaMemcpyDeviceToHost, h->hp.dn));
  CK(cudaEventRecord(h->hp.e_dn[b], h->hp.dn));
  h->hp.parity ^= 1;
  h->hp.calls++;
  return SSA_OK;
}

int ssa_ukf_host_join(ssa_ukf* h, void* stream) {
  if (!h) return SSA_EINVAL;
  if (!h->hp.init) return SSA_OK;
  CK(cudaSetDevice(h->device));
  const long nb = h->hp.calls >= 2 ? 2 : h->hp.calls;
  for (int b = 0; b < nb; ++b) CK(cudaStreamWaitEvent((cudaStream_t)stream, h->hp.e_dn[b], 0));
  return SSA_OK;
}

int ssa_ukf_host_io(ssa_ukf* h, int parity, double** z_noise, double** M, int32_t** actions, double** obs,
                    double** delta_pos, int32_t** status) {
  if (!h || parity < 0 || parity > 1) return SSA_EINVAL;
  int rc = hostpipe_init(h);
  if (rc) return rc;
  const PipeBlock& io = h->hp.host[parity];
  if (z_noise) *z_noise = io.z_noise;
  if (M) *M = io.M;
  if (actions) *actions = io.actions;
  if (obs) *obs = io.obs;
  if (delta_pos) *delta_pos = io.dpos;
  if (status) *status = io.status;
  return SSA_OK;
}

int ssa_ukf_host_stats(ssa_ukf* h, int parity, double** stats_host, double** stats_device) {
  if (!h || parity < 0 || parity > 1) return SSA_EINVAL;
  if (!h->cat_stats) { snprintf(g_err, sizeof(g_err), "call ssa_ukf_catalog_stats first"); return SSA_EINVAL; }
  int rc = hostpipe_init(h);
  if (rc) return rc;
  if (stats_host) *stats_host = h->hp.host[parity].stats;
  if (stats_device) *stats_device = h->cat_stats + 5 * (1 + parity);
  return SSA_OK;
}

int ssa_ukf_step_pinned(ssa_ukf* h, int flags, void* stream, int* parity_used) {
  if (!h) return SSA_EINVAL;
  const bool no_d2h = (flags & SSA_STEP_NO_D2H) != 0;
  flags &= ~SSA_STEP_NO_D2H;
  if (flags & SSA_STEP_M_PER_ENV) { snprintf(g_err, sizeof(g_err), "ssa_ukf_step_pinned: one trans_matrix per call"); return SSA_EINVAL; }
  int rc = hostpipe_init(h);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int b = h->hp.parity;
  const PipeBlock &blk = h->hp.dev[b], &io = h->hp.host[b];
  // upload stream: the device buffer is free once the compute of two calls ago has consumed it
  if (h->hp.calls >= 2) CK(cudaStreamWaitEvent(h->hp.up, h->hp.e_c[b], 0));
  CK(cudaMemcpyAsync(blk.z_noise, io.z_noise, sizeof(double) * blk.in, cudaMemcpyHostToDevice, h->hp.up));
  CK(cudaEventRecord(h->hp.e_up[b], h->hp.up));
  // compute on the caller's stream: needs this step's inputs and a drained output buffer
  CK(cudaStreamWaitEvent(st, h->hp.e_up[b], 0));
  if (h->hp.calls >= 2) CK(cudaStreamWaitEvent(st, h->hp.e_dn[b], 0));
  if (h->use_graph && !team_kernel(h)) {
    if (!h->hp.gexec[b] || h->hp.gflags[b] != flags) {  // (re)capture the kernel chain of this parity
      if (h->hp.gexec[b]) { cudaGraphExecDestroy(h->hp.gexec[b]); h->hp.gexec[b] = nullptr; }
      rc = capture_chain(h, [&](cudaStream_t cs) { return step_impl(h, nullptr, flags, cs, nullptr, b); }, nullptr, &h->hp.gexec[b],
                         &h->hp.gkernels[b]);
      if (rc) return rc;
      h->hp.gflags[b] = flags;
    }
    CK(cudaGraphLaunch(h->hp.gexec[b], st));
    h->launches += h->hp.gkernels[b];
  } else {
    rc = step_impl(h, nullptr, flags, stream, nullptr, b);
    if (rc) return rc;
  }
  h->last_dpos = blk.dpos; h->last_trace = blk.trace;
  CK(cudaEventRecord(h->hp.e_c[b], st));
  // download stream
  CK(cudaStreamWaitEvent(h->hp.dn, h->hp.e_c[b], 0));
  if (!no_d2h) CK(cudaMemcpyAsync(io.obs, blk.obs, sizeof(double) * blk.out, cudaMemcpyDeviceToHost, h->hp.dn));
  if ((flags & SSA_STEP_CATALOG_STATS) && h->cat_stats)  // the step's reward terms follow on the download stream (40 B)
    CK(cudaMemcpyAsync(io.stats, h->cat_stats + 5 * (1 + b), 5 * sizeof(double), cudaMemcpyDeviceToHost, h->hp.dn));
  CK(cudaEventRecord(h->hp.e_dn[b], h->hp.dn));
  if (parity_used) *parity_used = b;
  h->hp.parity ^= 1;
  h->hp.calls++;
  return SSA_OK;
}

// ---- device-resident episodic mode ------------------------------------------------------------------------------
static void rollout_params(ssa_ukf* h, RolloutParams* p, int only_done) {
  p->xt = h->xt; p->x = h->x; p->P = h->P; p->ld = h->ld;
  p->status = h->status; p->infl = h->infl; p->z_noise = h->z_noise;
  p->orbits = h->ro.orbits; p->n_orbits = h->ro.n_orbits;
  p->key = h->ro.key; p->episode = h->ro.episode; p->step_idx = h->step_idx;
  p->actions = h->ro.act_in; p->act_eff = h->ro.act_eff;
  p->done = only_done ? h->ro.dev.done : nullptr;
  p->sig = h->ro.sig;
  p->rew_hist = h->ro.rew_hist; p->spos_prev = h->ro.spos_prev;
  p->greedy = h->ro.dev.greedy; p->visible = h->visible;
  p->tasker = h->ro.tasker; p->spoil_p = h->ro.spoil_p;
  p->E = h->cfg.n_envs; p->m = h->cfg.m; p->update_interval = h->ro.update_interval; p->n_steps = h->cfg.n_steps;
  p->obs = h->ro.dev.obs; p->term = nullptr; p->term_aer = 0;
  p->table = h->ro.table; p->n_table = h->ro.n_table;
  memset(&p->ob, 0, sizeof(p->ob));
  memcpy(p->ob.obs_itrs, h->cfg.obs_itrs, sizeof(p->ob.obs_itrs));
  memcpy(p->ob.T, h->cfg.T, sizeof(p->ob.T));
}

// The reward / done reduction and greedy taskers of ssa_ukf_env_reduce: every environment at step_index (< 0: at its own
// step counter), into the handle's reward, done and greedy arrays; the 'shaped' reward is finished on the host.
static EnvParams env_params(ssa_ukf* h, int step_index) {
  EnvParams p = {};
  p.dpos = h->dpos; p.dvel = h->dvel; p.spos = h->spos; p.trace = h->trace; p.visible = h->visible;
  p.reward = h->reward; p.done = h->done; p.greedy = h->greedy; p.env_stats = h->env_stats;
  p.E = h->cfg.n_envs; p.m = h->cfg.m; p.reward_type = h->cfg.reward_type; p.n_steps = h->cfg.n_steps;
  p.step_index = step_index; p.step_idx = h->step_idx;
  p.P = h->P; p.ld = h->ld; p.det_prev = h->det_prev; p.det_last = h->det_last; p.det_step = h->det_step;
  p.det_cur = (p.m <= 64 && !h->det_kernel) ? nullptr : h->det_cur;  // null: determinants inside the reduction
  return p;
}

// the episodic mode's: into the output block, at the device's step counters, with its 'shaped' state (reset_mask: see EnvParams)
static EnvParams rollout_env_params(ssa_ukf* h, int increment, int greedy_only, const uint8_t* reset_mask) {
  EnvParams p = env_params(h, -1);
  p.reward = h->ro.dev.reward; p.greedy = h->ro.dev.greedy; p.done = h->ro.dev.done; p.truncated = h->ro.dev.truncated;
  p.increment = increment; p.greedy_only = greedy_only; p.reset_mask = reset_mask;
  p.rew_hist = h->ro.rew_hist; p.spos_prev = h->ro.spos_prev; p.act_in = h->ro.act_in;
  return p;
}

static void launch_env_reduce(ssa_ukf* h, const EnvParams& ep, cudaStream_t st) {
  const int N = h->cfg.n_objects;
  if (!ep.det_cur) {  // determinants inside the reduction
    ssa_env_reduce_kernel<true><<<(unsigned)((ep.E + 3) / 4), 128, 0, st>>>(ep);
    h->launches += 1;
    return;
  }
  ssa_det_kernel<<<(unsigned)((N + 127) / 128), 128, 0, st>>>(h->P, h->ld, N, h->det_cur, ep.greedy_only ? ep.reset_mask : nullptr, ep.m);
  if (ep.m <= 64) ssa_env_reduce_kernel<true><<<(unsigned)((ep.E + 3) / 4), 128, 0, st>>>(ep);
  else ssa_env_reduce_kernel<false><<<(unsigned)ep.E, 128, 0, st>>>(ep);
  h->launches += 2;
}

// obs / errors / visibility of the current states + greedy taskers (after a reset) of the environments in `mask` (the
// ones k_env_reset has just re-drawn; null: every environment)
static int rollout_refresh(ssa_ukf* h, cudaStream_t st, const uint8_t* mask) {
  // (observations, visibility, determinants and greedy actions of the other environments are this step's already)
  const StepOverride ov = rollout_override(h, 0, mask);
  int rc = step_impl(h, nullptr, SSA_STEP_EPILOGUE, st, nullptr, -1, &ov);
  if (rc) return rc;
  launch_env_reduce(h, rollout_env_params(h, 0, 1, mask), st);
  return SSA_OK;
}

int ssa_ukf_rollout_config(ssa_ukf* h, const double* orbits, int n_orbits, const double* trans_table, int n_table,
                           const uint64_t* seeds, const double x_sigma[6], const double z_sigma[3], const double P0[36],
                           int update_interval) {
  if (!h || !orbits || n_orbits < 1 || !trans_table || n_table < 1 || !seeds || !x_sigma || !z_sigma || !P0 || update_interval < 1)
    return SSA_EINVAL;
  CK(cudaSetDevice(h->device));
  const size_t N = h->cfg.n_objects, E = h->cfg.n_envs;
  // (the cached graphs of ssa_ukf_step stay valid: every pointer they captured belongs to the handle)
  rollout_free(h);
  episode_stats_free(h);  // (a new configuration runs without episode statistics until they are enabled again)
  norm_free(h);           // (nor normalization)
  h->ro.n_orbits = n_orbits; h->ro.n_table = n_table; h->ro.update_interval = update_interval;
  h->ro.tasker = SSA_TASKER_EXTERNAL; h->ro.spoil_p = 0.0;
  CK(cudaMalloc(&h->ro.dbuf, sizeof(double) * ((size_t)n_orbits * 6 + (size_t)n_table * 9 + 32)));
  h->ro.orbits = h->ro.dbuf; h->ro.table = h->ro.orbits + (size_t)n_orbits * 6; h->ro.sig = h->ro.table + (size_t)n_table * 9;
  CK(cudaMemcpy(h->ro.orbits, orbits, sizeof(double) * (size_t)n_orbits * 6, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(h->ro.table, trans_table, sizeof(double) * (size_t)n_table * 9, cudaMemcpyHostToDevice));
  double sig[30];
  for (int i = 0; i < 6; ++i) sig[i] = x_sigma[i];
  for (int i = 0; i < 3; ++i) sig[6 + i] = z_sigma[i];
  { int q = 0; for (int i = 0; i < 6; ++i) for (int j = i; j < 6; ++j) sig[9 + q++] = P0[6 * i + j]; }
  CK(cudaMemcpy(h->ro.sig, sig, sizeof(sig), cudaMemcpyHostToDevice));
  CK(cudaMalloc(&h->ro.ibuf, sizeof(uint32_t) * 5 * E));
  CK(cudaMemset(h->ro.ibuf, 0, sizeof(uint32_t) * 5 * E));
  h->ro.key = h->ro.ibuf; h->ro.episode = h->ro.key + 2 * E;
  h->ro.act_in = (int32_t*)(h->ro.episode + E); h->ro.act_eff = h->ro.act_in + E;
  CK(cudaMemcpy(h->ro.key, seeds, sizeof(uint64_t) * E, cudaMemcpyHostToDevice));  // little-endian: key[2e] = low word
  const size_t out_bytes = rollout_block(nullptr, N, E).bytes;
  void *dout, *hout;
  CK(cudaMalloc(&dout, out_bytes));
  h->ro.dev = rollout_block(dout, N, E);
  CK(cudaMemset(dout, 0, out_bytes));
  CK(cudaHostAlloc(&hout, out_bytes, cudaHostAllocDefault));
  h->ro.host = rollout_block(hout, N, E);
  CK(cudaHostAlloc(&h->ro.hin, sizeof(int32_t) * E, cudaHostAllocDefault));
  memset(hout, 0, out_bytes);
  memset(h->ro.hin, 0, sizeof(int32_t) * E);
  CK(cudaMalloc(&h->ro.dobs32, sizeof(float) * 12 * N));
  CK(cudaMemset(h->ro.dobs32, 0, sizeof(float) * 12 * N));
  CK(cudaHostAlloc(&h->ro.hobs32, sizeof(float) * 12 * N, cudaHostAllocDefault));
  memset(h->ro.hobs32, 0, sizeof(float) * 12 * N);
  CK(cudaMalloc(&h->ro.daer, sizeof(double) * 4 * N));
  CK(cudaMemset(h->ro.daer, 0, sizeof(double) * 4 * N));
  CK(cudaHostAlloc(&h->ro.haer, sizeof(double) * 4 * N, cudaHostAllocDefault));
  memset(h->ro.haer, 0, sizeof(double) * 4 * N);
  if (h->cfg.reward_type == SSA_REWARD_SHAPED) {  // the reward history lives on the device (env_reset_body clears it)
    const size_t hist = sizeof(double) * E * (size_t)h->cfg.n_steps;
    CK(cudaMalloc(&h->ro.rew_hist, hist + sizeof(int32_t) * E));
    CK(cudaMemset(h->ro.rew_hist, 0, hist + sizeof(int32_t) * E));
    h->ro.spos_prev = (int32_t*)((char*)h->ro.rew_hist + hist);
  }
  // the rows of a gathered download: n <= E final observations (term_w m <= 12 m doubles each), episode records
  // (SSA_EPR doubles) or normalized final observations (F / 2 <= 6 m doubles)
  const size_t grows = std::max(12 * N, (size_t)SSA_EPR * E);
  const size_t tbytes = sizeof(double) * (12 * N + grows) + sizeof(int32_t) * E + E;
  CK(cudaMalloc(&h->ro.tbuf, tbytes));
  CK(cudaMemset(h->ro.tbuf, 0, tbytes));
  h->ro.term = h->ro.tbuf; h->ro.gath = h->ro.term + 12 * N;
  h->ro.gidx = (int32_t*)(h->ro.gath + grows); h->ro.mask = (uint8_t*)(h->ro.gidx + E);
  CK(cudaHostAlloc(&h->ro.hgath, sizeof(double) * grows + sizeof(int32_t) * E, cudaHostAllocDefault));
  h->ro.hgidx = (int32_t*)(h->ro.hgath + grows);
  h->ro.term_w = 12;
  h->ro.init = 1;
  return SSA_OK;
}

int ssa_ukf_rollout_io(ssa_ukf* h, int32_t** actions, double** obs, double** reward, int32_t** greedy, uint8_t** done) {
  if (!rollout_ready(h)) return SSA_EINVAL;
  if (actions) *actions = h->ro.hin;
  if (obs) *obs = h->ro.host.obs;
  if (reward) *reward = h->ro.host.reward;
  if (greedy) *greedy = h->ro.host.greedy;
  if (done) *done = h->ro.host.done;
  return SSA_OK;
}

static void launch_obs_aer(ssa_ukf* h, cudaStream_t st);
// k_normalize's modes
#define SSA_NORM_STEP 0        // a step: statistics (training), normalized rows, rewards and final rows, returns[done] = 0
#define SSA_NORM_RESET 1       // ssa_ukf_rollout_reset: returns = 0, observation statistics from the fresh rows (training)
#define SSA_NORM_RESET_ENVS 2  // ssa_ukf_rollout_reset_envs: rows and returns of the masked environments, nothing updated
static void launch_normalize(ssa_ukf* h, cudaStream_t st, int mode, int auto_reset, const uint8_t* mask);
// normalized rewards and rows to their pinned host mirror (one copy: the two blocks are adjacent)
static cudaError_t norm_copy_out(ssa_ukf* h, cudaStream_t st) {
  const size_t E = h->cfg.n_envs;
  return cudaMemcpyAsync(h->nm.hbuf, h->nm.reward, sizeof(double) * E + sizeof(float) * E * h->nm.F, cudaMemcpyDeviceToHost, st);
}

// The end of ssa_ukf_rollout_reset (mask null, SSA_NORM_RESET) and of ssa_ukf_rollout_reset_envs (SSA_NORM_RESET_ENVS):
// re-draw the environments in mask (null: every environment), evaluate their fresh objects, then the output block, the
// 'aer' rows and the normalized rows to their host mirrors.
static int rollout_redraw(ssa_ukf* h, cudaStream_t st, const uint8_t* mask, int norm_mode) {
  RolloutParams rp;
  rollout_params(h, &rp, 0);
  rp.done = mask;
  k_env_reset<<<(unsigned)rp.E, 128, 0, st>>>(rp);
  h->launches++;
  int rc = rollout_refresh(h, st, mask);
  if (rc) return rc;
  launch_obs_aer(h, st);  // (the 'aer' rows of the fresh episodes, whichever layout the steps will use)
  CK(cudaMemcpyAsync(h->ro.host.obs, h->ro.dev.obs, h->ro.dev.bytes, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(h->ro.haer, h->ro.daer, sizeof(double) * 4 * h->cfg.n_objects, cudaMemcpyDeviceToHost, st));
  if (h->nm.on) {
    launch_normalize(h, st, norm_mode, 0, mask);
    CK(norm_copy_out(h, st));
  }
  CK(cudaGetLastError());
  return SSA_OK;
}

int ssa_ukf_rollout_reset(ssa_ukf* h, void* stream) {
  if (!rollout_ready(h)) return SSA_EINVAL;
  CK(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  if (h->es.on) {  // every environment starts an episode: accumulators and records cleared, accumulation from here on
    const size_t N = h->cfg.n_objects, E = h->cfg.n_envs;
    CK(cudaMemsetAsync(h->es.buf, 0, sizeof(double) * (N * SSA_EPO + E * (SSA_EPE + SSA_EPR)), st));
    if (!h->es.live) { rollout_drop_graphs(h); h->es.live = 1; }
  }
  return rollout_redraw(h, st, nullptr, SSA_NORM_RESET);
}

// the kernels of one episodic step (captured into a graph by ssa_ukf_rollout_step)
// What follows the reward / done reduction of an episodic step with auto-reset, in ONE launch: every finished environment
// is re-drawn (k_env_reset), the visibility, observations and errors of its fresh objects are evaluated (the truth slice of
// k_hx, the epilogue of k_update), the determinants of its fresh covariances stored (ssa_det_kernel) and its greedy actions
// re-evaluated (ssa_env_reduce_kernel) — one CTA per environment, the same device functions in the same order, so every
// value equals the five-launch chain's; the CTA of an environment that is still running exits at once.  With episodes of
// 480 steps the five launches found nothing to do in 479 steps of 480 and still cost ~20 us of a 130 us step.
__global__ void __launch_bounds__(128) k_env_refresh(const RolloutParams rp, const KParams p, const EnvParams ep) {
  const int e = blockIdx.x;
  if (!rp.done[e]) return;
  env_terminal_rows(rp, e);  // (the step graphs with auto-reset always record the final observations)
  env_reset_body(rp, e);  // (ends with thread 0 advancing the episode counter and zeroing the step index)
  __syncthreads();
  for (int j = threadIdx.x; j < rp.m; j += blockDim.x) {
    const long obj = (long)e * rp.m + j;
    hx_truth(p, obj, obj, false);
    update_body<false>(p, obj, obj, nullptr, 0);  // p.flags = SSA_STEP_EPILOGUE: obs row, errors, trace
    if (ep.det_cur) const_cast<double*>(ep.det_cur)[obj] = ssa_det6_sym(ep.P + obj, ep.ld);  // (h->det_cur: ssa_det_kernel's output)
  }
  __syncthreads();
  if (ep.m <= 64) {
    if (threadIdx.x < 32) env_reduce_body<true>(ep, e);
  } else {
    env_reduce_body<false>(ep, e);
  }
}

// SSA_ROLLOUT_OBS_F32: the step's observations as floats (round to nearest), two per thread
__global__ void __launch_bounds__(256) k_obs_to_f32(const double2* __restrict__ obs, float2* __restrict__ out, const long n2) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n2) {
    const double2 v = obs[i];
    out[i] = make_float2(__double2float_rn(v.x), __double2float_rn(v.y));
  }
}

// SSA_ROLLOUT_OBS_AER: the 'aer' observation of every object (obs_aer_row), one thread per object, through the
// environment's trans_matrix row min(step_idx, n_table - 1) (its row of the step just taken, step 0 after a re-draw).
__global__ void __launch_bounds__(128) k_obs_aer(const double* __restrict__ obs, const int32_t* __restrict__ step_idx,
                                                 const double* __restrict__ table, int n_table, const ssa_obs ob, int m, long N,
                                                 double* __restrict__ out) {
  const long n = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  const int i = step_idx[n / m];
  obs_aer_row(obs + n * 12, table + (long)(i < n_table - 1 ? i : n_table - 1) * 9, ob, out + n * 4);
}

static void launch_obs_aer(ssa_ukf* h, cudaStream_t st) {
  ssa_obs ob;
  memcpy(ob.obs_itrs, h->cfg.obs_itrs, sizeof(ob.obs_itrs));
  memcpy(ob.T, h->cfg.T, sizeof(ob.T));
  const long N = h->cfg.n_objects;
  k_obs_aer<<<(unsigned)((N + 127) / 128), 128, 0, st>>>(h->ro.dev.obs, h->step_idx, h->ro.table, h->ro.n_table, ob, h->cfg.m, N,
                                                         h->ro.daer);
  h->launches++;
}

// ---- running normalization of observations and returns (ssa_ukf_rollout_normalize; arithmetic: ssa_norm_* in
// ssa_ukf_core.h) ------------------------------------------------------------------------------------------------
// Device state (SSA_F_ROLLOUT_NORM_STATE): [ret mean, ret var, ret count, training][returns E][obs mean F][obs var F]
// [obs count F].  Every column keeps its own copy of the (common) observation count, so the CTA of a column reads and
// writes nothing another CTA writes and the kernel needs no grid-wide wait.
static constexpr int kNormThreads = 128;
static constexpr int kNormLeavesMax = 1024;  // ssa_norm_leaves(E) <= 1024 for every E (ssa_norm_leaf)
struct NormParams {
  const double* obs; int f32;        // rows [E][F] (the output block, or the 'aer' block); f32: float32-rounded values
  const double* term;                // final rows [E][F] (auto-reset steps), or null
  const uint8_t* done;               // [E]: the step's done flags, or the mask of SSA_NORM_RESET_ENVS
  const double* reward;              // [E]: the step's raw reward
  double* state;                     // SSA_F_ROLLOUT_NORM_STATE
  float* out; float* term_out;       // [E][F] normalized rows, normalized final rows of the finished environments
  double* reward_out;                // [E]
  float* obs32;                      // SSA_ROLLOUT_OBS_F32 steps: the float32 rows of k_obs_to_f32, or null
  int E, F, mode, norm_obs, norm_reward, reward_nan;
  double clip_obs, clip_reward, gamma, eps;
};

// the sum over the E rows of the column x[r * stride] in the order of ssa_norm_moments: the leaves in parallel, then
// every level of ssa_norm_tree in parallel over its pairs; sm holds ssa_norm_leaves(E) doubles
__device__ double norm_sum(const double* x, long stride, int E, int f32, int sq, double mean, double* sm) {
  const int L = ssa_norm_leaf(E), n = ssa_norm_leaves(E);
  for (int k = threadIdx.x; k < n; k += blockDim.x) sm[k] = ssa_norm_leaf_sum(x, stride, k * L, min(k * L + L, E), f32, sq, mean);
  __syncthreads();
  for (int s = 1; s < n; s <<= 1) {
    for (int i = 2 * s * threadIdx.x; i + s < n; i += 2 * s * blockDim.x) sm[i] = sm[i] + sm[i + s];
    __syncthreads();
  }
  const double t = sm[0];
  __syncthreads();  // (sm is reused by the next sum)
  return t;
}

// The last kernel of a step (or of a reset) with normalization on.  CTA c < F owns observation column c: batch mean and
// variance over the E rows (two passes, as np.var), merged into the column's running statistics, then the column of the
// normalized rows and of the finished environments' normalized final rows.  CTA F owns the returns: returns * gamma +
// reward, their batch moments merged into the return statistics, the normalized rewards, then returns[done] = 0.
// A column's values are F doubles apart: every load takes one 32-byte sector that the neighbouring columns' CTAs read
// too, so the rows cross from DRAM / L2 about once per pass.
__global__ void __launch_bounds__(kNormThreads) k_normalize(const NormParams p) {
  __shared__ double sm[kNormLeavesMax];
  const int c = blockIdx.x, E = p.E, F = p.F;
  double* rs = p.state;
  double* ret = rs + 4;
  const bool training = rs[3] != 0.0;
  if (c == F) {
    if (p.mode != SSA_NORM_STEP) {
      for (int e = threadIdx.x; e < E; e += blockDim.x)
        if (p.mode == SSA_NORM_RESET || p.done[e]) ret[e] = 0.0;
      return;
    }
    double m = rs[0], v = rs[1], n = rs[2];
    if (training) {
      for (int e = threadIdx.x; e < E; e += blockDim.x)
        ret[e] = ssa_norm_return(ret[e], p.gamma, ssa_norm_reward_in(p.reward[e], p.reward_nan));
      __syncthreads();
      const double bm = ssa_div(norm_sum(ret, 1, E, 0, 0, 0.0, sm), (double)E);
      const double bv = ssa_div(norm_sum(ret, 1, E, 0, 1, bm, sm), (double)E);
      ssa_norm_merge(&m, &v, &n, bm, bv, (double)E);
      if (threadIdx.x == 0) { rs[0] = m; rs[1] = v; rs[2] = n; }
    }
    const double sd = ssa_norm_sd(v, p.eps);
    for (int e = threadIdx.x; e < E; e += blockDim.x) {
      const double r = ssa_norm_reward_in(p.reward[e], p.reward_nan);
      p.reward_out[e] = p.norm_reward ? ssa_norm_reward(r, sd, p.clip_reward) : r;
      if (p.done[e]) ret[e] = 0.0;
    }
    return;
  }
  double* mean = ret + E;
  double* var = mean + F;
  double* cnt = var + F;
  double mu = mean[c], vr = var[c], n = cnt[c];
  if (p.mode != SSA_NORM_RESET_ENVS && training && p.norm_obs) {
    const double bm = ssa_div(norm_sum(p.obs + c, F, E, p.f32, 0, 0.0, sm), (double)E);
    const double bv = ssa_div(norm_sum(p.obs + c, F, E, p.f32, 1, bm, sm), (double)E);
    ssa_norm_merge(&mu, &vr, &n, bm, bv, (double)E);
    if (threadIdx.x == 0) { mean[c] = mu; var[c] = vr; cnt[c] = n; }
  }
  const double sd = ssa_norm_sd(vr, p.eps);
  constexpr int U = 8;  // rows per thread whose loads are issued together
  for (int e0 = threadIdx.x; e0 < E; e0 += U * blockDim.x) {
    double x[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int e = e0 + u * blockDim.x;
      x[u] = e < E ? p.obs[(long)e * F + c] : 0.0;
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int e = e0 + u * blockDim.x;
      if (e >= E) break;
      if (p.mode == SSA_NORM_RESET_ENVS && !p.done[e]) continue;
      const long i = (long)e * F + c;
      const double v = ssa_norm_in(x[u], p.f32);
      p.out[i] = (float)(p.norm_obs ? ssa_norm_obs(v, mu, sd, p.clip_obs) : v);
      if (p.obs32) p.obs32[i] = (float)x[u];
      if (p.term && p.done[e]) {
        const double t = ssa_norm_in(p.term[i], p.f32);
        p.term_out[i] = (float)(p.norm_obs ? ssa_norm_obs(t, mu, sd, p.clip_obs) : t);
      }
    }
  }
}

static void launch_normalize(ssa_ukf* h, cudaStream_t st, int mode, int auto_reset, const uint8_t* mask) {
  const size_t E = h->cfg.n_envs;
  const ssa_norm_cfg& c = h->nm.cfg;
  NormParams p;
  p.obs = c.obs_layout == SSA_NORM_OBS_AER ? h->ro.daer : h->ro.dev.obs;
  p.f32 = c.obs_layout == SSA_NORM_OBS_ROWS_F32;
  p.term = mode == SSA_NORM_STEP && auto_reset ? h->ro.term : nullptr;
  p.reward = h->ro.dev.reward;
  p.done = mode == SSA_NORM_RESET_ENVS ? mask : h->ro.dev.done;
  p.state = h->nm.state; p.out = h->nm.obs; p.term_out = h->nm.term; p.reward_out = h->nm.reward;
  p.obs32 = mode == SSA_NORM_STEP && p.f32 ? h->ro.dobs32 : nullptr;
  p.E = (int)E; p.F = h->nm.F; p.mode = mode;
  p.norm_obs = c.norm_obs; p.norm_reward = c.norm_reward; p.reward_nan = c.reward_nan_to_num;
  p.clip_obs = c.clip_obs; p.clip_reward = c.clip_reward; p.gamma = c.gamma; p.eps = c.epsilon;
  k_normalize<<<(unsigned)(p.F + 1), kNormThreads, 0, st>>>(p);
  h->launches++;
}

// ---- per-episode statistics (ssa_ukf_rollout_episode_stats_*; accumulator layouts in ssa_ukf_core.h) ---------------
struct EpParams {
  const double* xt; const double* x; const double* P; long ld;   // state (SoA)
  const int32_t* step_idx; const int32_t* act_eff;                // [E]
  const uint8_t* updated; const double* y; const double* S;       // [N], [N][3], [N][9] (SSA_STEP_RECORD)
  const double* reward; const uint8_t* done;                      // [E] of the output block
  const int32_t* status;                                          // [N]
  double* obj; double* env; double* rec;                          // [N][SSA_EPO], [E][SSA_EPE], [E][SSA_EPR]
  int E, m, auto_reset;
};
static_assert(SSA_EPR == SSA_EPISODE_STATS_DOUBLES, "episode record layout");

static void ep_params(ssa_ukf* h, EpParams* p, int auto_reset) {
  p->xt = h->xt; p->x = h->x; p->P = h->P; p->ld = h->ld;
  p->step_idx = h->step_idx; p->act_eff = h->ro.act_eff;
  p->updated = h->updated; p->y = h->y; p->S = h->S;
  p->reward = h->ro.dev.reward; p->done = h->ro.dev.done;
  p->status = h->status;
  p->obj = h->es.obj; p->env = h->es.env; p->rec = h->es.rec;
  p->E = h->cfg.n_envs; p->m = h->cfg.m; p->auto_reset = auto_reset;
}

// head of an episodic step: row 0 (the fresh draw, before the first predict) of the environments at step index 0, one
// thread per object
__global__ void __launch_bounds__(128) k_ep_row0(const EpParams p) {
  const long n = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= (long)p.E * p.m || p.step_idx[n / p.m] != 0) return;
  ssa_ep_nees_row(p.obj + n * SSA_EPO, p.xt + n, p.x + n, p.ld, p.P + n, p.ld);
}

// after the reward / done reduction, before a finished environment is re-drawn: one warp per environment, four per CTA.
// The lanes add the NEES of the step's row of every object; lane 0 then adds the tasked object's innovation terms and
// the step reward, and for a finished environment writes the record (and clears the accumulators with auto-reset).
__global__ void __launch_bounds__(128) k_ep_step(const EpParams p) {
  const int e = (int)(blockIdx.x * 4 + (threadIdx.x >> 5)), lane = threadIdx.x & 31;
  if (e >= p.E) return;  // (warp-uniform)
  const long b = (long)e * p.m;
  for (int j = lane; j < p.m; j += 32)
    ssa_ep_nees_row(p.obj + (b + j) * SSA_EPO, p.xt + b + j, p.x + b + j, p.ld, p.P + b + j, p.ld);
  __syncwarp();  // (lane 0 reads the object accumulators of the other lanes below)
  if (lane) return;
  double* env = p.env + (long)e * SSA_EPE;
  double* obj = p.obj + b * SSA_EPO;
  const int a = p.act_eff[e];
  if (a >= 0 && a < p.m && p.updated[b + a]) ssa_ep_observe(env, obj + (long)a * SSA_EPO, p.y + (b + a) * 3, p.S + (b + a) * 9);
  env[SSA_EPE_RET] = env[SSA_EPE_RET] + p.reward[e];
  if (p.done[e]) {
    ssa_ep_finalise(env, obj, p.status + b, p.m, (double)p.step_idx[e], p.rec + (long)e * SSA_EPR);
    if (p.auto_reset) ssa_ep_clear(env, obj, p.m);
  }
}

// rows idx[0 .. n) of `row` doubles each, packed into out (the downloads of episode records and final observations)
__global__ void __launch_bounds__(256) k_gather_rows(const double* __restrict__ src, const int32_t* __restrict__ idx, int n,
                                                     long row, double* __restrict__ out) {
  const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n * row) out[t] = src[(long)idx[t / row] * row + t % row];
}

static int rollout_chain(ssa_ukf* h, cudaStream_t st, int auto_reset, int obs_f32, int obs_aer) {
  RolloutParams rp;
  rollout_params(h, &rp, 1);
  const long N = h->cfg.n_objects;
  const bool stats = h->es.live != 0;
  EpParams sp;
  if (stats) {
    ep_params(h, &sp, auto_reset);
    k_ep_row0<<<(unsigned)((N + 127) / 128), 128, 0, st>>>(sp);
    h->launches++;
  }
  k_env_begin<<<(unsigned)((N + 127) / 128), 128, 0, st>>>(rp);
  h->launches++;
  const StepOverride ov = rollout_override(h, 1, nullptr);
  int rc = step_impl(h, nullptr, SSA_STEP_TRUTH | SSA_STEP_PREDICT | SSA_STEP_UPDATE_ACT | SSA_STEP_EPILOGUE | (stats ? SSA_STEP_RECORD : 0),
                     st, nullptr, -1, &ov);
  if (rc) return rc;
  launch_env_reduce(h, rollout_env_params(h, 1, 0, nullptr), st);
  if (auto_reset) { rp.term = h->ro.term; rp.term_aer = obs_aer; }  // (k_env_refresh / k_env_reset record them)
  if (stats) {
    k_ep_step<<<(unsigned)((rp.E + 3) / 4), 128, 0, st>>>(sp);
    h->launches++;
  }
  if (auto_reset && !team_kernel(h) && !h->refresh_chain) {  // one launch (k_env_refresh)
    const StepOverride rov = rollout_override(h, 0, rp.done);
    k_env_refresh<<<(unsigned)rp.E, 128, 0, st>>>(rp, step_params(h, nullptr, SSA_STEP_EPILOGUE, -1, &rov), rollout_env_params(h, 0, 1, rp.done));
    h->launches++;
  } else if (auto_reset) {  // SSA_UKF_REFRESH_CHAIN=1 / team kernel: k_env_reset, then the gated refresh chain
    k_env_reset<<<(unsigned)rp.E, 128, 0, st>>>(rp);
    h->launches++;
    rc = rollout_refresh(h, st, rp.done);
    if (rc) return rc;
  }
  const bool norm = h->nm.on != 0;
  if (obs_f32 && !norm) {  // (with normalization k_normalize writes the float32 rows)
    const long n2 = 6 * N;  // 12 N doubles, two at a time (the block is cudaMalloc-aligned)
    k_obs_to_f32<<<(unsigned)((n2 + 255) / 256), 256, 0, st>>>((const double2*)h->ro.dev.obs, (float2*)h->ro.dobs32, n2);
    h->launches++;
  }
  if (obs_aer) launch_obs_aer(h, st);
  if (norm) launch_normalize(h, st, SSA_NORM_STEP, auto_reset, nullptr);
  return SSA_OK;
}

int ssa_ukf_rollout_obs_aer(ssa_ukf* h, double** host, double** device) {
  if (!rollout_ready(h)) return SSA_EINVAL;
  if (host) *host = h->ro.haer;
  if (device) *device = h->ro.daer;
  return SSA_OK;
}

int ssa_ukf_rollout_obs_f32(ssa_ukf* h, float** host, float** device) {
  if (!rollout_ready(h)) return SSA_EINVAL;
  if (host) *host = h->ro.hobs32;
  if (device) *device = h->ro.dobs32;
  return SSA_OK;
}

int ssa_ukf_rollout_episode_stats_enable(ssa_ukf* h) {
  if (!rollout_ready(h)) return SSA_EINVAL;
  CK(cudaSetDevice(h->device));
  const size_t N = h->cfg.n_objects, E = h->cfg.n_envs;
  if (h->es.on) { CK(cudaDeviceSynchronize()); episode_stats_free(h); }
  const size_t acc = N * SSA_EPO + E * (SSA_EPE + SSA_EPR);
  CK(cudaMalloc(&h->es.buf, sizeof(double) * acc));
  CK(cudaMemset(h->es.buf, 0, sizeof(double) * acc));
  h->es.obj = h->es.buf; h->es.env = h->es.obj + N * SSA_EPO; h->es.rec = h->es.env + E * SSA_EPE;
  h->es.on = 1;
  h->es.live = 0;  // (from the next ssa_ukf_rollout_reset)
  rollout_drop_graphs(h);
  return SSA_OK;
}

// the environment list of a download / reset: 0 <= n <= E entries, each in [0, E) (and, for a download, an output)
static int check_envs(const ssa_ukf* h, const int32_t* envs, int n, const void* out) {
  const int E = h->cfg.n_envs;
  if (n < 0 || n > E || (n > 0 && (!envs || !out))) { snprintf(g_err, sizeof(g_err), "bad environment list"); return SSA_EINVAL; }
  for (int k = 0; k < n; ++k)
    if (envs[k] < 0 || envs[k] >= E) { snprintf(g_err, sizeof(g_err), "environment index %d out of range", envs[k]); return SSA_EINVAL; }
  return SSA_OK;
}

// the rows envs[0 .. n) (0 < n <= E, checked) of `row` doubles each of src into out, through the gather scratch of the
// handle; returns once copied, so the downloads can share that scratch (one host thread per handle)
static int gather_download(ssa_ukf* h, const double* src, long row, const int32_t* envs, int n, void* out, cudaStream_t st) {
  CK(cudaSetDevice(h->device));
  memcpy(h->ro.hgidx, envs, sizeof(int32_t) * n);
  CK(cudaMemcpyAsync(h->ro.gidx, h->ro.hgidx, sizeof(int32_t) * n, cudaMemcpyHostToDevice, st));
  k_gather_rows<<<(unsigned)((n * row + 255) / 256), 256, 0, st>>>(src, h->ro.gidx, n, row, h->ro.gath);
  h->launches++;
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(h->ro.hgath, h->ro.gath, sizeof(double) * n * row, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  memcpy(out, h->ro.hgath, sizeof(double) * n * row);
  return SSA_OK;
}

int ssa_ukf_rollout_episode_stats_download(ssa_ukf* h, const int32_t* envs, int n, double* out, void* stream) {
  if (!h) return SSA_EINVAL;
  if (!h->es.on) { snprintf(g_err, sizeof(g_err), "episode statistics not enabled"); return SSA_EINVAL; }
  if (check_envs(h, envs, n, out)) return SSA_EINVAL;
  if (n == 0) return SSA_OK;
  return gather_download(h, h->es.rec, SSA_EPR, envs, n, out, (cudaStream_t)stream);
}

int ssa_ukf_rollout_truncated(ssa_ukf* h, uint8_t** host, uint8_t** device) {
  if (!rollout_ready(h)) return SSA_EINVAL;
  if (host) *host = h->ro.host.truncated;
  if (device) *device = h->ro.dev.truncated;
  return SSA_OK;
}

int ssa_ukf_rollout_terminal_obs_download(ssa_ukf* h, const int32_t* envs, int n, double* out, void* stream) {
  if (!rollout_ready(h)) return SSA_EINVAL;
  if (check_envs(h, envs, n, out)) return SSA_EINVAL;
  if (n == 0) return SSA_OK;
  // (rows of term_w doubles per object: the layout of the last auto-reset step)
  return gather_download(h, h->ro.term, (long)h->ro.term_w * h->cfg.m, envs, n, out, (cudaStream_t)stream);
}

// ssa_ukf_rollout_reset_envs with episode statistics: the accumulators of the re-drawn environments start afresh
__global__ void __launch_bounds__(128) k_ep_clear(double* env, double* obj, const uint8_t* __restrict__ mask, int E, int m) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e < E && mask[e]) ssa_ep_clear(env + (long)e * SSA_EPE, obj + (long)e * m * SSA_EPO, m);
}

int ssa_ukf_rollout_reset_envs(ssa_ukf* h, const int32_t* envs, int n, void* stream) {
  if (!rollout_ready(h)) return SSA_EINVAL;
  if (check_envs(h, envs, n, envs)) return SSA_EINVAL;
  if (n == 0) return SSA_OK;
  CK(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  const int E = h->cfg.n_envs;
  // (a pageable source: the copy has read it when cudaMemcpyAsync returns, so the vector may go out of scope)
  std::vector<uint8_t> mask(E, 0);
  for (int k = 0; k < n; ++k) mask[envs[k]] = 1;
  CK(cudaMemcpyAsync(h->ro.mask, mask.data(), E, cudaMemcpyHostToDevice, st));
  if (h->es.live) {
    k_ep_clear<<<(unsigned)((E + 127) / 128), 128, 0, st>>>(h->es.env, h->es.obj, h->ro.mask, E, h->cfg.m);
    h->launches++;
  }
  return rollout_redraw(h, st, h->ro.mask, SSA_NORM_RESET_ENVS);
}

int ssa_ukf_rollout_step(ssa_ukf* h, int auto_reset, void* stream) {
  if (!rollout_ready(h)) return SSA_EINVAL;
  CK(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  const size_t E = h->cfg.n_envs;
  const bool obs_f32 = (auto_reset & SSA_ROLLOUT_OBS_F32) != 0, obs_aer = (auto_reset & SSA_ROLLOUT_OBS_AER) != 0;
  if (obs_f32 && obs_aer) {
    snprintf(g_err, sizeof(g_err), "SSA_ROLLOUT_OBS_F32 and SSA_ROLLOUT_OBS_AER exclude each other");
    return SSA_EINVAL;
  }
  if (h->nm.on && (obs_aer ? SSA_NORM_OBS_AER : obs_f32 ? SSA_NORM_OBS_ROWS_F32 : SSA_NORM_OBS_ROWS) != h->nm.cfg.obs_layout) {
    snprintf(g_err, sizeof(g_err), "the step's observation layout is not the one ssa_ukf_rollout_normalize was given");
    return SSA_EINVAL;
  }
  const int ar = (auto_reset & 1) ? 1 : 0;
  const int a = ar + (obs_f32 ? 2 : obs_aer ? 4 : 0);
  if (ar) h->ro.term_w = obs_aer ? 4 : 12;  // (the layout of the final observations this step records)
  const bool device_io = (auto_reset & SSA_ROLLOUT_DEVICE_IO) != 0, tasked = h->ro.tasker != SSA_TASKER_EXTERNAL;
  if (!device_io && !tasked) CK(cudaMemcpyAsync(h->ro.act_in, h->ro.hin, sizeof(int32_t) * E, cudaMemcpyHostToDevice, st));
  if (h->use_graph && !team_kernel(h)) {
    if (!h->ro.gexec[a]) {
      const int rc = capture_chain(h, [&](cudaStream_t cs) { return rollout_chain(h, cs, ar, obs_f32, obs_aer); }, nullptr,
                                   &h->ro.gexec[a], &h->ro.gkernels[a]);
      if (rc) return rc;
    }
    CK(cudaGraphLaunch(h->ro.gexec[a], st));
    h->launches += h->ro.gkernels[a];
  } else {
    const int rc = rollout_chain(h, st, ar, obs_f32, obs_aer);
    if (rc) return rc;
  }
  if (!device_io) {
    // the observations in the step's layout: normalized (with the normalized rewards), float, 'aer', or the double rows
    // of the output block; then the rest of the block (the raw reward, greedy, done and truncated tail)
    const size_t N = h->cfg.n_objects;
    size_t from = h->ro.dev.tail;
    if (h->nm.on) CK(norm_copy_out(h, st));
    else if (obs_f32) CK(cudaMemcpyAsync(h->ro.hobs32, h->ro.dobs32, sizeof(float) * 12 * N, cudaMemcpyDeviceToHost, st));
    else if (obs_aer) CK(cudaMemcpyAsync(h->ro.haer, h->ro.daer, sizeof(double) * 4 * N, cudaMemcpyDeviceToHost, st));
    else from = 0;
    CK(cudaMemcpyAsync((char*)h->ro.host.obs + from, (char*)h->ro.dev.obs + from, h->ro.dev.bytes - from, cudaMemcpyDeviceToHost, st));
    if (tasked) CK(cudaMemcpyAsync(h->ro.hin, h->ro.act_in, sizeof(int32_t) * E, cudaMemcpyDeviceToHost, st));  // taken
  }
  return SSA_OK;
}

int ssa_ukf_rollout_tasker(ssa_ukf* h, int tasker, double spoil_p) {
  if (!rollout_ready(h)) return SSA_EINVAL;
  if (tasker < SSA_TASKER_EXTERNAL || tasker > SSA_TASKER_VISIBLE_GREEDY_SPOILED) {
    snprintf(g_err, sizeof(g_err), "unknown tasker %d", tasker);
    return SSA_EINVAL;
  }
  if (!(spoil_p >= 0.0 && spoil_p <= 1.0)) {  // (NaN fails both comparisons)
    snprintf(g_err, sizeof(g_err), "spoil_p %g outside [0, 1]", spoil_p);
    return SSA_EINVAL;
  }
  if (tasker != h->ro.tasker || spoil_p != h->ro.spoil_p) rollout_drop_graphs(h);  // (both are captured kernel parameters)
  h->ro.tasker = tasker;
  h->ro.spoil_p = spoil_p;
  return SSA_OK;
}

int ssa_ukf_rollout_normalize(ssa_ukf* h, const ssa_norm_cfg* cfg) {
  if (!rollout_ready(h)) return SSA_EINVAL;
  CK(cudaSetDevice(h->device));
  if (!cfg) {
    if (h->nm.on) { CK(cudaDeviceSynchronize()); norm_free(h); rollout_drop_graphs(h); }
    return SSA_OK;
  }
  if (!(cfg->gamma >= 0.0 && cfg->gamma <= 1.0)) { snprintf(g_err, sizeof(g_err), "gamma %g outside [0, 1]", cfg->gamma); return SSA_EINVAL; }
  if (!(cfg->clip_obs > 0.0 && cfg->clip_reward > 0.0)) {
    snprintf(g_err, sizeof(g_err), "clip_obs %g and clip_reward %g must be > 0", cfg->clip_obs, cfg->clip_reward);
    return SSA_EINVAL;
  }
  if (!(cfg->epsilon >= 0.0)) { snprintf(g_err, sizeof(g_err), "epsilon %g must be >= 0", cfg->epsilon); return SSA_EINVAL; }
  if (cfg->obs_layout < SSA_NORM_OBS_ROWS || cfg->obs_layout > SSA_NORM_OBS_AER) {
    snprintf(g_err, sizeof(g_err), "unknown obs_layout %d", cfg->obs_layout);
    return SSA_EINVAL;
  }
  ssa_norm_cfg c = *cfg;
  c.norm_obs = c.norm_obs != 0; c.norm_reward = c.norm_reward != 0; c.training = c.training != 0;
  c.reward_nan_to_num = c.reward_nan_to_num != 0;
  const size_t E = h->cfg.n_envs, F = (size_t)(c.obs_layout == SSA_NORM_OBS_AER ? 4 : 12) * h->cfg.m;
  if (h->nm.on && h->nm.F == (int)F) {  // the statistics carry over; only training is read from device memory
    const ssa_norm_cfg& o = h->nm.cfg;
    if (o.norm_obs != c.norm_obs || o.norm_reward != c.norm_reward || o.obs_layout != c.obs_layout ||
        o.reward_nan_to_num != c.reward_nan_to_num || o.clip_obs != c.clip_obs || o.clip_reward != c.clip_reward ||
        o.gamma != c.gamma || o.epsilon != c.epsilon)
      rollout_drop_graphs(h);  // (captured kernel parameters)
    if (o.training != c.training) {
      const double t = c.training;
      CK(cudaDeviceSynchronize());  // (no step in flight reads the flag while it changes)
      CK(cudaMemcpy(h->nm.state + 3, &t, sizeof(double), cudaMemcpyHostToDevice));
    }
    h->nm.cfg = c;
    return SSA_OK;
  }
  if (h->nm.on) { CK(cudaDeviceSynchronize()); norm_free(h); }
  const size_t sd = 4 + E + 3 * F;  // state doubles
  const size_t bytes = sizeof(double) * (sd + E) + sizeof(float) * 2 * E * F;
  CK(cudaMalloc(&h->nm.buf, bytes));
  CK(cudaMemset(h->nm.buf, 0, bytes));
  h->nm.state = h->nm.buf; h->nm.reward = h->nm.state + sd;
  h->nm.obs = (float*)(h->nm.reward + E); h->nm.term = h->nm.obs + E * F;
  // RunningMeanStd(): mean 0, var 1, count 1e-4; the returns 0
  std::vector<double> st(sd, 0.0);
  st[1] = 1.0; st[2] = 1e-4; st[3] = c.training;
  for (size_t k = 0; k < F; ++k) { st[4 + E + F + k] = 1.0; st[4 + E + 2 * F + k] = 1e-4; }
  CK(cudaMemcpy(h->nm.state, st.data(), sizeof(double) * sd, cudaMemcpyHostToDevice));
  const size_t hbytes = sizeof(double) * E + sizeof(float) * E * F;
  CK(cudaHostAlloc(&h->nm.hbuf, hbytes, cudaHostAllocDefault));
  memset(h->nm.hbuf, 0, hbytes);
  h->nm.hobs = (float*)(h->nm.hbuf + E);
  h->nm.cfg = c; h->nm.F = (int)F; h->nm.on = 1;
  rollout_drop_graphs(h);
  return SSA_OK;
}

int ssa_ukf_rollout_norm_io(ssa_ukf* h, float** obs, double** reward) {
  if (!h || !h->nm.on) { snprintf(g_err, sizeof(g_err), "normalization not enabled"); return SSA_EINVAL; }
  if (obs) *obs = h->nm.hobs;
  if (reward) *reward = h->nm.hbuf;
  return SSA_OK;
}

// the saved state [obs mean F][obs var F][obs count][ret mean][ret var][ret count][returns E] <-> the device state
static int norm_state_check(ssa_ukf* h, const void* buf, size_t n) {
  if (!h || !h->nm.on) { snprintf(g_err, sizeof(g_err), "normalization not enabled"); return SSA_EINVAL; }
  const size_t want = 2 * (size_t)h->nm.F + 4 + h->cfg.n_envs;
  if (!buf || n != want) { snprintf(g_err, sizeof(g_err), "state buffer of %zu doubles, want %zu", n, want); return SSA_EINVAL; }
  return SSA_OK;
}

int ssa_ukf_rollout_norm_state_download(ssa_ukf* h, double* out, size_t n, void* stream) {
  if (norm_state_check(h, out, n)) return SSA_EINVAL;
  CK(cudaSetDevice(h->device));
  const size_t E = h->cfg.n_envs, F = h->nm.F;
  std::vector<double> d(4 + E + 3 * F);
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaMemcpyAsync(d.data(), h->nm.state, sizeof(double) * d.size(), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  const double* col = d.data() + 4 + E;
  memcpy(out, col, sizeof(double) * 2 * F);
  out[2 * F] = col[2 * F];
  memcpy(out + 2 * F + 1, d.data(), sizeof(double) * 3);
  memcpy(out + 2 * F + 4, d.data() + 4, sizeof(double) * E);
  return SSA_OK;
}

int ssa_ukf_rollout_norm_state_upload(ssa_ukf* h, const double* in, size_t n, void* stream) {
  if (norm_state_check(h, in, n)) return SSA_EINVAL;
  CK(cudaSetDevice(h->device));
  const size_t E = h->cfg.n_envs, F = h->nm.F;
  std::vector<double> d(4 + E + 3 * F);
  memcpy(d.data(), in + 2 * F + 1, sizeof(double) * 3);
  d[3] = h->nm.cfg.training;
  memcpy(d.data() + 4, in + 2 * F + 4, sizeof(double) * E);
  memcpy(d.data() + 4 + E, in, sizeof(double) * 2 * F);
  for (size_t k = 0; k < F; ++k) d[4 + E + 2 * F + k] = in[2 * F];
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaMemcpyAsync(h->nm.state, d.data(), sizeof(double) * d.size(), cudaMemcpyHostToDevice, st));
  CK(cudaStreamSynchronize(st));
  return SSA_OK;
}

int ssa_ukf_rollout_terminal_obs_norm_download(ssa_ukf* h, const int32_t* envs, int n, float* out, void* stream) {
  if (!h || !h->nm.on) { snprintf(g_err, sizeof(g_err), "normalization not enabled"); return SSA_EINVAL; }
  if (check_envs(h, envs, n, out)) return SSA_EINVAL;
  if (n == 0) return SSA_OK;
  // (a row of F floats as F / 2 doubles: F = 12 m or 4 m is even)
  return gather_download(h, (const double*)h->nm.term, h->nm.F / 2, envs, n, out, (cudaStream_t)stream);
}

int ssa_ukf_step_profile(ssa_ukf* h, const double M[9], int flags, void* stream, double ms[5]) {
  if (!h || !ms) return SSA_EINVAL;
  CK(cudaSetDevice(h->device));
  cudaEvent_t ev[6];
  for (int i = 0; i < 6; ++i) CK(cudaEventCreate(&ev[i]));
  int rc = step_impl(h, M, flags, stream, ev);
  if (rc == SSA_OK) {
    CK(cudaEventSynchronize(ev[5]));
    for (int i = 0; i < 5; ++i) {
      float t = 0.f;
      CK(cudaEventElapsedTime(&t, ev[i], ev[i + 1]));
      ms[i] = t;
    }
  }
  for (int i = 0; i < 6; ++i) cudaEventDestroy(ev[i]);
  return rc;
}

int ssa_ukf_predict(ssa_ukf* h, void* stream) {
  return ssa_ukf_step(h, nullptr, SSA_STEP_TRUTH | SSA_STEP_PREDICT, stream);
}
int ssa_ukf_update(ssa_ukf* h, const double M[9], int all, void* stream) {
  return ssa_ukf_step(h, M, (all ? SSA_STEP_UPDATE_ALL : SSA_STEP_UPDATE_ACT) | SSA_STEP_EPILOGUE, stream);
}

int ssa_ukf_env_reduce(ssa_ukf* h, const double M[9], int step_index, void* stream) {
  (void)M;
  if (!h) return SSA_EINVAL;
  CK(cudaSetDevice(h->device));
  launch_env_reduce(h, env_params(h, step_index), (cudaStream_t)stream);
  CK(cudaGetLastError());
  return SSA_OK;
}

size_t ssa_ukf_snapshot_bytes(const ssa_ukf* h) {
  return h ? (size_t)h->cfg.n_objects * (kSnapDoubles * sizeof(double) + sizeof(int32_t) + 2) : 0;
}

int ssa_ukf_snapshot(ssa_ukf* h, void* host, size_t bytes, void* stream) {
  if (!h || !host) return SSA_EINVAL;
  const size_t need = ssa_ukf_snapshot_bytes(h);
  if (bytes != need) { snprintf(g_err, sizeof(g_err), "ssa_ukf_snapshot: got %zu bytes, want %zu", bytes, need); return SSA_EINVAL; }
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(h->device));
  if (!h->snap) CK(cudaMalloc(&h->snap, need));
  SnapParams p;
  p.xt = h->xt; p.x = h->x; p.P = h->P; p.obs = h->obs; p.dpos = h->dpos; p.dvel = h->dvel; p.spos = h->spos; p.svel = h->svel;
  p.z_true = h->z_true; p.y = h->y; p.S = h->S; p.sigmas_h = h->sigmas_h;
  p.status = h->status; p.visible = h->visible; p.updated = h->updated;
  p.ld = h->ld; p.N = h->cfg.n_objects; p.out = (double*)h->snap;
  ssa_snapshot_kernel<<<(unsigned)((p.N + 127) / 128), 128, 0, st>>>(p);
  h->launches++;
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(host, h->snap, need, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return SSA_OK;
}

static int cat_stats_launch(ssa_ukf* h, const double* dpos, const double* trace, long index_offset, cudaStream_t st, double* out) {
  if (!h->cat_part) {
    snprintf(g_err, sizeof(g_err), "SSA_STEP_CATALOG_STATS: call ssa_ukf_catalog_stats once first (it sets the index offset)");
    return SSA_EINVAL;
  }
  const long N = h->cfg.n_objects;
  int nb = (int)((N + 255) / 256);
  nb = nb > kStatBlocks ? kStatBlocks : nb;
  ssa_cat_stats_stage1<<<nb, 256, 0, st>>>(dpos, trace, N, (CatPart*)h->cat_part);
  ssa_cat_stats_stage2<<<1, 256, 0, st>>>((const CatPart*)h->cat_part, nb, N, index_offset, out);
  h->launches += 2;
  return SSA_OK;
}

int ssa_ukf_catalog_stats(ssa_ukf* h, long index_offset, void* stream) {
  if (!h) return SSA_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(h->device));
  if (!h->cat_part) {
    CK(cudaMalloc(&h->cat_part, sizeof(CatPart) * kStatBlocks + 16 * sizeof(double)));
    h->cat_stats = (double*)((CatPart*)h->cat_part + kStatBlocks);  // [3][5]: plain steps | pinned parity 0 | pinned parity 1
    CK(cudaMemsetAsync(h->cat_stats, 0, 16 * sizeof(double), st));
  }
  h->cat_index_offset = index_offset;
  // the reward terms of the MOST RECENT step: its delta_pos / trace live in the handle's arrays or, after a pinned /
  // host-pipelined step, in that call's output block
  const int rc = cat_stats_launch(h, h->last_dpos ? h->last_dpos : h->dpos, h->last_trace ? h->last_trace : h->trace, index_offset, st, h->cat_stats);
  if (rc) return rc;
  CK(cudaGetLastError());
  return SSA_OK;
}

int ssa_ukf_diagnostics(ssa_ukf* h, void* stream) {
  if (!h) return SSA_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(h->device));
  const int N = h->cfg.n_objects;
  ssa_diag_kernel<<<(unsigned)((N + 127) / 128), 128, 0, st>>>(h->xt, h->x, h->P, h->y, h->S, h->updated, h->diag, h->innov_flags,
                                                             h->ld, N);
  h->launches++;
  CK(cudaGetLastError());
  return SSA_OK;
}

// HOST: the trans_matrix table of an episode (csrc/ssa_frames.h); no device needed
int ssa_trans_matrix_table(int year, int month, int day, double seconds_of_day, double dt, int n, const double* eop, int n_eop,
                           double* out) {
  if (n < 1 || !out || month < 1 || month > 12 || day < 1 || day > 31 || !(dt == dt) || (eop && n_eop < 2)) return SSA_EINVAL;
  const long mjd0 = (long)ssa_frames::cal2mjd(year, month, day);
  for (int i = 0; i < n; ++i) {
    const double total = seconds_of_day + dt * (double)i;
    const double days = floor(total / 86400.0);
    const double sec = floor(total - days * 86400.0);  // whole seconds, like the reference's datetime.hour / minute / second
    const ssa_frames::M3 m = ssa_frames::gcrs2itrs(mjd0 + (long)days, sec, eop, n_eop);
    for (int r = 0; r < 3; ++r)
      for (int c = 0; c < 3; ++c) out[9 * (size_t)i + 3 * r + c] = m.a[r][c];
  }
  return SSA_OK;
}

int ssa_orbit_gen_eval(const double* cand, int K, const double* trans_table, int n, double step_s, const double obs_itrs[3],
                       const double T[9], double obs_limit, double min_alt, int first_window, int max_gap, uint8_t* accept,
                       double* elev, double* alt, int device) {
  if (!cand || K < 1 || !trans_table || n < 1 || !obs_itrs || !T || !accept) return SSA_EINVAL;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { snprintf(g_err, sizeof(g_err), "no CUDA device"); return SSA_ENODEV; }
  CK(cudaSetDevice(device));
  const size_t KN = (size_t)K * n;
  double *d_c = nullptr, *d_t = nullptr, *d_e = nullptr, *d_a = nullptr;
  uint8_t *d_f = nullptr, *d_acc = nullptr;
  int rc = SSA_OK;
  cudaError_t e;
#define OG(call) do { if ((e = (call)) != cudaSuccess) { rc = set_err(#call, e); goto done; } } while (0)
  OG(cudaMalloc(&d_c, sizeof(double) * 6 * K));
  OG(cudaMalloc(&d_t, sizeof(double) * 9 * n));
  OG(cudaMalloc(&d_f, KN));
  OG(cudaMalloc(&d_acc, K));
  if (elev) OG(cudaMalloc(&d_e, sizeof(double) * KN));
  if (alt) OG(cudaMalloc(&d_a, sizeof(double) * KN));
  OG(cudaMemcpy(d_c, cand, sizeof(double) * 6 * K, cudaMemcpyHostToDevice));
  OG(cudaMemcpy(d_t, trans_table, sizeof(double) * 9 * n, cudaMemcpyHostToDevice));
  {
    ssa_obs ob;
    memset(&ob, 0, sizeof(ob));
    memcpy(ob.obs_itrs, obs_itrs, sizeof(ob.obs_itrs));
    memcpy(ob.T, T, sizeof(ob.T));
    ssa_orbit_eval_kernel<<<(unsigned)((KN + 127) / 128), 128>>>(d_c, K, d_t, n, step_s, ob, obs_limit, min_alt, d_f, d_e, d_a);
    ssa_orbit_accept_kernel<<<(unsigned)((K + 127) / 128), 128>>>(d_f, K, n, first_window, max_gap, d_acc);
  }
  OG(cudaGetLastError());
  OG(cudaMemcpy(accept, d_acc, K, cudaMemcpyDeviceToHost));
  if (elev) OG(cudaMemcpy(elev, d_e, sizeof(double) * KN, cudaMemcpyDeviceToHost));
  if (alt) OG(cudaMemcpy(alt, d_a, sizeof(double) * KN, cudaMemcpyDeviceToHost));
#undef OG
done:
  cudaFree(d_c); cudaFree(d_t); cudaFree(d_f); cudaFree(d_acc); cudaFree(d_e); cudaFree(d_a);
  return rc;
}

int ssa_innovation_stats(const double* y, const uint8_t* valid, int n_series, int n, int nlags, double* dw, double* acf, int device) {
  if (!y || !valid || n_series < 1 || n < 2 || nlags < 0 || nlags >= n || !dw || !acf) return SSA_EINVAL;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { snprintf(g_err, sizeof(g_err), "no CUDA device"); return SSA_ENODEV; }
  CK(cudaSetDevice(device));
  const size_t ny = (size_t)n_series * n * 3, nb = (size_t)n_series * 3;
  double *d_y = nullptr, *d_dw = nullptr, *d_acf = nullptr, *d_w = nullptr;
  uint8_t* d_v = nullptr;
  int rc = SSA_OK;
  cudaError_t e;
#define IS(call) do { if ((e = (call)) != cudaSuccess) { rc = set_err(#call, e); goto done; } } while (0)
  IS(cudaMalloc(&d_y, sizeof(double) * ny));
  IS(cudaMalloc(&d_v, (size_t)n_series * n));
  IS(cudaMalloc(&d_dw, sizeof(double) * nb));
  IS(cudaMalloc(&d_acf, sizeof(double) * nb * (nlags + 1)));
  IS(cudaMalloc(&d_w, sizeof(double) * nb * n));
  IS(cudaMemcpy(d_y, y, sizeof(double) * ny, cudaMemcpyHostToDevice));
  IS(cudaMemcpy(d_v, valid, (size_t)n_series * n, cudaMemcpyHostToDevice));
  ssa_innov_stats_kernel<<<(unsigned)nb, 64>>>(d_y, d_v, n, nlags, d_dw, d_acf, d_w);
  IS(cudaGetLastError());
  IS(cudaMemcpy(dw, d_dw, sizeof(double) * nb, cudaMemcpyDeviceToHost));
  IS(cudaMemcpy(acf, d_acf, sizeof(double) * nb * (nlags + 1), cudaMemcpyDeviceToHost));
#undef IS
done:
  cudaFree(d_y); cudaFree(d_v); cudaFree(d_dw); cudaFree(d_acf); cudaFree(d_w);
  return rc;
}

int ssa_ukf_scores(ssa_ukf* h, void* stream) {
  if (!h) return SSA_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(h->device));
  const int N = h->cfg.n_objects;
  ssa_scores_kernel<<<(unsigned)((N + 127) / 128), 128, 0, st>>>(h->P, h->dpos, h->scores, h->ld, N, h->cfg.dt);
  h->launches++;
  CK(cudaGetLastError());
  return SSA_OK;
}

int ssa_ukf_sync(ssa_ukf* h, void* stream) {
  if (!h) return SSA_EINVAL;
  CK(cudaSetDevice(h->device));
  CK(cudaStreamSynchronize((cudaStream_t)stream));
  return SSA_OK;
}

int ssa_ukf_fp64_peak(int device, void* stream, double* tflops) {
  if (!tflops) return SSA_EINVAL;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { snprintf(g_err, sizeof(g_err), "no CUDA device"); return SSA_ENODEV; }
  CK(cudaSetDevice(device));
  cudaStream_t st = (cudaStream_t)stream;
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 4096;
  double* out;
  CK(cudaMalloc(&out, sizeof(double) * blocks * threads));
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0));
  CK(cudaEventCreate(&e1));
  ssa_dfma_peak_kernel<<<blocks, threads, 0, st>>>(out, iters, 0.999999, 1e-9);  // warm-up
  float best = 1e30f;
  for (int r = 0; r < 5; ++r) {
    CK(cudaEventRecord(e0, st));
    ssa_dfma_peak_kernel<<<blocks, threads, 0, st>>>(out, iters, 0.999999, 1e-9);
    CK(cudaEventRecord(e1, st));
    CK(cudaEventSynchronize(e1));
    float ms;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    if (ms < best) best = ms;
  }
  CK(cudaGetLastError());
  const double flop = 2.0 * 8.0 * (double)iters * (double)blocks * (double)threads;
  *tflops = flop / (best * 1e-3) / 1e12;
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(out);
  return SSA_OK;
}

// ---- unit entry points (host buffers in, host buffers out; synchronous) ------------------------------
static int unit_alloc(const void* host, size_t bytes, void** d) {
  CK(cudaMalloc(d, bytes ? bytes : 8));
  if (host) CK(cudaMemcpy(*d, host, bytes, cudaMemcpyHostToDevice));
  return SSA_OK;
}
#define UNIT_BEGIN(device)                                                                                  \
  int ndev_ = 0;                                                                                            \
  if (cudaGetDeviceCount(&ndev_) != cudaSuccess || ndev_ == 0) {                                            \
    snprintf(g_err, sizeof(g_err), "no CUDA device: libssa_ukf has no CPU fallback");                       \
    return SSA_ENODEV;                                                                                      \
  }                                                                                                         \
  CK(cudaSetDevice(device));

int ssa_unit_math(int op, const double* a, const double* b, double* out, int n, int device) {
  UNIT_BEGIN(device)
  double *da = nullptr, *db = nullptr, *dout = nullptr;
  int rc;
  if ((rc = unit_alloc(a, sizeof(double) * n, (void**)&da))) return rc;
  if (b && (rc = unit_alloc(b, sizeof(double) * n, (void**)&db))) return rc;
  if ((rc = unit_alloc(nullptr, sizeof(double) * n, (void**)&dout))) return rc;
  ssa_unit_math_kernel<<<(n + 127) / 128, 128>>>(op, da, db, dout, n);
  CK(cudaGetLastError());
  CK(cudaMemcpy(out, dout, sizeof(double) * n, cudaMemcpyDeviceToHost));
  cudaFree(da); cudaFree(db); cudaFree(dout);
  return SSA_OK;
}
int ssa_unit_fx(const double* x, double dt, double* out, int32_t* exc, int n, int device) {
  UNIT_BEGIN(device)
  double *dx = nullptr, *dout = nullptr; int32_t* dexc = nullptr;
  int rc;
  if ((rc = unit_alloc(x, sizeof(double) * 6 * n, (void**)&dx))) return rc;
  if ((rc = unit_alloc(nullptr, sizeof(double) * 6 * n, (void**)&dout))) return rc;
  if ((rc = unit_alloc(nullptr, sizeof(int32_t) * n, (void**)&dexc))) return rc;
  ssa_unit_fx_kernel<<<(n + 127) / 128, 128>>>(dx, dt, dout, dexc, n);
  CK(cudaGetLastError());
  CK(cudaMemcpy(out, dout, sizeof(double) * 6 * n, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(exc, dexc, sizeof(int32_t) * n, cudaMemcpyDeviceToHost));
  cudaFree(dx); cudaFree(dout); cudaFree(dexc);
  return SSA_OK;
}
int ssa_unit_hx_aer(const double* x, int stride, const double M[9], const double obs_itrs[3], const double T[9],
                    double* out, int n, int device) {
  UNIT_BEGIN(device)
  ssa_obs ob;
  memcpy(ob.M, M, sizeof(ob.M)); memcpy(ob.obs_itrs, obs_itrs, sizeof(ob.obs_itrs)); memcpy(ob.T, T, sizeof(ob.T));
  double *dx = nullptr, *dout = nullptr;
  int rc;
  if ((rc = unit_alloc(x, sizeof(double) * stride * n, (void**)&dx))) return rc;
  if ((rc = unit_alloc(nullptr, sizeof(double) * 3 * n, (void**)&dout))) return rc;
  ssa_unit_hx_kernel<<<(n + 127) / 128, 128>>>(dx, ob, dout, n, stride);
  CK(cudaGetLastError());
  CK(cudaMemcpy(out, dout, sizeof(double) * 3 * n, cudaMemcpyDeviceToHost));
  cudaFree(dx); cudaFree(dout);
  return SSA_OK;
}
int ssa_unit_aer(int op, const double* a, const double* b, double* out, int n, int device) {
  UNIT_BEGIN(device)
  double *da = nullptr, *db = nullptr, *dout = nullptr;
  int rc;
  if ((rc = unit_alloc(a, sizeof(double) * 3 * n, (void**)&da))) return rc;
  if (b && (rc = unit_alloc(b, sizeof(double) * 3 * n, (void**)&db))) return rc;
  if ((rc = unit_alloc(nullptr, sizeof(double) * 3 * n, (void**)&dout))) return rc;
  ssa_unit_aer_kernel<<<(n + 127) / 128, 128>>>(op, da, db, dout, n);
  CK(cudaGetLastError());
  CK(cudaMemcpy(out, dout, sizeof(double) * 3 * n, cudaMemcpyDeviceToHost));
  cudaFree(da); cudaFree(db); cudaFree(dout);
  return SSA_OK;
}
int ssa_unit_robust_chol(const double* P_packed, double lam, double* U_packed, int32_t* ret, int n, int device) {
  UNIT_BEGIN(device)
  double *dp = nullptr, *du = nullptr; int32_t* dr = nullptr;
  int rc;
  if ((rc = unit_alloc(P_packed, sizeof(double) * 21 * n, (void**)&dp))) return rc;
  if ((rc = unit_alloc(nullptr, sizeof(double) * 21 * n, (void**)&du))) return rc;
  if ((rc = unit_alloc(nullptr, sizeof(int32_t) * n, (void**)&dr))) return rc;
  ssa_unit_chol_kernel<<<(n + 127) / 128, 128>>>(dp, lam, du, dr, n);
  CK(cudaGetLastError());
  CK(cudaMemcpy(U_packed, du, sizeof(double) * 21 * n, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(ret, dr, sizeof(int32_t) * n, cudaMemcpyDeviceToHost));
  cudaFree(dp); cudaFree(du); cudaFree(dr);
  return SSA_OK;
}
int ssa_unit_inv3(const double* S, double* SI, int32_t* ok, int n, int device) {
  UNIT_BEGIN(device)
  double *ds = nullptr, *di = nullptr; int32_t* dk = nullptr;
  int rc;
  if ((rc = unit_alloc(S, sizeof(double) * 9 * n, (void**)&ds))) return rc;
  if ((rc = unit_alloc(nullptr, sizeof(double) * 9 * n, (void**)&di))) return rc;
  if ((rc = unit_alloc(nullptr, sizeof(int32_t) * n, (void**)&dk))) return rc;
  ssa_unit_inv3_kernel<<<(n + 127) / 128, 128>>>(ds, di, dk, n);
  CK(cudaGetLastError());
  CK(cudaMemcpy(SI, di, sizeof(double) * 9 * n, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(ok, dk, sizeof(int32_t) * n, cudaMemcpyDeviceToHost));
  cudaFree(ds); cudaFree(di); cudaFree(dk);
  return SSA_OK;
}

}  // extern "C"
