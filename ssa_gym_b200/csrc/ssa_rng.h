// Counter-based random numbers for the device-resident episodic mode (SURVEY 8f-2: vectorised reset).
//
// The reference draws every episode from one sequential MT19937 stream per environment (SS2:206-221:
// m x [randint, normal(6)] then normal(n*m*3)), 14 400+ normals per reset on one host thread.  A sequential
// stream cannot be drawn in parallel, so this mode replaces it by Philox4x32-10 (Salmon et al., SC'11) keyed by
// the environment's seed and addressed by (episode, stream, object, step): any draw of any environment can be
// computed by any thread, at reset time or on the fly, and nothing is stored.  The distributions are the
// reference's (uniform catalog row, N(0, x_sigma), N(0, z_sigma)); the streams are NOT the reference's (the
// host-RNG mode of VecSSATaskerEnv keeps np_random stream parity).  Shared by the CUDA kernels and the host twin:
// integer arithmetic plus this library's own log / sqrt / sincos, so both produce the same bits.
#ifndef SSA_RNG_H
#define SSA_RNG_H
#include "ssa_math.h"
#include "../../include/ssa_ukf.h"  // SSA_TASKER_*

#define SSA_RNG_STREAM_ORBIT 0u
#define SSA_RNG_STREAM_X 1u
#define SSA_RNG_STREAM_Z 2u
#define SSA_RNG_STREAM_ACT 3u

struct ssa_u4 { uint32_t v[4]; };

SSA_HD uint32_t ssa_mulhi32(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * (uint64_t)b) >> 32); }

// Philox4x32-10: counter c[4], key k[2]
SSA_HD ssa_u4 ssa_philox4x32(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = ssa_mulhi32(M0, c0), lo0 = M0 * c0;
    const uint32_t hi1 = ssa_mulhi32(M1, c2), lo1 = M1 * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += W0; k1 += W1;
  }
  ssa_u4 o;
  o.v[0] = c0; o.v[1] = c1; o.v[2] = c2; o.v[3] = c3;
  return o;
}

// 52-bit uniform in (0, 1): (k + 0.5) / 2^52, exact in fp64 and never 0 or 1, so log() is finite and non-zero
SSA_HD double ssa_u52(uint32_t hi, uint32_t lo) {
  const uint64_t k = (((uint64_t)hi << 32) | (uint64_t)lo) >> 12;
  return ssa_mul((double)k + 0.5, 2.220446049250313e-16);
}

// two independent N(0,1) from one Philox block (Box-Muller)
SSA_HD void ssa_normal2(const ssa_u4& r, double* n0, double* n1) {
  const double u1 = ssa_u52(r.v[0], r.v[1]), u2 = ssa_u52(r.v[2], r.v[3]);
  const double rad = ssa_sqrt(ssa_mul(-2.0, ssa_log(u1)));
  const ssa_sc sc = ssa_sincos_v(ssa_mul(SSA_C(TWOPI), u2));
  *n0 = ssa_mul(rad, sc.c);
  *n1 = ssa_mul(rad, sc.s);
}

// Draws of one object j of environment (key k0,k1) in episode ep.
// catalog row: uniform over [0, n_orbits)
SSA_HD uint32_t ssa_draw_orbit(uint32_t k0, uint32_t k1, uint32_t ep, uint32_t j, uint32_t n_orbits) {
  const ssa_u4 r = ssa_philox4x32(ep, SSA_RNG_STREAM_ORBIT, j, 0u, k0, k1);
  return ssa_mulhi32(r.v[0], n_orbits);
}
// initial filter error: 6 x N(0,1)
SSA_HD void ssa_draw_x(uint32_t k0, uint32_t k1, uint32_t ep, uint32_t j, double* n6) {
#pragma unroll
  for (uint32_t q = 0; q < 3; ++q) {
    const ssa_u4 r = ssa_philox4x32(ep, SSA_RNG_STREAM_X | (q << 8), j, 0u, k0, k1);
    ssa_normal2(r, n6 + 2 * q, n6 + 2 * q + 1);
  }
}
// measurement noise of step i: 3 x N(0,1)
SSA_HD void ssa_draw_z(uint32_t k0, uint32_t k1, uint32_t ep, uint32_t j, uint32_t step, double* n3) {
  double a, b, c, d;
  ssa_normal2(ssa_philox4x32(ep, SSA_RNG_STREAM_Z, j, step, k0, k1), &a, &b);
  ssa_normal2(ssa_philox4x32(ep, SSA_RNG_STREAM_Z | (1u << 8), j, step, k0, k1), &c, &d);
  (void)d;
  n3[0] = a; n3[1] = b; n3[2] = c;
}

// The action a device tasker (ssa_ukf_rollout_tasker) takes in environment (k0,k1), episode ep, for step `step`, from
// the state the previous step left: greedy = the environment's row of the greedy block, vis = its m visibility flags.
// One Philox block: v0 is action_space.sample() (uniform over m), v1 the choice among the visible objects, v2:v3 the
// spoiled agent's uniform.  The candidates are empty where agents.py:37 `not np.any(idx)` holds: nothing visible, or
// only object 0.  tasker: 0 .. SSA_TASKER_VISIBLE_GREEDY_SPOILED.
SSA_HD int ssa_tasker_pick(uint32_t k0, uint32_t k1, uint32_t ep, uint32_t step, int m, int tasker, const int32_t* greedy,
                           const uint8_t* vis, double spoil_p) {
  const ssa_u4 r = ssa_philox4x32(ep, SSA_RNG_STREAM_ACT, 0u, step, k0, k1);
  const int fallback = (int)ssa_mulhi32(r.v[0], (uint32_t)m);
  if (tasker < SSA_N_TASKERS) return greedy[tasker] >= 0 ? greedy[tasker] : fallback;
  if (tasker == SSA_TASKER_NAIVE_RANDOM) return fallback;
  uint32_t n_vis = 0;
  int any = 0;
  for (int j = 0; j < m; ++j)
    if (vis[j]) { n_vis += 1; any |= (j != 0); }
  if (!any) return fallback;
  if (tasker == SSA_TASKER_VISIBLE_RANDOM) {  // np.random.choice(idx): the k-th visible index in increasing order
    uint32_t k = ssa_mulhi32(r.v[1], n_vis);
    int j = 0;
    for (;; ++j)
      if (vis[j] && k-- == 0) break;
    return j;
  }
  // SSA_TASKER_VISIBLE_GREEDY_SPOILED: np.random.choice([greedy, fallback], p=[1 - p, p]) is searchsorted(cdf, u,
  // side='right'): the greedy pick for u < 1 - p
  return ssa_u52(r.v[2], r.v[3]) < 1.0 - spoil_p ? greedy[SSA_TASKER_VISIBLE_GREEDY] : fallback;
}

#endif  // SSA_RNG_H
