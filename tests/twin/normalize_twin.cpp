// normalize_twin.cpp — HOST build of the running normalization of the episodic mode (ssa_norm_* in
// ssa_gym_b200/csrc/ssa_ukf_core.h, run on the device by k_normalize), for tests only.  Built with the host twin's flags
// (contraction off, explicit FMAs) into a temporary directory by tests/test_normalize_host.py; the product never links
// or loads it.
#include <stddef.h>
#include <stdint.h>

#include <vector>

#include "../../include/ssa_ukf.h"
#include "../../ssa_gym_b200/csrc/ssa_math.h"
#include "../../ssa_gym_b200/csrc/ssa_ukf_core.h"

extern "C" {

// the pieces, one call each (n values element-wise where a count is given)
void twin_norm_moments(const double* x, long stride, int E, int f32, double* mean, double* var) {
  std::vector<double> buf(ssa_norm_leaves(E));
  ssa_norm_moments(x, stride, E, f32, buf.data(), mean, var);
}
void twin_norm_merge(double* mean, double* var, double* count, double bmean, double bvar, double bcount) {
  ssa_norm_merge(mean, var, count, bmean, bvar, bcount);
}
void twin_norm_obs(int n, const double* v, const double* mean, const double* var, double eps, double clip, double* out) {
  for (int i = 0; i < n; ++i) out[i] = ssa_norm_obs(v[i], mean[i], ssa_norm_sd(var[i], eps), clip);
}
void twin_norm_reward(int n, const double* r, double var, double eps, double clip, double* out) {
  for (int i = 0; i < n; ++i) out[i] = ssa_norm_reward(r[i], ssa_norm_sd(var, eps), clip);
}
void twin_norm_return(int n, const double* ret, double gamma, const double* r, int nan_to_num, double* out) {
  for (int i = 0; i < n; ++i) out[i] = ssa_norm_return(ret[i], gamma, ssa_norm_reward_in(r[i], nan_to_num));
}

// One k_normalize of E environments of F columns.  mode 0: a step, 1: ssa_ukf_rollout_reset, 2: reset_envs of the
// environments with done[e] set.  obs / term: rows [E][F] (term null: no auto-reset), reward / done [E], state in the
// saved layout of ssa_ukf_rollout_norm_state_download (2 F + 4 + E doubles), outputs [E][F] / [E].
void twin_normalize(int mode, int E, int F, const double* obs, int f32, const double* term, const uint8_t* done,
                    const double* reward, int training, int norm_obs, int norm_reward, int reward_nan, double clip_obs,
                    double clip_reward, double gamma, double eps, double* state, float* out, float* term_out,
                    double* reward_out) {
  double *mean = state, *var = state + F, *cnt = state + 2 * F, *rs = state + 2 * F + 1, *ret = state + 2 * F + 4;
  std::vector<double> buf(ssa_norm_leaves(E));
  if (mode != 2 && training && norm_obs) {
    double n_new = *cnt;
    for (int c = 0; c < F; ++c) {
      double bm, bv, n = *cnt;
      ssa_norm_moments(obs + c, F, E, f32, buf.data(), &bm, &bv);
      ssa_norm_merge(mean + c, var + c, &n, bm, bv, (double)E);
      n_new = n;
    }
    *cnt = n_new;
  }
  for (int e = 0; e < E; ++e) {
    if (mode == 2 && !done[e]) continue;
    for (int c = 0; c < F; ++c) {
      const size_t i = (size_t)e * F + c;
      const double v = ssa_norm_in(obs[i], f32);
      out[i] = (float)(norm_obs ? ssa_norm_obs(v, mean[c], ssa_norm_sd(var[c], eps), clip_obs) : v);
      if (mode == 0 && term && done[e]) {
        const double t = ssa_norm_in(term[i], f32);
        term_out[i] = (float)(norm_obs ? ssa_norm_obs(t, mean[c], ssa_norm_sd(var[c], eps), clip_obs) : t);
      }
    }
  }
  if (mode != 0) {
    for (int e = 0; e < E; ++e)
      if (mode == 1 || done[e]) ret[e] = 0.0;
    return;
  }
  if (training) {
    for (int e = 0; e < E; ++e) ret[e] = ssa_norm_return(ret[e], gamma, ssa_norm_reward_in(reward[e], reward_nan));
    double bm, bv;
    ssa_norm_moments(ret, 1, E, 0, buf.data(), &bm, &bv);
    ssa_norm_merge(rs, rs + 1, rs + 2, bm, bv, (double)E);
  }
  for (int e = 0; e < E; ++e) {
    const double r = ssa_norm_reward_in(reward[e], reward_nan);
    reward_out[e] = norm_reward ? ssa_norm_reward(r, ssa_norm_sd(rs[1], eps), clip_reward) : r;
    if (done[e]) ret[e] = 0.0;
  }
}

}  // extern "C"
