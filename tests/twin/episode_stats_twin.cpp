// episode_stats_twin.cpp — HOST build of the per-episode statistics of the episodic mode (ssa_ep_* in
// ssa_gym_b200/csrc/ssa_ukf_core.h, run on the device by k_ep_row0 / k_ep_step), for tests only.  Built with the host
// twin's flags (contraction off, explicit FMAs) into a temporary directory by tests/test_episode_stats_host.py; the
// product never links or loads it.
#include <stddef.h>
#include <stdint.h>

#include "../../include/ssa_ukf.h"
#include "../../ssa_gym_b200/csrc/ssa_math.h"
#include "../../ssa_gym_b200/csrc/ssa_ukf_core.h"

extern "C" {

// ---- episodic device mode: per-episode statistics (k_ep_row0 / k_ep_step) ------------------------------------------
// host layouts: x_true / x [N][6], P packed [N][21], y [N][3], S [N][9]; accumulators obj [N][SSA_EPO], env
// [E][SSA_EPE], records [E][SSA_EPR]
// row 0 of the environments whose step index is 0 (the head of an episodic step)
void twin_episode_stats_row0(int E, int m, const int32_t* step_idx, const double* x_true, const double* x, const double* P,
                             double* obj) {
  for (int e = 0; e < E; ++e) {
    if (step_idx[e] != 0) continue;
    for (int j = 0; j < m; ++j) {
      const size_t n = (size_t)e * m + j;
      ssa_ep_nees_row(obj + n * SSA_EPO, x_true + n * 6, x + n * 6, 1, P + n * SSA_NP, 1);
    }
  }
}
// the rest of a step, after the reward / done reduction: step_idx is the step just taken, act_eff the effective action
// (-1 on steps update_interval skips); finished environments get their record and, with auto_reset, cleared accumulators
void twin_episode_stats_step(int E, int m, const int32_t* step_idx, const double* x_true, const double* x, const double* P,
                             const int32_t* act_eff, const uint8_t* updated, const double* y, const double* S,
                             const double* reward, const uint8_t* done, const int32_t* status, int auto_reset, double* obj,
                             double* env, double* rec) {
  for (int e = 0; e < E; ++e) {
    const size_t b = (size_t)e * m;
    for (int j = 0; j < m; ++j)
      ssa_ep_nees_row(obj + (b + j) * SSA_EPO, x_true + (b + j) * 6, x + (b + j) * 6, 1, P + (b + j) * SSA_NP, 1);
    double* ea = env + (size_t)e * SSA_EPE;
    const int a = act_eff[e];
    if (a >= 0 && a < m && updated[b + a]) ssa_ep_observe(ea, obj + (b + a) * SSA_EPO, y + (b + a) * 3, S + (b + a) * 9);
    ea[SSA_EPE_RET] = ea[SSA_EPE_RET] + reward[e];
    if (done[e]) {
      ssa_ep_finalise(ea, obj + b * SSA_EPO, status + b, m, (double)step_idx[e], rec + (size_t)e * SSA_EPR);
      if (auto_reset) ssa_ep_clear(ea, obj + b * SSA_EPO, m);
    }
  }
}

}  // extern "C"
