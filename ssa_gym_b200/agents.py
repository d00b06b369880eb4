"""Heuristic tasking agents: the reference's names and call signature `agent(obs, env)` (agents.py:7-81), written
as one selection rule with different scores.

Every agent of the reference is "among the candidate objects, task the one with the largest score; if there is no
candidate, sample the action space".  The candidates are all objects (naive) or `env.visible_objects()`; the scores
are trace(P), the tracking errors, the last column of the 'aer' observation or the log-determinant ratio.  Three
numpy conventions decide ties and corner cases and are kept on purpose, because the tasking decisions are integer
work that has to match exactly:
  * trace(P) is `np.trace` of each 6x6 (diagonal summed left to right);
  * `np.argmax` returns the FIRST maximum;
  * "no candidate" is tested as `not np.any(indices)` (agents.py:37) - the INDEX array, so the case "only object 0
    is visible" also counts as empty and a random action is sampled.
The arrays read here (`env.P_filter[env.i]`, `env.delta_pos`, ...) were produced by the GPU step.  For vectorised
environments the argmax rules run on the device (`ssa_ukf_env_reduce`, SSA_TASKER_*), see vec_env.py; there
agent_shannon's P_{i-1} is the covariance of the previous step index the reduction ran at, and a fresh episode (step 0)
gets ratio 1 everywhere, as the reference's zeroed history row gives equal ratios.
In the device-resident episodic mode all nine agents, the random ones included, also run inside the step graph
(`VecSSATaskerEnv.set_tasker`, ssa_ukf_rollout_tasker): the device draws `action_space.sample()` and
`np.random.choice` from counter-based Philox streams instead (same distributions, other streams; csrc/ssa_rng.h,
ssa_tasker_pick).
"""
import numpy as np


def _candidates(env):
    """Indices of the visible objects, or None where the reference falls back to a random action."""
    idx = env.visible_objects()
    return idx if np.any(idx) else None


def _traces(covariances):
    return [np.trace(P) for P in covariances]


def _task_best(env, score):
    """score(idx) -> one value per candidate; the first maximum is tasked."""
    idx = _candidates(env)
    if idx is None:
        return env.action_space.sample()
    return idx[np.argmax(score(idx))]


# -- uninformed ------------------------------------------------------------------------------------------------------
def agent_naive_random(obs=None, env=None):
    return env.action_space.sample()


def agent_naive_greedy(obs, env=None):
    return np.argmax(_traces(env.P_filter[env.i]))          # every object is a candidate, visible or not


def agent_visible_random(obs, env):
    idx = _candidates(env)
    return env.action_space.sample() if idx is None else np.random.choice(idx)


# -- largest score among the visible objects -------------------------------------------------------------------------
def agent_visible_greedy(obs, env):
    return _task_best(env, lambda idx: _traces(env.P_filter[env.i][idx]))


def agent_pos_error_greedy(obs, env):
    return _task_best(env, lambda idx: env.delta_pos[env.i, idx])


def agent_vel_error_greedy(obs, env):
    return _task_best(env, lambda idx: env.delta_vel[env.i, idx])


def agent_visible_greedy_aer(obs, env):
    # 'aer' observations are [az, el, range, trace P] per object (SS2:834-840)
    return _task_best(env, lambda idx: obs.reshape(len(obs) // 4, 4)[idx, 3])


def agent_shannon(obs, env):
    def log_det_ratio(idx):
        now, before = env.P_filter[env.i][idx], env.P_filter[env.i - 1][idx]
        with np.errstate(divide='ignore', invalid='ignore'):
            return [np.log(np.linalg.det(a) / np.linalg.det(b)) for a, b in zip(now, before)]
    return _task_best(env, log_det_ratio)


def agent_visible_greedy_spoiled(obs, env, p=0.25):
    """visible-greedy, replaced by a random action with probability p.  The random action is drawn first, whether it
    is used or not (the reference consumes the action-space generator on every call)."""
    fallback = env.action_space.sample()
    idx = _candidates(env)
    if idx is None:
        return fallback
    greedy = idx[np.argmax(_traces(env.P_filter[env.i][idx]))]
    return np.random.choice(a=[greedy, fallback], p=[1 - p, p])
