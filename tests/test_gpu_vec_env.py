"""-m gpu: BASELINE.json config 3 — E parallel environments advanced by one device step must reproduce E
independent single environments (same seeds): observations, rewards, dones, auto-resets and the device-side
greedy tasker decisions, all EXACT (the single envs run on the host twin of the same arithmetic)."""
import numpy as np
import pytest

import helpers as H
import ssa_gym_b200
from ssa_gym_b200 import _lib as F
from ssa_gym_b200 import agents
from ssa_gym_b200.transformations import gcrs2irts_matrix_approx, time_table
from ssa_gym_b200.vec_env import VecSSATaskerEnv
from test_gpu_env import make_env

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("over,tasker,agent", [
    ({"steps": 40, "reward_type": "jones"}, F.TASKER_VISIBLE_GREEDY, agents.agent_visible_greedy),
    ({"steps": 30, "reward_type": "trinary", "obs_limit": 15}, F.TASKER_POS_ERROR_GREEDY, agents.agent_pos_error_greedy),
    ({"steps": 25, "reward_type": "shaped", "rso_count": 6}, F.TASKER_NAIVE_GREEDY, agents.agent_naive_greedy),
    # the other two observation layouts of SS2:164-177 / 355-361
    ({"steps": 20, "reward_type": "jones", "rso_count": 7, "obs_returned": "aer"}, F.TASKER_VISIBLE_GREEDY, agents.agent_visible_greedy),
    ({"steps": 20, "reward_type": "trinary", "rso_count": 5, "obs_returned": "2d"}, F.TASKER_NAIVE_GREEDY, agents.agent_naive_greedy),
    # agent_shannon: log-determinant ratios of consecutive steps (np.linalg.det here, ssa_det6_sym on the device)
    ({"steps": 30, "reward_type": "jones", "obs_limit": 10}, F.TASKER_SHANNON, agents.agent_shannon),
])
def test_vec_env_equals_independent_envs(over, tasker, agent):
    E, total_steps = 24, 55
    cfg = dict(ssa_gym_b200.env_config)
    cfg.update(over)
    cfg["trans_matrix"] = gcrs2irts_matrix_approx(time_table(cfg["t_0"], cfg["time_step"], cfg["steps"]))
    seeds = list(range(100, 100 + E))
    vec = VecSSATaskerEnv(cfg, E, seeds=seeds)
    singles = []
    for e in range(E):
        env = make_env("twin", **{k: v for k, v in cfg.items()})
        env.seed(seeds[e]); env.action_space.seed(seeds[e]); vec.action_spaces[e].seed(seeds[e])
        singles.append(env)
    vec.seed(seeds)
    obs_v = vec.vector_reset()
    obs_s = [env.reset() for env in singles]
    assert all(H.bits_equal(obs_v[e], obs_s[e]) for e in range(E))
    n_resets = ties = 0
    for t in range(total_steps):
        a_v = vec.greedy_actions(tasker)
        a_s = [int(agent(obs_s[e], singles[e])) for e in range(E)]
        for e in np.where(np.asarray(a_v) != a_s)[0]:
            assert tasker == F.TASKER_SHANNON and _shannon_tie(singles[e], a_v[e], a_s[e]), (t, e, a_v[e], a_s[e])
            ties += 1
            a_v[e] = a_s[e]  # both sides go on with the same action
        assert list(a_v) == a_s, (t, list(a_v), a_s)                                  # tasking: bit-exact
        obs_v, r_v, d_v, _ = vec.vector_step(a_v)
        for e, env in enumerate(singles):
            o, r, d, _ = env.step(a_s[e])
            assert H.bits_equal(np.float64(r), np.float64(r_v[e])) and bool(d) == bool(d_v[e]), (t, e, r, r_v[e], d, d_v[e])
            if d:
                o = env.reset()
                n_resets += 1
            obs_s[e] = o
            assert H.bits_equal(obs_v[e], np.asarray(o)), (t, e)
    assert n_resets >= E  # every env went through at least one auto-reset
    assert ties <= 2, ties  # none seen; a tie of two log-determinant ratios within 1e-12 is a rare event
    vec.close()


def _shannon_tie(env, a, b):
    """The only allowed difference between the device's and the reference's agent_shannon pick: the two objects' EXACT
    determinant ratios det P_i / det P_{i-1} (every double is an exact rational) agree to 1e-12 relative, inside the
    rounding of the determinants (tests/test_det_exact.py: up to 1e-12 apart on these covariances)."""
    if env.i == 0:
        return False
    r = []
    for j in (a, b):
        now, before = H.exact_det(env.P_filter[env.i][j]), H.exact_det(env.P_filter[env.i - 1][j])
        if now == 0 or before == 0:
            return False
        r.append(now / before)
    return abs(float((r[0] - r[1]) / r[1])) <= 1e-12


# ---- device-resident episodic mode (rng='device'): vectorised reset + counter-based noise --------------------------
@pytest.mark.parametrize("over", [{"steps": 14, "reward_type": "jones", "update_interval": 1},
                                  {"steps": 9, "reward_type": "trinary", "update_interval": 2, "obs_limit": 10},
                                  # m > 64: the per-environment reductions (step and refresh) run CTA-wide instead of per warp
                                  {"steps": 7, "reward_type": "trinary", "update_interval": 1, "rso_count": 70}])
def test_device_episodic_mode_equals_twin_emulation(over):
    """ssa_ukf_rollout_reset / ssa_ukf_rollout_step (one graph launch per step: noise, UKF kernels, reward / done,
    auto-reset, fresh obs, greedy taskers) against a step-by-step emulation built from the host twin
    (helpers.EpisodicTwin: the same counter-based draws, twin_step with the per-env trans_matrix, numpy reward / done /
    taskers, agent_shannon's determinant history).  Observations, rewards, dones and all six tasker decisions must be
    EXACT over many auto-resets; the launch paths are in tests/test_gpu_env_reduce_paths.py."""
    cfg = dict(ssa_gym_b200.env_config)
    cfg.update(over)
    cfg["trans_matrix"] = gcrs2irts_matrix_approx(time_table(cfg["t_0"], cfg["time_step"], cfg["steps"]))
    seen = H.episodic_vs_twin(cfg, 48, 40)
    assert seen["resets"] >= 48


def test_device_resident_step_equals_host_io_step():
    """vector_step_device (actions read from the device buffer, obs / reward / done / greedy left on the device, no copies,
    no synchronisation) is the same step as vector_step: every output bit-equal over auto-resets."""
    import torch
    E = 64
    cfg = dict(ssa_gym_b200.env_config, steps=12)
    cfg["trans_matrix"] = gcrs2irts_matrix_approx(time_table(cfg["t_0"], cfg["time_step"], cfg["steps"]))
    seeds = list(range(900, 900 + E))
    a_env = VecSSATaskerEnv(cfg, E, seeds=seeds, rng="device")
    b_env = VecSSATaskerEnv(cfg, E, seeds=seeds, rng="device")
    v = b_env.device_views()
    assert np.array_equal(v["obs"].cpu().numpy(), a_env.obs)
    rng = np.random.RandomState(4)
    n_done = 0
    for t in range(30):
        act = rng.randint(0, cfg["rso_count"], size=E).astype(np.int32)
        obs, rew, done, _ = a_env.vector_step(act)
        v["actions"].copy_(torch.from_numpy(act).to(v["actions"].device))
        b_env.vector_step_device()
        torch.cuda.synchronize()
        assert H.bits_equal(v["obs"].cpu().numpy(), obs) and H.bits_equal(v["reward"].cpu().numpy(), rew)
        assert np.array_equal(v["done"].cpu().numpy().astype(bool), done)
        assert np.array_equal(v["greedy"].cpu().numpy(), a_env._io["greedy"])
        n_done += int(done.sum())
    assert n_done > E
    a_env.close(); b_env.close()


@pytest.mark.parametrize("layout", ["flatten", "2d"])
def test_float32_observations_are_the_rounded_float64_ones(layout):
    """obs_dtype='float32' (SSA_ROLLOUT_OBS_F32): the step's observations leave the device as floats — the float64 rows
    rounded to nearest, bit for bit numpy's astype(float32) — and reward / done / greedy are untouched, over auto-resets."""
    E = 48
    cfg = dict(ssa_gym_b200.env_config, steps=10, obs_returned=layout)
    cfg["trans_matrix"] = gcrs2irts_matrix_approx(time_table(cfg["t_0"], cfg["time_step"], cfg["steps"]))
    seeds = list(range(300, 300 + E))
    a_env = VecSSATaskerEnv(cfg, E, seeds=seeds, rng="device")
    b_env = VecSSATaskerEnv(dict(cfg, obs_dtype="float32"), E, seeds=seeds, rng="device")
    assert b_env.observation_space.dtype == np.float32 and a_env.observation_space.dtype == np.float64
    o64, o32 = a_env.vector_reset(), b_env.vector_reset()
    assert o32.dtype == np.float32 and np.array_equal(o32, o64.astype(np.float32))
    rng = np.random.RandomState(5)
    n_done = 0
    for t in range(25):
        act = rng.randint(0, cfg["rso_count"], size=E).astype(np.int32)
        o64, r64, d64, _ = a_env.vector_step(act)
        o32, r32, d32, _ = b_env.vector_step(act)
        assert o32.dtype == np.float32 and o32.shape == o64.shape
        assert np.array_equal(o32.view(np.uint32), o64.astype(np.float32).view(np.uint32))
        assert H.bits_equal(r32, r64) and np.array_equal(d32, d64)
        assert np.array_equal(a_env._io["greedy"], b_env._io["greedy"])
        n_done += int(d64.sum())
    assert n_done > E
    a_env.close(); b_env.close()
    with pytest.raises(ValueError):
        VecSSATaskerEnv(dict(cfg, obs_dtype="float32", obs_returned="aer"), 4, rng="device")
    with pytest.raises(ValueError):
        VecSSATaskerEnv(dict(cfg, obs_dtype="float32"), 4, rng="host")
