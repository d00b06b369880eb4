"""-m gpu: running normalization of observations and returns in the device-resident episodic mode
(VecSSATaskerEnv(config | {'normalize': ...}, rng='device'), k_normalize), EXACT against the host build of the same
arithmetic (test_normalize_host.TwinNormalize, tests/twin/normalize_twin.cpp) applied to the raw stream of a
normalization-off environment with the same seeds and actions, on every launch path.

Every step checks: the raw stream (get_original_obs / get_original_reward, done, greedy, truncated, episode records)
bit-equal to the switch-off environment's; the normalized obs, rewards and final observations (infos and device views)
and the saved state bit-equal to the twin's.  The batch moments of the first reset are also checked against numpy's
within the CPU test's bound."""
import ctypes

import numpy as np
import pytest

import helpers as H
from ssa_gym_b200 import _lib as F
from ssa_gym_b200.ukf import BatchedUKF
from ssa_gym_b200.vec_env import VecSSATaskerEnv
from test_gpu_env_reduce_paths import SWITCHES, _cfg, launch_path  # noqa: F401  (launch_path: fixture)
from test_normalize_host import TwinNormalize, _moment_bound, bits, twin_moments

pytestmark = pytest.mark.gpu
E = 45
PATHS = ["default"] + sorted(SWITCHES)


def _rows(obs):
    return np.asarray(obs).reshape(len(obs), -1)


def _state_vec(d):
    return np.concatenate([d["obs_mean"], d["obs_var"], [d["obs_count"], d["ret_mean"], d["ret_var"], d["ret_count"]], d["returns"]])


def _twin_for(vec, kw):
    return TwinNormalize(vec.E, vec.ukf.norm_F, f32=vec.obs_dtype == np.float32, reward_nan=vec.obs_returned != "flatten",
                         **{k: v for k, v in kw.items()})


def norm_vs_off(cfg, total_steps, kw=None, auto_reset=True, toggle=(), seed0=700, action_seed=5, episode_stats=True, E=E):
    """A normalized environment against a switch-off one and the twin, step by step (see the module docstring).
    toggle: steps at which `training` flips.  Returns (vec, off, twin, counters)."""
    kw = dict(kw or {})
    seeds = list(range(seed0, seed0 + E))
    base = dict(cfg, terminal_observation=True, episode_stats=episode_stats)
    vec = VecSSATaskerEnv(dict(base, normalize=kw or True), E, seeds=seeds, rng="device", auto_reset=auto_reset)
    off = VecSSATaskerEnv(base, E, seeds=seeds, rng="device", auto_reset=auto_reset)
    tw = _twin_for(vec, kw)
    raw0 = _rows(off.obs).astype(np.float64)
    assert bits(_rows(vec.get_original_obs()), _rows(off.obs))
    assert bits(_rows(vec.obs), tw.reset(raw0)) and bits(_state_vec(vec.normalizer_state()), tw.state)
    if not tw.f32:
        _moment_bound(raw0, *twin_moments(raw0))
    views = vec.device_views()
    rng = np.random.RandomState(action_seed)
    seen = {"done": 0, "term": 0}
    for t in range(total_steps):
        if t in toggle:
            vec.training = not vec.training
            tw.training = vec.training
        a = np.asarray(rng.randint(0, cfg["rso_count"], size=E) if t % 2 == 0 else off.greedy_actions(F.TASKER_VISIBLE_GREEDY),
                       dtype=np.int32)
        o_v, r_v, d_v, i_v = vec.vector_step(a)
        o_v, r_v = np.array(o_v, copy=True), np.array(r_v, copy=True)
        o_o, r_o, d_o, i_o = off.vector_step(a)
        # raw stream
        assert bits(_rows(vec.get_original_obs()), _rows(o_o)) and bits(vec.get_original_reward(), r_o), t
        assert np.array_equal(d_v, d_o) and np.array_equal(vec.truncated, off.truncated), t
        assert np.array_equal(vec._io["greedy"], off._io["greedy"]), t
        # normalized stream against the twin over the raw one
        term = np.zeros((E, tw.F))
        de = np.flatnonzero(d_o)
        for e in de:
            if "terminal_observation" in i_o[e]:
                term[e] = np.asarray(i_o[e]["terminal_observation"], np.float64).reshape(-1)
        out, rout = tw.step(_rows(o_o).astype(np.float64), r_o, d_o, term if auto_reset else None)
        assert bits(_rows(o_v), out) and bits(r_v, rout), t
        assert bits(views["obs_norm"].cpu().numpy(), out) and bits(views["reward_norm"].cpu().numpy(), rout), t
        for e in de:
            assert set(i_v[e]) == set(i_o[e]), t
            if episode_stats:  # (the raw return, as Monitor below VecNormalize reports it)
                for k, val in i_o[e]["episode"].items():
                    assert bits(np.asarray(i_v[e]["episode"][k], np.float64), np.asarray(val, np.float64)), (t, k)
            if auto_reset:
                assert bits(np.asarray(i_v[e]["terminal_observation"]).reshape(-1), tw.term[e]), t
                seen["term"] += 1
        if auto_reset and len(de):
            assert bits(views["terminal_obs_norm"].cpu().numpy()[de], tw.term[de]), t
        assert bits(_state_vec(vec.normalizer_state()), tw.state), t
        seen["done"] += len(de)
    return vec, off, tw, seen


@pytest.mark.parametrize("m", [10, 70])
@pytest.mark.parametrize("path", PATHS)
def test_every_launch_path(launch_path, path, m):
    launch_path(SWITCHES.get(path, {}))
    _, _, _, seen = norm_vs_off(_cfg(rso_count=m, steps=5, reward_type="jones"), 12, toggle=(5, 8))
    assert seen["done"] >= E and seen["term"] >= E, seen


@pytest.mark.parametrize("n_envs,m", [(5000, 2), (40000, 1)])
def test_many_environments(launch_path, n_envs, m):
    """E past one leaf per thread (5000: 157 leaves of 32 rows, a tree of 8 levels) and past the fixed leaf length
    (40000: leaves of 40 rows): the device's parallel leaves and tree equal the host build's order."""
    _, _, tw, seen = norm_vs_off(_cfg(rso_count=m, steps=3, reward_type="trinary"), 4, E=n_envs, episode_stats=False,
                                 toggle=(2,))
    assert seen["done"] > 0 and tw.E == n_envs


@pytest.mark.parametrize("over,kw,auto_reset", [
    ({"obs_returned": "flatten", "reward_type": "trinary"}, {}, True),
    ({"obs_returned": "2-d", "reward_type": "shaped"}, {"gamma": 1.0, "clip_obs": 3.0}, True),
    ({"obs_returned": "aer", "reward_type": "jones"}, {"gamma": 0.0}, True),
    ({"obs_returned": "flatten", "obs_dtype": "float32", "reward_type": "shaped"}, {"norm_reward": False}, True),
    ({"obs_returned": "2-d", "obs_dtype": "float32", "reward_type": "jones"}, {"epsilon": 0.0}, False),
    ({"obs_returned": "aer", "reward_type": "trinary"}, {"norm_obs": False, "clip_reward": 0.5}, False),
    ({"obs_returned": "flatten", "reward_type": "jones"}, {"training": False}, True),
])
@pytest.mark.parametrize("m", [10, 70])
def test_layouts_dtypes_rewards(launch_path, over, kw, auto_reset, m):
    norm_vs_off(_cfg(rso_count=m, steps=4, **over), 10, kw=kw, auto_reset=auto_reset, toggle=(3,))


def test_state_reload_continues_bit_identically(launch_path):
    """A state saved from one environment and loaded into a fresh one with the same raw stream: from there on both return
    the same normalized obs, rewards and states."""
    cfg = _cfg(rso_count=10, steps=5)
    seeds = list(range(900, 900 + E))
    a = VecSSATaskerEnv(dict(cfg, normalize=True), E, seeds=seeds, rng="device")
    b = VecSSATaskerEnv(dict(cfg, normalize={"training": False}), E, seeds=seeds, rng="device")
    rng = np.random.RandomState(1)
    acts = [rng.randint(0, 10, size=E).astype(np.int32) for _ in range(14)]
    for t in range(7):
        a.vector_step(acts[t]), b.vector_step(acts[t])
    b.load_normalizer_state(a.normalizer_state())
    b.training = True
    assert bits(_state_vec(a.normalizer_state()), _state_vec(b.normalizer_state()))
    for t in range(7, 14):
        oa, ra, da, _ = a.vector_step(acts[t])
        oa, ra = np.array(oa, copy=True), np.array(ra, copy=True)
        ob, rb, db, _ = b.vector_step(acts[t])
        assert bits(oa, ob) and bits(ra, rb) and np.array_equal(da, db), t
    assert bits(_state_vec(a.normalizer_state()), _state_vec(b.normalizer_state()))


@pytest.mark.parametrize("path", ["default", "refresh_chain", "team"])
def test_reset_at_and_vector_reset(launch_path, path):
    """reset_at(e): returns[e] = 0 and its fresh row normalized with the current statistics, nothing updated; vector_reset:
    returns zeroed and the observation statistics updated from the fresh rows."""
    launch_path(SWITCHES.get(path, {}))
    cfg = _cfg(rso_count=10, steps=6, obs_returned="2-d")
    vec, off, tw, _ = norm_vs_off(cfg, 4)
    for e in (3, 17):
        vec.reset_at(e), off.reset_at(e)
        mask = np.zeros(E, bool)
        mask[e] = True
        out, _ = tw.run(2, _rows(off.obs).astype(np.float64), done=mask)
        assert bits(_rows(vec.obs)[e], out[e]) and bits(_rows(vec.get_original_obs()), _rows(off.obs))
        assert bits(_state_vec(vec.normalizer_state()), tw.state)
    o = vec.vector_reset()
    off.vector_reset()
    assert bits(_rows(o), tw.reset(_rows(off.obs).astype(np.float64)))
    assert bits(_state_vec(vec.normalizer_state()), tw.state) and not np.any(vec.normalizer_state()["returns"])


@pytest.mark.parametrize("over", [{}, {"obs_returned": "aer"}, {"obs_dtype": "float32"}])
def test_device_step_views_equal_host_step(launch_path, over):
    import torch
    cfg = _cfg(rso_count=10, steps=5, **over)
    seeds = list(range(300, 300 + E))
    host = VecSSATaskerEnv(dict(cfg, normalize=True), E, seeds=seeds, rng="device")
    dev = VecSSATaskerEnv(dict(cfg, normalize=True), E, seeds=seeds, rng="device")
    v = dev.device_views()
    rng = np.random.RandomState(2)
    for t in range(10):
        a = rng.randint(0, 10, size=E).astype(np.int32)
        o, r, d, _ = host.vector_step(a)
        v["actions"].copy_(torch.from_numpy(a))
        dev.vector_step_device()
        torch.cuda.synchronize()
        assert bits(v["obs_norm"].cpu().numpy(), _rows(o)) and bits(v["reward_norm"].cpu().numpy(), r), t
        assert np.array_equal(v["done"].cpu().numpy().astype(bool), d), t
    assert bits(_state_vec(host.normalizer_state()), _state_vec(dev.normalizer_state()))


@pytest.mark.parametrize("over", [{}, {"obs_returned": "aer"}, {"obs_dtype": "float32"}])
def test_launch_counts(launch_path, over):
    """One kernel more per step and per reset with normalization on (none for a float32 step: k_normalize writes its
    float32 rows in place of k_obs_to_f32); unchanged with it off again."""
    cfg = _cfg(rso_count=10, steps=5, **over)
    on = VecSSATaskerEnv(dict(cfg, normalize=True), E, seeds=list(range(E)), rng="device")
    off = VecSSATaskerEnv(cfg, E, seeds=list(range(E)), rng="device")
    a = np.zeros(E, np.int32)

    def per_step(env):
        env.vector_step(a)
        l0 = env.ukf.launch_count
        env.vector_step(a)
        return env.ukf.launch_count - l0

    extra = 0 if over.get("obs_dtype") == "float32" else 1
    assert per_step(on) == per_step(off) + extra
    l0, l1 = on.ukf.launch_count, off.ukf.launch_count
    on.vector_reset(), off.vector_reset()
    assert on.ukf.launch_count - l0 == off.ukf.launch_count - l1 + 1
    on.ukf.rollout_normalize(False)
    on.normalize = False
    assert per_step(on) == per_step(off)


def test_refusals(launch_path):
    cfg = _cfg(rso_count=4, steps=5)
    with pytest.raises(ValueError):
        VecSSATaskerEnv(dict(cfg, normalize=True), 4, seeds=list(range(4)), rng="host")
    with pytest.raises(ValueError):
        VecSSATaskerEnv(dict(cfg, normalize={"gama": 0.9}), 4, seeds=list(range(4)), rng="device")
    off = VecSSATaskerEnv(cfg, 4, seeds=list(range(4)), rng="device")
    with pytest.raises(ValueError):
        off.normalizer_state()
    u = BatchedUKF(n_envs=4, m=4, dt=20.0, Q=np.eye(6), R=np.eye(3), obs_lla=[0.5, 0.1, 0.0], obs_limit_rad=0.0)
    with pytest.raises(F.SsaUkfError):  # before rollout_config
        u.rollout_normalize()
    u.close()
    vec = VecSSATaskerEnv(dict(cfg, normalize=True), 4, seeds=list(range(4)), rng="device")
    u = vec.ukf
    for bad in [dict(gamma=1.5), dict(gamma=-0.1), dict(gamma=float("nan")), dict(clip_obs=0.0), dict(clip_reward=-1.0),
                dict(epsilon=-1e-8), dict(epsilon=float("nan")), dict(obs_layout=3)]:
        with pytest.raises(F.SsaUkfError):
            u.rollout_normalize(**bad)
    lib, h = u.lib, u.h
    n = 2 * u.norm_F + 4 + 4
    buf = np.zeros(n + 1)
    assert lib.ssa_ukf_rollout_norm_state_download(h, H.p(buf), n + 1, None) == F.SSA_EINVAL
    assert lib.ssa_ukf_rollout_norm_state_upload(h, H.p(buf), n - 1, None) == F.SSA_EINVAL
    assert lib.ssa_ukf_rollout_norm_state_download(h, None, n, None) == F.SSA_EINVAL
    assert lib.ssa_ukf_rollout_norm_state_download(h, H.p(buf), n, None) == F.SSA_OK
    with pytest.raises(F.SsaUkfError):  # the step's layout differs from the normalization's
        u.rollout_step(True, obs_aer=True)
    with pytest.raises(F.SsaUkfError):
        u.rollout_terminal_obs_norm([4])
    u.rollout_normalize(False)
    assert lib.ssa_ukf_rollout_norm_state_download(h, H.p(buf), n, None) == F.SSA_EINVAL
    assert lib.ssa_ukf_rollout_norm_io(h, None, None) == F.SSA_EINVAL
    p = ctypes.c_void_p()
    assert lib.ssa_ukf_device_ptr(h, F.F_ROLLOUT_OBS_NORM, ctypes.byref(p), None) == F.SSA_EINVAL
