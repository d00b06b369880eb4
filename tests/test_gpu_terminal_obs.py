"""-m gpu: episode boundaries of the device-resident episodic mode (VecSSATaskerEnv(rng='device')): the truncation flag,
the final observations of finished episodes and reset_at, EXACT against a host emulation on every launch path.

TermTwin extends test_gpu_episodic_layouts.LayoutTwin (helpers.EpisodicTwin with the 'shaped' reward and the 'aer'
layout): before an auto-reset re-draws the finished environments it records their observation rows in the layout of
the step (format(st.obs) at the step index the episode ended on) and the truncation rule: done raised by the step limit
alone, a lost (max delta_pos > 5e6) or successful (< 3e4) last step being a termination, 'trinary' ending at the limit
only.  reset_at is emulated by the twin's own _draw / _refresh of one environment."""
import collections

import numpy as np
import pytest

import helpers as H
from ssa_gym_b200 import _lib as F
from ssa_gym_b200 import dynamics
from ssa_gym_b200.ukf import BatchedUKF
from ssa_gym_b200.vec_env import VecSSATaskerEnv
from test_gpu_env_reduce_paths import SWITCHES, _cfg, launch_path  # noqa: F401  (launch_path: fixture)
from test_gpu_episode_stats import StatsTwin, check_against_formulas
from test_gpu_episodic_layouts import LayoutTwin

pytestmark = pytest.mark.gpu
E = 45


class TermTwin(LayoutTwin):
    """LayoutTwin that also gives, for the last step, `truncated` [E] and `term` [finished, row] (the final rows)."""

    def __init__(self, vec, cfg):
        super().__init__(vec, cfg)
        self.trinary = cfg["reward_type"] == "trinary"
        self.truncated = np.zeros(self.E, bool)
        self.term = None

    def step(self, actions, auto_reset=True):
        obs, reward, done, greedy = super().step(actions, auto_reset=False)
        max_dpos = self.st.dpos.reshape(self.E, self.m).max(1)
        self.truncated = done & (self.trinary | ~((max_dpos > 5e6) | (max_dpos < 3e4)))
        self.term = obs.reshape(self.E, -1)[done].copy()  # (format at the ending step index, before the re-draw)
        if auto_reset and done.any():
            self.reset_envs(done)
            obs, greedy = self.format(self.st.obs), self.greedy.copy()
        return obs, reward, done, greedy

    def reset_envs(self, mask):
        """ssa_ukf_rollout_reset_envs / an auto-reset of the environments in `mask` (bool [E])."""
        self._draw(mask)
        self._refresh(mask)
        self.rew_hist[mask] = 0.0
        self.spos_prev[mask] = 0.0


def _rows(obs, shape):
    return np.asarray(obs).reshape(shape)


def term_vs_twin(cfg, total_steps, E=E, seed0=500, action_seed=11, auto_reset=True):
    """VecSSATaskerEnv(terminal_observation=True) against TermTwin and against a switch-off environment with the same
    seeds and actions.  Every step: obs, reward, done, greedy equal to both; vec.truncated, device_views()['truncated'] and
    every infos[e]['TimeLimit.truncated'] equal to the twin's rule; with auto-reset the infos' terminal_observation, the
    'terminal_obs' device view and rollout_terminal_obs of the finished environments equal the twin's final rows.
    Returns counters: time-limit endings ('truncated') and lost / successful ones ('terminated')."""
    seeds = list(range(seed0, seed0 + E))
    vec = VecSSATaskerEnv(dict(cfg, terminal_observation=True), E, seeds=seeds, rng="device", auto_reset=auto_reset)
    off = VecSSATaskerEnv(cfg, E, seeds=seeds, rng="device", auto_reset=auto_reset)
    emu = TermTwin(vec, cfg)
    obs_e, _ = emu.reset()
    assert H.bits_equal(_rows(vec.obs, obs_e.shape), obs_e)
    views = vec.device_views()
    rng = np.random.RandomState(action_seed)
    seen = collections.Counter()
    for t in range(total_steps):
        a = rng.randint(0, emu.m, size=E) if t % 2 == 0 else vec.greedy_actions(F.TASKER_VISIBLE_GREEDY)
        a = np.asarray(a, dtype=np.int32)
        o_v, r_v, d_v, infos = vec.vector_step(a)
        o_v, g_v = np.array(o_v, copy=True), vec._io["greedy"].copy()
        o_o, r_o, d_o, i_o = off.vector_step(a)
        assert H.bits_equal(o_v, o_o) and H.bits_equal(r_v, r_o) and np.array_equal(d_v, d_o), t
        assert np.array_equal(g_v, off._io["greedy"]) and not any(i_o), t
        o_e, r_e, d_e, g_e = emu.step(a, auto_reset)
        assert np.array_equal(d_v, d_e) and H.bits_equal(r_v, r_e), (t, np.where(d_v != d_e))
        assert H.bits_equal(_rows(o_v, o_e.shape), o_e) and np.array_equal(g_v, g_e), t
        assert np.array_equal(vec.truncated, emu.truncated), (t, np.where(vec.truncated != emu.truncated))
        assert np.array_equal(views["truncated"].cpu().numpy().astype(bool), emu.truncated), t
        de = np.flatnonzero(d_v)
        assert [e for e in range(E) if infos[e]] == de.tolist(), t
        for e in de:
            tr = infos[e]["TimeLimit.truncated"]
            assert isinstance(tr, bool) and tr == emu.truncated[e], (t, e)
        if auto_reset and len(de):
            assert H.bits_equal(vec.ukf.rollout_terminal_obs(de), emu.term), t
            assert H.bits_equal(views["terminal_obs"].cpu().numpy()[de], emu.term), t
            for k, e in enumerate(de):
                assert H.bits_equal(np.asarray(infos[e]["terminal_observation"]).reshape(-1), emu.term[k]), (t, e)
        elif len(de):
            assert all("terminal_observation" not in infos[e] for e in de), t
        seen["truncated"] += int(emu.truncated.sum())
        seen["terminated"] += int((d_e & ~emu.truncated).sum())
    vec.close()
    off.close()
    return seen


@pytest.mark.parametrize("update_interval", [1, 2])
@pytest.mark.parametrize("m", [10, 70])
@pytest.mark.parametrize("switch", ["default"] + sorted(SWITCHES))
def test_terminal_obs_equal_twin_on_every_launch_path(launch_path, switch, m, update_interval):  # noqa: F811
    """Every launch path (k_env_refresh, and k_env_reset on the refresh-chain and team paths), one warp (m = 10) and one
    CTA (m = 70) per environment; the flatten rows with update_interval 1, the 'aer' rows with 2, over >= E auto-resets."""
    if switch != "default":
        launch_path(SWITCHES[switch])
    cfg = _cfg(rso_count=m, steps=7, reward_type="jones" if m == 10 else "shaped", update_interval=update_interval,
               obs_returned="flatten" if update_interval == 1 else "aer", obs_limit=10 if m == 70 else -90)
    seen = term_vs_twin(cfg, 30)
    assert seen["truncated"] >= E, seen


# time-limit endings next to successes (three objects, default x_sigma, 4-step episodes: about half of the episodes
# succeed) or losses (two objects, x_sigma of 2500 km).  (Two objects with the default x_sigma succeed before any
# 8-step limit: no time-limit ending at all.)
ENDINGS = {"success": {"rso_count": 3, "steps": 4},
           "lost": {"rso_count": 2, "steps": 8, "x_sigma": (2.5e6, 2.5e6, 2.5e6, 100.0, 100.0, 100.0), "P_0": None}}


@pytest.mark.parametrize("ending", sorted(ENDINGS))
@pytest.mark.parametrize("reward_type", ["jones", "trinary", "shaped"])
def test_truncation_equals_rule(reward_type, ending):
    """The device's flag equals the rule for all three rewards, with both kinds of ending in each run ('trinary' has
    time-limit endings only); the host-RNG mode puts the same rule on the states it steps."""
    cfg = _cfg(reward_type=reward_type, update_interval=1, **ENDINGS[ending])
    m = cfg["rso_count"]
    seen = term_vs_twin(cfg, 30)
    assert seen["truncated"] > 0 and (reward_type == "trinary" or seen["terminated"] > 0), seen
    # host mode: auto-reset emulated with reset_at after reading this step's delta_pos
    host = VecSSATaskerEnv(dict(cfg, terminal_observation=True), E, seeds=list(range(40, 40 + E)), auto_reset=False)
    rng = np.random.RandomState(1)
    kinds = collections.Counter()
    for t in range(30):
        _, _, d, infos = host.vector_step(rng.randint(0, m, size=E))
        max_dpos = host.ukf.download(F.F_DELTA_POS).reshape(E, m).max(1)
        rule = d & ((reward_type == "trinary") | ~((max_dpos > 5e6) | (max_dpos < 3e4)))
        assert [e for e in range(E) if "TimeLimit.truncated" in infos[e]] == np.flatnonzero(d).tolist(), t
        assert all(infos[e]["TimeLimit.truncated"] is bool(rule[e]) for e in np.flatnonzero(d)), t
        kinds["truncated"] += int(rule.sum())
        kinds["terminated"] += int((d & ~rule).sum())
        for e in np.flatnonzero(d):
            host.reset_at(int(e))
    assert kinds["truncated"] > 0 and (reward_type == "trinary" or kinds["terminated"] > 0), kinds
    host.close()


def _host_aer(vec, rows12, steps):
    """vec_env._format_obs's host formatting of flatten rows [k, m*12] at the step indices `steps` [k]."""
    o = np.asarray(rows12).reshape(len(rows12), vec.m, 12)
    out = np.empty((len(o), vec.m, 4))
    for k, i in enumerate(np.minimum(steps, len(vec.trans_matrix) - 1)):
        out[k, :, :3] = dynamics.hx_aer_erfa(o[k:k + 1, :, :6], vec.trans_matrix[i], vec.obs_lla, vec.obs_itrs)[0]
    d = o[:, :, 6:]
    out[:, :, 3] = ((((d[:, :, 0] + d[:, :, 1]) + d[:, :, 2]) + d[:, :, 3]) + d[:, :, 4]) + d[:, :, 5]
    return np.nan_to_num(out.reshape(len(o), vec.m * 4), nan=0.001, posinf=0.001, neginf=0.001)


@pytest.mark.parametrize("layout,dtype", [("flatten", "float64"), ("2d", "float64"), ("aer", "float64"),
                                          ("flatten", "float32"), ("2d", "float32")])
def test_terminal_observation_layouts(layout, dtype):
    """infos[e]['terminal_observation'] has the shape and dtype of the host mode's (float32: numpy's astype of the
    float64 rows) and equals the flatten rows of a float64 device env with the same seeds and actions, formatted on the
    host at the ending step index for 'aer'."""
    cfg = _cfg(rso_count=2, steps=8, reward_type="jones", update_interval=1, obs_returned=layout, terminal_observation=True)
    seeds = list(range(200, 200 + E))
    host = VecSSATaskerEnv(cfg, E, seeds=seeds)
    ref_shape = None
    while ref_shape is None:
        _, _, d, infos = host.vector_step(np.zeros(E, np.int32))
        if d.any():
            t0 = infos[int(np.flatnonzero(d)[0])]["terminal_observation"]
            ref_shape, ref_dtype = t0.shape, t0.dtype
    host.close()
    dev = VecSSATaskerEnv(dict(cfg, obs_dtype=dtype), E, seeds=seeds, rng="device")
    flat = VecSSATaskerEnv(dict(cfg, obs_returned="flatten"), E, seeds=seeds, rng="device")
    rng = np.random.RandomState(7)
    finished = 0
    for t in range(25):
        a = rng.randint(0, 2, size=E)
        i_end = flat.i + 1
        _, _, d, infos = dev.vector_step(a)
        _, _, d_f, infos_f = flat.vector_step(a)
        assert np.array_equal(d, d_f), t
        de = np.flatnonzero(d)
        if not len(de):
            continue
        rows = np.array([infos_f[e]["terminal_observation"] for e in de])
        want = _host_aer(flat, rows, i_end[de]) if layout == "aer" else rows.astype(dtype).reshape((len(de),) + ref_shape)
        for k, e in enumerate(de):
            got = infos[e]["terminal_observation"]
            assert got.shape == ref_shape and got.dtype == (ref_dtype if dtype == "float64" else np.float32), (got.shape, got.dtype)
            assert H.bits_equal(got, want[k]), (t, e)
        finished += len(de)
    assert finished >= E
    dev.close()
    flat.close()


@pytest.mark.parametrize("layout", ["flatten", "aer"])
def test_device_io_equals_vector_step(layout):
    """vector_step_device leaves in device_views() the truncated flags and final rows that vector_step returns."""
    import torch
    cfg = _cfg(rso_count=6, steps=9, update_interval=2, reward_type="jones", obs_returned=layout, terminal_observation=True)
    seeds = list(range(300, 300 + E))
    vh = VecSSATaskerEnv(cfg, E, seeds=seeds, rng="device")
    vd = VecSSATaskerEnv(cfg, E, seeds=seeds, rng="device")
    views = vd.device_views()
    width = 4 if layout == "aer" else 12
    assert tuple(views["terminal_obs"].shape) == (E, 6 * width) and tuple(views["truncated"].shape) == (E,)
    rng = np.random.RandomState(5)
    resets = 0
    for t in range(40):
        a = rng.randint(0, 6, size=E).astype(np.int32)
        _, _, dh, infos = vh.vector_step(a)
        views["actions"].copy_(torch.from_numpy(a))
        vd.vector_step_device()
        torch.cuda.synchronize()
        assert np.array_equal(views["done"].cpu().numpy().astype(bool), dh), t
        assert np.array_equal(views["truncated"].cpu().numpy().astype(bool), vh.truncated), t
        de = np.flatnonzero(dh)
        if len(de):
            term = np.array([infos[e]["terminal_observation"] for e in de])
            assert H.bits_equal(views["terminal_obs"].cpu().numpy()[de], term), t
        resets += len(de)
    assert resets >= E
    vh.close()
    vd.close()


def test_switch_off_and_launch_counts():
    """Without the switch the infos are those of before (device mode: empty; host mode: terminal_observation only), and
    the step graphs launch the same kernels with the switch on and off."""
    cfg = _cfg(rso_count=6, steps=5, reward_type="jones", update_interval=1)
    seeds = list(range(100, 100 + E))
    on = VecSSATaskerEnv(dict(cfg, terminal_observation=True), E, seeds=seeds, rng="device")
    off = VecSSATaskerEnv(cfg, E, seeds=seeds, rng="device")
    host = VecSSATaskerEnv(cfg, E, seeds=seeds)
    n_done = 0
    for t in range(12):
        a = np.zeros(E, np.int32)
        _, _, d, infos = off.vector_step(a)
        assert not any(infos), t
        _, _, dh, infos_h = host.vector_step(a)
        assert all(set(infos_h[e]) == ({"terminal_observation"} if dh[e] else set()) for e in range(E)), t
        n_done += int(d.sum())
    assert n_done >= E

    def per_step(v):
        c0 = v.ukf.launch_count
        v.vector_step_device()
        return v.ukf.launch_count - c0
    for _ in range(3):
        assert per_step(on) == per_step(off)
    for v in (on, off, host):
        v.close()


@pytest.mark.parametrize("auto_reset", [True, False])
@pytest.mark.parametrize("over", [{"reward_type": "jones", "obs_returned": "flatten"},
                                  {"reward_type": "shaped", "obs_returned": "aer"}])
def test_reset_at_equals_twin(auto_reset, over):
    """reset_at(e) in the device mode, mid-episode and after a done: obs, all six greedy columns (agent_shannon's history
    restarts), the 'shaped' history and the following steps equal the twin's _draw / _refresh of that environment; the
    state of the environments never reset equals a run without resets."""
    cfg = _cfg(rso_count=10, steps=7, update_interval=1, **over)
    seeds = list(range(600, 600 + E))
    vec = VecSSATaskerEnv(cfg, E, seeds=seeds, rng="device", auto_reset=auto_reset)
    ref = VecSSATaskerEnv(cfg, E, seeds=seeds, rng="device", auto_reset=auto_reset)
    emu = TermTwin(vec, cfg)
    emu.reset()
    rng = np.random.RandomState(4)
    touched = np.zeros(E, bool)
    kinds = collections.Counter()
    for t in range(20):
        a = rng.randint(0, 10, size=E).astype(np.int32)
        o_v, r_v, d_v, _ = vec.vector_step(a)
        ref.vector_step(a)
        o_e, r_e, d_e, g_e = emu.step(a, auto_reset)
        assert np.array_equal(d_v, d_e) and H.bits_equal(r_v, r_e) and H.bits_equal(_rows(o_v, o_e.shape), o_e), t
        assert np.array_equal(vec._io["greedy"], g_e) and np.array_equal(vec.i, emu.step_idx), t
        e = int(np.flatnonzero(d_v)[0]) if d_v.any() and t % 2 else (7 * t) % E
        kinds["after_done" if d_v[e] else "mid_episode"] += 1
        mask = np.zeros(E, bool)
        mask[e] = touched[e] = True
        ep0 = vec.episodes[e]
        obs = vec.reset_at(e)
        emu.reset_envs(mask)
        obs_e = emu.format(emu.st.obs)
        assert obs is vec.obs and H.bits_equal(_rows(obs, obs_e.shape), obs_e), (t, e)
        assert np.array_equal(vec._io["greedy"], emu.greedy), (t, e)
        assert vec.i[e] == 0 and vec.episodes[e] == ep0 + 1 and np.array_equal(vec.i, emu.step_idx)
        rows = np.repeat(~touched, 10)
        for f in (F.F_X_FILTER, F.F_X_TRUE, F.F_P_FILTER, F.F_STATUS, F.F_INFLATIONS):
            assert H.bits_equal(vec.ukf.download(f)[rows], ref.ukf.download(f)[rows]), (t, f)
    assert kinds["after_done"] > 0 and kinds["mid_episode"] > 0, kinds
    vec.close()
    ref.close()


def test_reset_at_restarts_episode_statistics():
    """With episode_stats, the next record of a reset environment covers only its new episode: equal to StatsTwin with
    that environment's accumulators cleared at the reset."""
    cfg = _cfg(rso_count=10, steps=7, reward_type="jones", update_interval=1)
    vec = VecSSATaskerEnv(dict(cfg, episode_stats=True), E, seeds=list(range(500, 500 + E)), rng="device")
    emu = StatsTwin(vec, cfg)
    emu.reset()
    m = emu.m
    rng = np.random.RandomState(9)
    records = 0
    for t in range(24):
        a = rng.randint(0, m, size=E).astype(np.int32)
        _, r_v, d_v, infos = vec.vector_step(a)
        _, r_e, d_e, g_e = emu.step(a)
        assert np.array_equal(d_v, d_e) and H.bits_equal(r_v, r_e) and np.array_equal(vec._io["greedy"], g_e), t
        fin = [f[0] for f in emu.finished]
        if fin:
            recs = vec.ukf.rollout_episode_stats(fin)
            for k, (e, rec_e, hist) in enumerate(emu.finished):
                assert H.bits_equal(recs[k], rec_e) and infos[e]["episode"]["l"] == rec_e[0], (t, e)
                check_against_formulas(rec_e, hist, m, emu.seen)
                records += 1
        if t % 3 == 1:  # mid-episode resets (episodes last up to 7 steps)
            e = (5 * t) % E
            mask = np.zeros(E, bool)
            mask[e] = True
            vec.reset_at(e)
            emu._draw(mask)
            emu._refresh(mask)
            emu.acc.obj[e * m:(e + 1) * m] = 0.0
            emu.acc.env[e] = 0.0
            assert np.array_equal(vec._io["greedy"], emu.greedy), t
    assert records >= E
    vec.close()


def test_c_abi_refusals():
    """reset_envs and the terminal download refuse bad lists and calls before rollout_config with SSA_EINVAL."""
    cfg = _cfg(rso_count=4, steps=5, reward_type="jones")
    vec = VecSSATaskerEnv(cfg, 4, seeds=[1, 2, 3, 4], rng="device")
    u, lib = vec.ukf, vec.ukf.lib
    out = np.empty((5, 4 * 12))
    for idx, n, what in ((np.array([4], np.int32), 1, b"out of range"), (np.array([-1], np.int32), 1, b"out of range"),
                         (np.zeros(5, np.int32), 5, b"bad environment list"), (np.zeros(1, np.int32), -1, b"bad environment list")):
        assert lib.ssa_ukf_rollout_reset_envs(u.h, H.p(idx), n, None) == F.SSA_EINVAL
        assert what in lib.ssa_ukf_last_error()
        assert lib.ssa_ukf_rollout_terminal_obs_download(u.h, H.p(idx), n, H.p(out), None) == F.SSA_EINVAL
        assert what in lib.ssa_ukf_last_error()
    with pytest.raises(F.SsaUkfError):
        vec.reset_at(4)
    vec.close()
    b = BatchedUKF(n_envs=2, m=2, dt=20.0, Q=np.eye(6), R=np.eye(3), obs_lla=[0.6, -1.3, 20.0], obs_limit_rad=-1.0)
    zero = np.zeros(1, np.int32)
    assert b.lib.ssa_ukf_rollout_reset_envs(b.h, H.p(zero), 1, None) == F.SSA_EINVAL
    assert b"not configured" in b.lib.ssa_ukf_last_error()
    assert b.lib.ssa_ukf_rollout_terminal_obs_download(b.h, H.p(zero), 1, H.p(out), None) == F.SSA_EINVAL
    assert b"not configured" in b.lib.ssa_ukf_last_error()
    assert b.lib.ssa_ukf_rollout_truncated(b.h, None, None) == F.SSA_EINVAL
    b.close()
