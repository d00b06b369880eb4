"""-m gpu: the device-resident episodic mode (VecSSATaskerEnv(rng='device')) with the 'shaped' reward and the 'aer'
observation layout, EXACT against a host emulation over many auto-resets.

LayoutTwin extends helpers.EpisodicTwin: the 'shaped' reward of every step comes from episode.step_reward (the rule the
drop-in env and the host-RNG vec env use) with the REQUESTED actions, the environment's own reward history and the
sigma_pos of its previous step; the 'aer' rows are twin_hx_aer of the filter means through the environment's
trans_matrix row, np.trace's order over the diag P columns and nan_to_num(0.001) - what vec_env._format_obs computes on
the host.  The 'aer' device path is also compared with the pre-change host formatting of the flatten rows, device_views
with vector_step, and the C ABI refuses the two observation bits together."""
import collections

import numpy as np
import pytest

import helpers as H
from ssa_gym_b200 import _lib as F
from ssa_gym_b200 import dynamics
from ssa_gym_b200.episode import step_reward
from ssa_gym_b200.vec_env import VecSSATaskerEnv
from test_gpu_env_reduce_paths import SWITCHES, _cfg, launch_path  # noqa: F401  (launch_path: fixture)

pytestmark = pytest.mark.gpu
E = 45


class LayoutTwin(H.EpisodicTwin):
    """EpisodicTwin with the 'shaped' reward and the 'aer' layout of the device mode.  `branches` counts the shaped
    reward's branches: 'lost', 'success<8' / 'success8-128' / 'success>128' (by the length i of the summed history),
    '+1/n', '-1/n', and 'skipped+1/n' (a matched action on a step that update_interval skips)."""

    def __init__(self, vec, cfg):
        super().__init__(vec, cfg)
        self.shaped = self.reward_type == "shaped"
        if self.shaped:
            self.reward_type = "jones"  # the base class's done rule and greedy columns; the reward is replaced below
        self.aer = cfg.get("obs_returned", "flatten") == "aer"
        self.rew_hist = np.zeros((self.E, self.n))
        self.spos_prev = np.zeros((self.E, self.m))  # all equal on a fresh state: np.argmax gives 0
        self.obs_itrs = np.array(self.cfg.obs_itrs[:])
        self.T = np.array(self.cfg.T[:]).reshape(3, 3)
        self.branches = collections.Counter()

    def format(self, obs12):
        """The observation rows the device returns: [N, 12] (flatten) or [E, m*4] ('aer')."""
        if not self.aer:
            return obs12.copy()
        E, m = self.E, self.m
        o = obs12.reshape(E, m, 12)
        rows = self.table[np.minimum(self.step_idx, self.n - 1)]
        out = np.empty((E, m, 4))
        for e in range(E):
            out[e, :, :3] = H.lib_hx("twin", o[e, :, :6], rows[e].reshape(3, 3), self.obs_itrs, self.T)
        d = o[:, :, 6:]
        out[:, :, 3] = ((((d[:, :, 0] + d[:, :, 1]) + d[:, :, 2]) + d[:, :, 3]) + d[:, :, 4]) + d[:, :, 5]
        return np.nan_to_num(out.reshape(E, m * 4), nan=0.001, posinf=0.001, neginf=0.001)

    def reset(self):
        obs, greedy = super().reset()
        self.rew_hist[:] = 0.0
        self.spos_prev[:] = 0.0
        return self.format(obs), greedy

    def step(self, actions, auto_reset=True):
        _, reward, done, _ = super().step(actions, auto_reset=False)
        st, n = self.st, self.n
        if self.shaped:
            dpos, spos = st.dpos.reshape(self.E, self.m), st.spos.reshape(self.E, self.m)
            reward = np.zeros(self.E)
            for e in range(self.E):
                i = int(self.step_idx[e])
                r, d = step_reward("shaped", i, n, int(actions[e]), dpos[e], self.spos_prev[e], self.rew_hist[e, :i])
                assert d == done[e], (e, i)
                reward[e] = r
                if i < n:
                    self.rew_hist[e, i] = r
                worst = np.max(dpos[e])
                if worst > 5e6:
                    self.branches["lost"] += 1
                elif worst < 3e4:
                    self.branches["success<8" if i < 8 else "success8-128" if i <= 128 else "success>128"] += 1
                elif r > 0:
                    self.branches["+1/n"] += 1
                    if i % self.update_interval:
                        self.branches["skipped+1/n"] += 1
                else:
                    self.branches["-1/n"] += 1
            self.spos_prev = spos.copy()
        if auto_reset and done.any():
            self._draw(done)
            self._refresh(done)
            self.rew_hist[done] = 0.0
            self.spos_prev[done] = 0.0
        return self.format(st.obs), reward, done, self.greedy.copy()


def layouts_vs_twin(cfg, total_steps, E=E, seed0=500, action_seed=11, random_every=2):
    """VecSSATaskerEnv(cfg, rng='device') against LayoutTwin, step by step: obs, reward, done, the six greedy columns
    and vec.i exact.  Actions: random on every `random_every`-th step, the device's visible-greedy pick otherwise.
    Returns (branch counts, auto-resets)."""
    vec = VecSSATaskerEnv(cfg, E, seeds=list(range(seed0, seed0 + E)), rng="device")
    emu = LayoutTwin(vec, cfg)
    obs_e, g_e = emu.reset()
    assert H.bits_equal(np.asarray(vec.obs).reshape(obs_e.shape), obs_e)
    assert np.array_equal(vec._io["greedy"], g_e)
    rng = np.random.RandomState(action_seed)
    resets = 0
    for t in range(total_steps):
        a = rng.randint(0, emu.m, size=E) if t % random_every == 0 else vec.greedy_actions(F.TASKER_VISIBLE_GREEDY)
        a = np.asarray(a, dtype=np.int32)
        obs_v, r_v, d_v, _ = vec.vector_step(a)
        obs_e, r_e, d_e, g_e = emu.step(a)
        assert np.array_equal(d_v, d_e), (t, np.where(d_v != d_e))
        assert H.bits_equal(r_v, r_e), (t, np.where(r_v != r_e), r_v, r_e)
        assert H.bits_equal(np.asarray(obs_v).reshape(obs_e.shape), obs_e), (t, np.where(obs_v.reshape(obs_e.shape) != obs_e))
        assert np.array_equal(vec._io["greedy"], g_e), t
        assert np.array_equal(vec.i, emu.step_idx), t
        resets += int(d_e.sum())
    vec.close()
    return emu.branches, resets


@pytest.mark.parametrize("update_interval", [1, 2])
@pytest.mark.parametrize("m", [10, 70])
@pytest.mark.parametrize("switch", ["default"] + sorted(SWITCHES))
def test_shaped_aer_equals_twin_on_every_launch_path(launch_path, switch, m, update_interval):  # noqa: F811
    """'shaped' + 'aer' through every launch path (SSA_UKF_REFRESH_CHAIN=1 and the team kernel reset through
    k_env_reset), one warp per environment (m = 10) and one CTA (m = 70), over at least E auto-resets."""
    if switch != "default":
        launch_path(SWITCHES[switch])
    cfg = _cfg(rso_count=m, steps=7, reward_type="shaped", update_interval=update_interval, obs_returned="aer",
               obs_limit=10 if m == 70 else -90)
    branches, resets = layouts_vs_twin(cfg, 30)
    assert resets >= E and branches["+1/n"] > 0 and branches["-1/n"] > 0, (resets, branches)
    if update_interval > 1:
        assert branches["skipped+1/n"] > 0, branches


@pytest.mark.parametrize("over", [
    {"reward_type": "jones", "obs_returned": "aer"},
    {"reward_type": "trinary", "obs_returned": "aer"},
    {"reward_type": "shaped", "obs_returned": "flatten"},
    {"reward_type": "shaped", "obs_returned": "2d"},
])
def test_layouts_equal_twin(over):
    """The other corners of the configuration matrix: 'aer' with the device-finished rewards, 'shaped' with the
    state-vector layouts."""
    branches, resets = layouts_vs_twin(_cfg(rso_count=10, steps=7, update_interval=2, **over), 25)
    assert resets >= E


# Configurations (found with the host twin) in which the shaped reward reaches every branch: successes after few steps
# (two objects), after tens of steps and after more than 128 (a sparse update_interval), and a lost object (below:
# x_sigma of 3000 km).  The history sums therefore run through all three regimes of numpy's pairwise order.
SHAPED_BRANCHES = [
    ({"rso_count": 2, "steps": 40, "update_interval": 1}, {"success<8"}),
    ({"rso_count": 3, "steps": 200, "update_interval": 4}, {"success8-128"}),
    ({"rso_count": 4, "steps": 400, "update_interval": 24}, {"success>128"}),
]


@pytest.mark.parametrize("over,need", SHAPED_BRANCHES)
def test_shaped_reward_branches_equal_twin(over, need):
    cfg = _cfg(reward_type="shaped", obs_returned="aer", **over)
    branches, _ = layouts_vs_twin(cfg, cfg["steps"] + 60, E=24, random_every=1)
    assert all(branches[k] > 0 for k in need | {"+1/n", "-1/n"}), branches
    if over["update_interval"] > 1:
        assert branches["skipped+1/n"] > 0, branches


def test_shaped_lost_branch_equals_twin():
    cfg = _cfg(reward_type="shaped", rso_count=2, steps=20, update_interval=1, x_sigma=(3e6, 3e6, 3e6, 100.0, 100.0, 100.0),
               P_0=None)
    branches, _ = layouts_vs_twin(cfg, 30, E=24)
    assert branches["lost"] > 0, branches


def _old_aer(vec, obs12):
    """The host formatting of the 'aer' rows before the device computed them: one hx_aer_erfa call per distinct step
    index, trace in np.trace's order, nan_to_num(0.001)."""
    o = np.asarray(obs12).reshape(-1, vec.m, 12)
    steps = np.minimum(vec.i, len(vec.trans_matrix) - 1)
    out = np.empty((len(o), vec.m, 4))
    for i in np.unique(steps):
        sel = np.where(steps == i)[0]
        out[sel, :, :3] = dynamics.hx_aer_erfa(o[sel, :, :6], vec.trans_matrix[i], vec.obs_lla, vec.obs_itrs)
    d = o[:, :, 6:]
    out[:, :, 3] = ((((d[:, :, 0] + d[:, :, 1]) + d[:, :, 2]) + d[:, :, 3]) + d[:, :, 4]) + d[:, :, 5]
    return np.nan_to_num(out.reshape(len(o), vec.m * 4), nan=0.001, posinf=0.001, neginf=0.001)


@pytest.mark.parametrize("reward_type", ["jones", "trinary"])
def test_device_aer_equals_host_formatting_of_flatten_rows(reward_type):
    """Same seeds and actions: the 'aer' device env's observations equal the flatten device env's rows formatted by the
    host code it replaces, at every step; with 'jones' the episodes end at different step indices (successes of two
    objects), so that the old code makes many hx_aer_erfa calls per step."""
    cfg = _cfg(rso_count=2, steps=60, reward_type=reward_type, update_interval=1)
    seeds = list(range(900, 900 + E))
    va = VecSSATaskerEnv(dict(cfg, obs_returned="aer"), E, seeds=seeds, rng="device")
    vf = VecSSATaskerEnv(dict(cfg, obs_returned="flatten"), E, seeds=seeds, rng="device")
    assert H.bits_equal(va.obs, _old_aer(vf, vf.obs))
    rng = np.random.RandomState(3)
    distinct = set()
    for t in range(70):
        a = rng.randint(0, 2, size=E)
        oa, ra, da, _ = va.vector_step(a)
        of, rf, df, _ = vf.vector_step(a)
        assert np.array_equal(da, df) and H.bits_equal(ra, np.nan_to_num(rf, nan=0.5, posinf=0.5, neginf=0.5)), t
        assert np.array_equal(va.i, vf.i)
        assert H.bits_equal(oa, _old_aer(vf, of)), t
        distinct.add(len(np.unique(vf.i)))
    assert reward_type == "trinary" or max(distinct) > 5, distinct
    va.close()
    vf.close()


@pytest.mark.parametrize("over", [{"reward_type": "shaped", "obs_returned": "aer"},
                                  {"reward_type": "shaped", "obs_returned": "flatten"},
                                  {"reward_type": "jones", "obs_returned": "aer"}])
def test_device_io_equals_vector_step(over):
    """vector_step_device + device_views() give what vector_step gives, over auto-resets."""
    import torch
    cfg = _cfg(rso_count=6, steps=9, update_interval=2, **over)
    seeds = list(range(300, 300 + E))
    vh = VecSSATaskerEnv(cfg, E, seeds=seeds, rng="device")
    vd = VecSSATaskerEnv(cfg, E, seeds=seeds, rng="device")
    views = vd.device_views()
    width = 4 if over["obs_returned"] == "aer" else 12
    assert tuple(views["obs"].shape) == (E, 6 * width)
    rng = np.random.RandomState(5)
    resets = 0
    for t in range(40):
        a = rng.randint(0, 6, size=E).astype(np.int32)
        oh, rh, dh, _ = vh.vector_step(a)
        views["actions"].copy_(torch.from_numpy(a))
        vd.vector_step_device()
        torch.cuda.synchronize()
        assert H.bits_equal(views["obs"].cpu().numpy(), np.asarray(oh).reshape(E, 6 * width)), t
        assert H.bits_equal(views["reward"].cpu().numpy(), vh._io["reward"]), t
        assert np.array_equal(views["done"].cpu().numpy().astype(bool), dh), t
        assert np.array_equal(views["greedy"].cpu().numpy(), vh._io["greedy"]), t
        resets += int(dh.sum())
    assert resets >= E
    vh.close()
    vd.close()


def test_obs_aer_and_obs_f32_together_are_refused():
    cfg = _cfg(rso_count=4, steps=5, reward_type="jones", obs_returned="aer")
    vec = VecSSATaskerEnv(cfg, 4, seeds=[1, 2, 3, 4], rng="device")
    u = vec.ukf
    rc = u.lib.ssa_ukf_rollout_step(u.h, 1 | F.ROLLOUT_OBS_AER | F.ROLLOUT_OBS_F32, None)
    assert rc == F.SSA_EINVAL and b"exclude" in u.lib.ssa_ukf_last_error()
    with pytest.raises(F.SsaUkfError):
        u.rollout_step(obs_f32=True, obs_aer=True)
    ptr, nbytes = u.device_ptr(F.F_ROLLOUT_OBS_AER)
    assert ptr and nbytes == 4 * 4 * 8 * 4
    with pytest.raises(ValueError):
        VecSSATaskerEnv(dict(cfg, obs_dtype="float32"), 4, rng="device")
    vec.close()
