"""Vectorised environments: E independent copies of the reference env advanced by ONE device step.

BASELINE.json config 3 ("4 096 parallel envs x default RSO count feeding an RLlib PPO rollout").  The reference
has no in-process vectorisation (one env per Ray worker, SURVEY.md 2.3); the shape of the API follows RLlib's
`VectorEnv` (`vector_reset`, `reset_at`, `vector_step`).  Each environment keeps the reference's semantics exactly:
its own seeded generator with the reference's draw order (SS2:206-221), its own step counter and therefore its own
`trans_matrix[i]` (shipped as a per-env table, SSA_STEP_M_PER_ENV), reward / done from `ssa_ukf_env_reduce`
(SS2:324-354), auto-reset on done.  Environment e of a `VecSSATaskerEnv` seeded with `seeds[e]` produces the same
episode as a single `SSA_Tasker_Env` seeded the same way (tests/test_gpu_vec_env.py).

`rng='device'` (SURVEY 8f-2) moves the whole host side of the step onto the device: catalog sampling and the initial
filter error at reset, the measurement noise of every step (counter-based Philox streams keyed by the env's seed,
csrc/ssa_rng.h), step counters, the trans_matrix lookup, the update_interval gate, reward / done and the auto-reset
of finished episodes.  A vector_step is then one 4*E-byte upload, one CUDA-graph launch and one download of
obs / reward / done / greedy (ssa_ukf_rollout_step).  Same distributions as the reference, NOT the same random
streams: seed-for-seed episode parity with `SSA_Tasker_Env` holds only for `rng='host'`, whose reset has to draw
n*m*3 + 7m numbers per environment from a sequential MT19937 stream on the host (measured at E = 4096: 102 ms per
vector_step in host mode against 0.45 ms in device mode).  The device mode covers the reference's whole configuration
matrix: the 'shaped' reward keeps its per-environment reward history on the device (the episode's own 1 - np.sum(
rewards[:i]) in numpy's summation order), and the 'aer' layout is computed by the last kernel of the step's graph, so
only its [E, m*4] rows (32 B per object instead of 96) cross PCIe and the host formats nothing.  With
`config['episode_stats'] = True` the step graph also accumulates every episode's return, length and the reference's
filter-consistency figures (ANEES, NIS, innovation bounds, Durbin-Watson statistics) on the device; a finished
environment reports them in `infos[e]['episode']` (see `episode_info`).  `set_tasker(agent)` runs one of the nine
agents of agents.py inside the step graph (device taskers, ssa_ukf_rollout_tasker): `vector_step()` then takes no
actions, and a loop of `vector_step_device()` compares agents with no host round trip at all.

At an episode boundary an RL learner needs to know why the episode ended and what its last observation was: PPO and A2C
bootstrap the value of an episode cut by the step limit from its final observation (Stable-Baselines3's VecEnv keys
'terminal_observation' and 'TimeLimit.truncated').  The device mode records both inside the step graph: `vec.truncated`
([E] bool, every step) says which finished episodes ended at the step limit alone (a lost or successful last step is a
termination, gym's TimeLimit rule), and with auto-reset the final observation rows of the finished environments are
kept on the device before their re-draw (device_views()['terminal_obs'], `BatchedUKF.rollout_terminal_obs`).  With
`config['terminal_observation'] = True` (either mode; off by default, since filling the dicts costs host time on every
step where environments finish) every finished environment gets `infos[e]['TimeLimit.truncated']`, and in the device
mode with auto-reset also `infos[e]['terminal_observation']` in the layout and dtype of the observations (the host mode
always fills that key on its auto-resets).  `reset_at(e)` re-draws environment e alone in either mode.

No policy learns from these observations raw (positions up to 4e7 m, covariance diagonals from 1e10 m^2 down by eight
orders of magnitude), and the usual remedy, Stable-Baselines3's VecNormalize, is a numpy pass over the [E, F] block on
every step.  With `config['normalize'] = True` (or a dict of VecNormalize's keyword arguments: training, norm_obs,
norm_reward, clip_obs, clip_reward, gamma, epsilon) the device mode does the same inside the step graph
(ssa_ukf_rollout_normalize, one kernel): observations and rewards come back normalized, the observations as float32,
and the step copies those instead of the raw float64 rows.  VecNormalize's semantics, its order of updates and its
defaults; infos[e]['terminal_observation'] is normalized as VecNormalize does, infos[e]['episode'] keeps the raw
return.  get_original_obs() / get_original_reward(), normalizer_state() / load_normalizer_state() and `training` follow
VecNormalize's names.
"""
import numpy as np

from . import _lib, agents, dynamics
from .episode import draw_episode
from .gym_shim import seeding, spaces
from .transformations import arcsec2rad, default_eops, deg2rad, gcrs2irts_matrix_b, lla2ecef, load_eop_c04, time_table
from .ukf import BatchedUKF, Q_discrete_white_noise_block

F = _lib


# the agents of agents.py that the device runs (ssa_ukf_rollout_tasker), by function and by name
_TASKERS = {
    agents.agent_naive_greedy: F.TASKER_NAIVE_GREEDY, agents.agent_visible_greedy: F.TASKER_VISIBLE_GREEDY,
    agents.agent_pos_error_greedy: F.TASKER_POS_ERROR_GREEDY, agents.agent_vel_error_greedy: F.TASKER_VEL_ERROR_GREEDY,
    agents.agent_visible_greedy_aer: F.TASKER_VISIBLE_GREEDY_AER, agents.agent_shannon: F.TASKER_SHANNON,
    agents.agent_naive_random: F.TASKER_NAIVE_RANDOM, agents.agent_visible_random: F.TASKER_VISIBLE_RANDOM,
    agents.agent_visible_greedy_spoiled: F.TASKER_VISIBLE_GREEDY_SPOILED,
}
_TASKER_NAMES = {f.__name__[len("agent_"):]: k for f, k in _TASKERS.items()}

# VecNormalize's keyword arguments and defaults (config['normalize'])
_NORM_DEFAULTS = {"training": True, "norm_obs": True, "norm_reward": True, "clip_obs": 10.0, "clip_reward": 10.0,
                  "gamma": 0.99, "epsilon": 1e-8}


def episode_info(rec):
    """infos[e]['episode'] of a finished episode from its device record (include/ssa_ukf.h, SSA_EPISODE_STATS_DOUBLES):
    'r' return and 'l' length (gymnasium's RecordEpisodeStatistics / SB3's Monitor keys), 'anees' (SS2:436-446, the mean
    of the finite NEES values over rows 0 .. l and all objects), 'nis' (mean NIS of the tasked observations, SS2:564-569),
    'observations', 'innovation_bounds' [2, 3] percentages inside 1 / 2 sigmas (SS2:598-604), 'durbin_watson' [3, 3]
    rows all observations / min per object / max per object (SS2:782-832, rounded like innovation_dw_test) and 'failed'
    (objects whose filter failed)."""
    return episode_infos(np.asarray(rec).reshape(1, -1))[0]


def episode_infos(recs):
    """episode_info of the records [n, EPISODE_STATS_DOUBLES]: one numpy pass over all of them, then one dict each (a
    step on which thousands of environments finish together builds its dicts in ~1 us each)."""
    recs = np.asarray(recs, dtype=np.float64)
    n_obs = recs[:, 6]
    with np.errstate(invalid='ignore', divide='ignore'):
        anees = np.where(recs[:, 3] > 0, recs[:, 2] / recs[:, 3], np.nan)
        nis = np.where(recs[:, 5] > 0, recs[:, 4] / recs[:, 5], np.nan)
        bounds = np.round(recs[:, 7:13].reshape(-1, 2, 3) / n_obs[:, None, None] * 100, 2)
    bounds[n_obs == 0] = np.nan
    dw = np.round(recs[:, 13:22].reshape(-1, 3, 3), 3)
    scal = zip(recs[:, 1].tolist(), recs[:, 0].astype(np.int64).tolist(), anees.tolist(), nis.tolist(),
               n_obs.astype(np.int64).tolist(), recs[:, 22].astype(np.int64).tolist())
    return [{"r": r, "l": l, "anees": a, "nis": v, "observations": o, "innovation_bounds": b, "durbin_watson": d, "failed": f}
            for (r, l, a, v, o, f), b, d in zip(scal, bounds, dw)]


class VecSSATaskerEnv:
    def __init__(self, config, num_envs, seeds=None, device=0, auto_reset=True, rng='host'):
        self.E = int(num_envs)
        assert rng in ('host', 'device')
        self.rng = rng
        self.n, self.m, self.dt = config['steps'], config['rso_count'], config['time_step']
        self.N = self.E * self.m
        self.obs_limit = np.radians(config['obs_limit'])
        self.reward_type = config['reward_type']
        self.obs_type = config['obs_type']
        self.obs_returned = config.get('obs_returned', 'flatten')
        # 'float32' (device mode, state-vector layouts): the observations cross PCIe as floats — half the bytes of the
        # step's only large copy — rounded on the device exactly like numpy's astype(float32) of the float64 rows
        self.obs_dtype = np.dtype(config.get('obs_dtype', 'float64'))
        if self.obs_dtype == np.float32:
            if rng != 'device' or self.obs_returned == 'aer':
                raise ValueError("obs_dtype='float32' needs rng='device' and a state-vector layout (obs_returned != 'aer')")
        elif self.obs_dtype != np.float64:
            raise ValueError("obs_dtype must be 'float64' or 'float32'")
        # per-episode statistics accumulated inside the step graph (device mode only: the host mode has no device episodes)
        self.episode_stats = bool(config.get('episode_stats', False))
        if self.episode_stats and rng != 'device':
            raise ValueError("episode_stats=True needs rng='device'")
        # infos[e]['TimeLimit.truncated'] on every finished environment, and the device mode's terminal_observation
        self.terminal_observation = bool(config.get('terminal_observation', False))
        # running normalization of observations and returns inside the step graph (VecNormalize; device mode only)
        nz = config.get('normalize', False)
        if nz is not True and not isinstance(nz, dict) and nz not in (False, None):
            raise ValueError("normalize must be True, False or a dict of VecNormalize keyword arguments")
        self.normalize = nz is True or isinstance(nz, dict)
        if self.normalize:
            if rng != 'device':
                raise ValueError("normalize needs rng='device'")
            kw = {} if nz is True else dict(nz)
            unknown = sorted(set(kw) - set(_NORM_DEFAULTS))
            if unknown:
                raise ValueError(f"unknown normalize keys {unknown}; VecNormalize's are {sorted(_NORM_DEFAULTS)}")
            self._norm_kw = dict(_NORM_DEFAULTS, **kw)
            self._norm_kw["training"] = bool(self._norm_kw["training"])
        self.update_interval = config['update_interval']
        self.auto_reset = auto_reset
        if config.get('orbits') is not None:
            self.orbits = np.asarray(config['orbits'])
        else:
            from .env import _default_orbits
            self.orbits = _default_orbits()
        self.obs_lla = np.array(config['observer']) * [deg2rad, deg2rad, 1]
        self.obs_itrs = lla2ecef(self.obs_lla)
        self.z_sigma = (config['z_sigma'] * np.array([arcsec2rad, arcsec2rad, 1]) if self.obs_type == 'aer'
                        else np.asarray(config['z_sigma'], dtype=float))
        self.x_sigma = np.array(config['x_sigma'])
        self.Q = Q_discrete_white_noise_block(self.dt, config['q_sigma'] ** 2, 3)
        dynamics.validate_operators(config, self.obs_type)
        self.P_0 = np.copy(np.diag(self.x_sigma ** 2)) if config.get('P_0') is None else np.copy(config['P_0'])
        self.R = np.diag(self.z_sigma ** 2) if config.get('R') is None else np.copy(config['R'])
        if config.get('trans_matrix') is not None:
            self.trans_matrix = np.ascontiguousarray(config['trans_matrix'], dtype=np.float64)
        else:
            eops = load_eop_c04(config['eop_file']) if config.get('eop_file') else default_eops()
            self.trans_matrix = np.ascontiguousarray(gcrs2irts_matrix_b(time_table(config.get('t_0'), self.dt, self.n), eops))
        self.ukf = BatchedUKF(n_envs=self.E, m=self.m, dt=self.dt, Q=self.Q, R=self.R, obs_lla=self.obs_lla,
                              obs_limit_rad=self.obs_limit, alpha=config['alpha'], beta=config['beta'], kappa=config['kappa'],
                              obs_type=self.obs_type, reward_type=self.reward_type, n_steps=self.n,
                              resample_after_predict=config.get('resample_after_predict', True), device=device)
        self.action_spaces = [spaces.Discrete(self.m) for _ in range(self.E)]
        # SS2:164-177: 'flatten' [m*12] (x and diag P per RSO), 'aer' [m*4] (az, el, range of the filter mean and trace P),
        # anything else the 2-d [m, 12] array
        oshape = {'flatten': (self.m * 12,), 'aer': (self.m * 4,)}.get(self.obs_returned, (self.m, 12))
        self.observation_space = spaces.Box(low=np.full(oshape, -np.inf), high=np.full(oshape, np.inf), dtype=self.obs_dtype.type)
        self._device = device
        self.np_randoms = [None] * self.E
        self.i = np.zeros(self.E, dtype=np.int32)
        self.z_noise = np.empty((self.E, self.n, self.m, 3)) if rng == 'host' else None
        self.x_true0 = np.empty((self.E, self.m, 6))
        self.x_filter0 = np.empty((self.E, self.m, 6))
        self.rewards_hist = np.zeros((self.E, self.n))  # for 'shaped': 1 - np.sum(rewards[:i]) (SS2:345)
        self.prev_spos_argmax = np.zeros(self.E, dtype=np.int64)
        self.episodes = np.zeros(self.E, dtype=np.int64)
        self._P0_packed = self.P_0[np.triu_indices(6)]
        self._views = None
        self.tasker = F.TASKER_EXTERNAL
        self.last_actions = np.zeros(self.E, dtype=np.int64)  # the actions the last vector_step took
        self.seed(seeds)
        # device mode, 'aer': the observation rows are computed on the device (SSA_ROLLOUT_OBS_AER), not by _format_obs
        self._obs_aer = rng == 'device' and self.obs_returned == 'aer'
        if self.rng == 'device':
            keys = np.array([int(s_) & 0xFFFFFFFFFFFFFFFF for s_ in self.init_seeds], dtype=np.uint64)
            self._io = self.ukf.rollout_config(self.orbits, self.trans_matrix, keys, self.x_sigma, self.z_sigma, self.P_0,
                                               self.update_interval)
            self.z_noise = None  # drawn on the device, step by step
            self._infos = [{} for _ in range(self.E)]
            self._infos_filled = []  # environments whose info dict holds the 'episode' entry of the previous step
            if self.episode_stats:
                self.ukf.rollout_episode_stats_enable()  # (accumulates from the rollout_reset of vector_reset on)
            if self.normalize:
                self._apply_normalize()  # (vector_reset below updates the observation statistics, VecNormalize.reset)
            self._old_reward = np.zeros(self.E)
        self.obs = self.vector_reset()

    # -- seeding / reset --------------------------------------------------------------------------------
    def seed(self, seeds=None):
        if seeds is None:
            seeds = [None] * self.E
        out = []
        for e in range(self.E):
            self.np_randoms[e], s = seeding.np_random(seeds[e])
            out.append(s)
        self.init_seeds = out
        return out

    def _draw(self, e):
        """The RNG draw sequence of SS2:206-221 for environment e."""
        x_true0, x_noise, self.z_noise[e] = draw_episode(self.np_randoms[e], self.orbits, self.m, self.n, self.x_sigma,
                                                          self.z_sigma)
        self.x_true0[e] = x_true0
        self.x_filter0[e] = x_true0 + x_noise
        self.i[e] = 0
        self.rewards_hist[e] = 0.0
        self.prev_spos_argmax[e] = 0  # argmax of the (all equal) sigma_pos[0]

    def _format_obs(self, obs12, idx=None):
        """The per-env observation in the layout config['obs_returned'] asks for (SS2:355-361).  obs12 = [E', m*12] rows
        (x [6], diag P [6] per RSO) of the environments `idx` (default: all); 'aer' evaluates az / el / range of every
        filter mean on the device with the env's own trans_matrix[i] (SS2:834-840) — environments at the same step index
        share one launch — and replaces NaN / inf by 0.001 as the reference does.  (rng='device' computes the 'aer' rows
        inside the step instead, k_obs_aer.)"""
        if self.obs_returned == 'flatten':
            return obs12
        o = np.asarray(obs12).reshape(-1, self.m, 12)
        if self.obs_returned != 'aer':
            return o
        idx = np.arange(self.E) if idx is None else np.asarray(idx)
        steps = np.minimum(self.i[idx], len(self.trans_matrix) - 1)
        out = np.empty((len(o), self.m, 4))
        for i in np.unique(steps):
            sel = np.where(steps == i)[0]
            out[sel, :, :3] = dynamics.hx_aer_erfa(o[sel, :, :6], self.trans_matrix[i], self.obs_lla, self.obs_itrs,
                                                   device=self._device)
        d = o[:, :, 6:]
        out[:, :, 3] = ((((d[:, :, 0] + d[:, :, 1]) + d[:, :, 2]) + d[:, :, 3]) + d[:, :, 4]) + d[:, :, 5]  # np.trace order
        return np.nan_to_num(out.reshape(len(o), self.m * 4), copy=False, nan=0.001, posinf=0.001, neginf=0.001)

    def _format_reward(self, rewards):
        # SS2:358-361: every layout but 'flatten' returns nan_to_num(reward, nan = +-inf = 0.5)
        return rewards if self.obs_returned == 'flatten' else np.nan_to_num(rewards, copy=False, nan=0.5, posinf=0.5, neginf=0.5)

    def _dev_views(self):
        if self._views is None:
            tv = self.ukf.torch_view
            self._views = {k: tv(f) for k, f in (("xt", F.F_X_TRUE), ("x", F.F_X_FILTER), ("P", F.F_P_FILTER),
                                                  ("status", F.F_STATUS), ("infl", F.F_INFLATIONS))}
        return self._views

    def vector_reset(self):
        if self.rng == 'device':
            self.ukf.rollout_reset()
            self.ukf.sync()
            self.i[:] = 0
            self.truncated = np.zeros(self.E, bool)
            return self._device_obs()
        for e in range(self.E):
            self._draw(e)
        self.ukf.reset(self.x_true0.reshape(self.N, 6), self.x_filter0.reshape(self.N, 6), self.P_0)
        self._epilogue_only()
        return self._format_obs(self.ukf.download(F.F_OBS).reshape(self.E, self.m * 12))

    def _epilogue_only(self):
        self.ukf.upload(F.F_TRANS_ENV, self.trans_matrix[self.i])
        self.ukf.step(None, F.STEP_EPILOGUE | F.STEP_M_PER_ENV)
        # greedy taskers of the fresh state; agent_shannon's history of a re-drawn environment starts at its P0 (step 0)
        self.ukf.upload(F.F_STEP_INDEX, self.i)
        self.ukf.env_reduce(step_index=-1)

    def _device_obs(self):
        """rng='device': the observations of the output block after a (partial) reset, in the configured layout and dtype
        (normalized float32 with config['normalize'])."""
        if self.normalize:
            rows = self.ukf.rollout_norm_io["obs"]
            return rows if self._obs_aer else self._format_obs(rows)
        if self._obs_aer:
            return self._io["obs_aer"].reshape(self.E, self.m * 4)
        return self._format_obs(self._io["obs"].reshape(self.E, self.m * 12).astype(self.obs_dtype, copy=False))

    def reset_at(self, e):
        """Reset environment e only (device state of the other environments is untouched).  rng='device': one
        ssa_ukf_rollout_reset_envs call (a new episode of the environment's own counter-based streams; with
        episode_stats its accumulation starts afresh); self.obs is refreshed and returned."""
        if self.rng == 'device':
            self.ukf.rollout_reset_envs([e])
            self.ukf.sync()
            self.i[e] = 0
            self.episodes[e] += 1
            self.obs = self._device_obs()
            return self.obs
        import torch
        self._draw(e)
        v = self._dev_views()
        lo, hi = e * self.m, (e + 1) * self.m
        dev = v["x"].device
        v["xt"][:, lo:hi] = torch.from_numpy(np.ascontiguousarray(self.x_true0[e].T)).to(dev)
        v["x"][:, lo:hi] = torch.from_numpy(np.ascontiguousarray(self.x_filter0[e].T)).to(dev)
        v["P"][:, lo:hi] = torch.from_numpy(self._P0_packed.copy()).to(dev)[:, None]
        v["status"][lo:hi] = 0
        v["infl"][lo:hi] = 0
        self.episodes[e] += 1

    # -- step ---------------------------------------------------------------------------------------------
    def set_tasker(self, agent, p=0.25):
        """Run `agent` inside the step graph (rng='device'): one of the nine functions of agents.py, or its name without
        the 'agent_' prefix ('visible_greedy', 'naive_random', ...); None returns to the caller's actions.  p is
        agent_visible_greedy_spoiled's probability of a random action.  Each step then picks every environment's action
        from the state the previous step left (the greedy block, the visibility flags), with the reference's
        distributions and counter-based random streams (include/ssa_ukf.h, ssa_ukf_rollout_tasker).  Any other callable
        raises ValueError: there is no host fallback."""
        if self.rng != 'device':
            raise ValueError("device taskers need rng='device'")
        if agent is None:
            tasker = F.TASKER_EXTERNAL
        elif isinstance(agent, str):
            if agent not in _TASKER_NAMES:
                raise ValueError(f"unknown agent {agent!r}; device taskers: {sorted(_TASKER_NAMES)}")
            tasker = _TASKER_NAMES[agent]
        else:
            tasker = next((k for f, k in _TASKERS.items() if f is agent), None)
        if tasker is None:
            raise ValueError(f"{agent!r} is not an agent of ssa_gym_b200.agents: the device runs only those")
        self.ukf.rollout_tasker(tasker, p)
        self.tasker = tasker

    def vector_step(self, actions=None):
        """One step of every environment with `actions` [E]; with a tasker set (set_tasker) the device picks them and
        `actions` must be None.  `last_actions` holds the actions the step took."""
        if self.tasker != F.TASKER_EXTERNAL:
            if actions is not None:
                raise ValueError("a device tasker is set (set_tasker): vector_step takes no actions")
            return self._device_step(None)
        if actions is None:
            raise ValueError("vector_step needs actions (or a device tasker, set_tasker)")
        actions = np.ascontiguousarray(actions, dtype=np.int32).reshape(self.E)
        assert np.all((actions >= 0) & (actions < self.m)), "invalid action"
        if self.rng == 'device':
            return self._device_step(actions)
        self.last_actions = actions.astype(np.int64)
        self.i += 1
        idx = self.i
        ar = np.arange(self.E)
        self.ukf.upload(F.F_ACTIONS, actions)
        self.ukf.upload(F.F_Z_NOISE, self.z_noise[ar, idx].reshape(self.N, 3))
        self.ukf.upload(F.F_TRANS_ENV, self.trans_matrix[idx])
        self.ukf.upload(F.F_STEP_INDEX, idx)
        flags = F.STEP_TRUTH | F.STEP_PREDICT | F.STEP_EPILOGUE | F.STEP_M_PER_ENV
        if self.update_interval == 1:
            flags |= F.STEP_UPDATE_ACT
        elif np.any(idx % self.update_interval == 0):
            # envs off their update step get an out-of-range action = "task nothing" (upd_object returns -1)
            a2 = np.where(idx % self.update_interval == 0, actions, -1).astype(np.int32)
            self.ukf.upload(F.F_ACTIONS, a2)
            flags |= F.STEP_UPDATE_ACT
        self.ukf.step(None, flags)
        self.ukf.env_reduce(step_index=-1)
        obs = self.ukf.download(F.F_OBS).reshape(self.E, self.m * 12)
        rewards = self.ukf.download(F.F_REWARD)
        dones = self.ukf.download(F.F_DONE).astype(bool)
        if self.reward_type == 'shaped':  # SS2:339-351 needs the reward history: finished on the host
            stats = self.ukf.download(F.F_ENV_STATS)
            for e in range(self.E):
                if stats[e, 0] > 5e6:
                    rewards[e] = 0
                elif stats[e, 0] < 3e4:
                    rewards[e] = 1 - np.sum(self.rewards_hist[e, :idx[e]])
                elif actions[e] == self.prev_spos_argmax[e]:
                    rewards[e] = 1 / self.n
                else:
                    rewards[e] = -1 / self.n
                self.rewards_hist[e, idx[e]] = rewards[e]
            self.prev_spos_argmax = stats[:, 2].astype(np.int64)
        infos = [{} for _ in range(self.E)]
        if self.terminal_observation and dones.any():
            max_dpos = (stats if self.reward_type == 'shaped' else self.ukf.download(F.F_ENV_STATS))[:, 0]
            for e, t in zip(np.flatnonzero(dones).tolist(), self._truncated(dones, max_dpos)[dones].tolist()):
                infos[e]["TimeLimit.truncated"] = t
        if self.auto_reset and dones.any():
            de = np.where(dones)[0]
            term = self._format_obs(obs[de], de)   # in the layout the caller sees, at the step index the episode ended on
            for k, e in enumerate(de):
                infos[e]["terminal_observation"] = np.array(term[k], copy=True)
                self.reset_at(int(e))
            self._epilogue_only()
            fresh = self.ukf.download(F.F_OBS).reshape(self.E, self.m * 12)
            obs[dones] = fresh[dones]
        self.obs = self._format_obs(obs)
        return self.obs, self._format_reward(rewards), dones, infos

    def _truncated(self, dones, max_dpos):
        """done raised by the step limit alone (gym's TimeLimit rule; the device's rule, include/ssa_ukf.h): a lost or
        successful last step is a termination, 'trinary' ends at the step limit only."""
        if self.reward_type == 'trinary':
            return dones.copy()
        return dones & ~((max_dpos > 5e6) | (max_dpos < 3e4))

    def _device_step(self, actions):
        """rng='device': the whole step (noise, UKF, reward / done, auto-reset, fresh obs, greedy taskers) is one
        H2D copy of the actions, one CUDA-graph launch and one D2H copy (ssa_ukf_rollout_step).  The returned obs
        is a VIEW of the handle's pinned output block: it is overwritten by the next step.  actions None: a device
        tasker picks them, and the step copies them back into the same block."""
        io = self._io
        if actions is not None:
            io["actions"][:] = actions
        f32 = self.obs_dtype == np.float32
        self.ukf.rollout_step(self.auto_reset, obs_f32=f32, obs_aer=self._obs_aer)
        self.ukf.sync()
        self.last_actions = io["actions"].astype(np.int64)
        dones = io["done"].astype(bool)
        self.truncated = io["truncated"].astype(bool)
        rewards = io["reward"].copy()
        self.i += 1
        if self.auto_reset:
            self.i[dones] = 0
            self.episodes[dones] += 1
        if self.normalize:
            self._old_reward = self._format_reward(rewards)
            rewards = self.ukf.rollout_norm_io["reward"].copy()
            self.obs = self._device_obs()
        elif self._obs_aer:
            self.obs = io["obs_aer"].reshape(self.E, self.m * 4)
        else:
            self.obs = self._format_obs(io["obs_f32" if f32 else "obs"].reshape(self.E, self.m * 12))
        # E dicts allocated once (4096 dict constructions cost 100 us): empty, except on the step an episode finished
        infos = self._infos
        for e in self._infos_filled:
            infos[e].clear()
        self._infos_filled = []
        if (self.episode_stats or self.terminal_observation) and dones.any():
            de = np.flatnonzero(dones).tolist()
            if self.episode_stats:
                for e, ep in zip(de, episode_infos(self.ukf.rollout_episode_stats(de))):
                    infos[e]["episode"] = ep
            if self.terminal_observation:
                for e, t in zip(de, self.truncated[de].tolist()):
                    infos[e]["TimeLimit.truncated"] = t
                if self.auto_reset:  # one download of the final rows, in the layout and dtype of the observations
                    if self.normalize:  # (normalized with the step's statistics, as VecNormalize does)
                        rows = self.ukf.rollout_terminal_obs_norm(de)
                        term = rows if self._obs_aer else self._format_obs(rows)
                    else:
                        rows = self.ukf.rollout_terminal_obs(de)
                        term = rows if self._obs_aer else self._format_obs(rows.astype(self.obs_dtype, copy=False))
                    for k, e in enumerate(de):
                        infos[e]["terminal_observation"] = term[k]
            self._infos_filled = de
        return self.obs, (rewards if self.normalize else self._format_reward(rewards)), dones, infos

    # -- running normalization (config['normalize']; Stable-Baselines3 VecNormalize's names) -------------------------
    def _need_normalize(self):
        if not self.normalize:
            raise ValueError("normalization is off: construct with config['normalize'] = True (rng='device')")

    def _apply_normalize(self):
        layout = F.NORM_OBS_AER if self._obs_aer else F.NORM_OBS_ROWS_F32 if self.obs_dtype == np.float32 else F.NORM_OBS_ROWS
        self.ukf.rollout_normalize(obs_layout=layout, reward_nan_to_num=self.obs_returned != 'flatten', **self._norm_kw)

    @property
    def training(self):
        """VecNormalize.training: with False the statistics and the returns stay as they are (a device flag: setting it
        re-captures nothing)."""
        self._need_normalize()
        return self._norm_kw["training"]

    @training.setter
    def training(self, value):
        self._need_normalize()
        self._norm_kw["training"] = bool(value)
        self._apply_normalize()

    def get_original_obs(self):
        """The observations of the last step or reset before normalization, in the layout and dtype they would have without
        it (downloaded from the device on demand)."""
        self._need_normalize()
        if self._obs_aer:
            return self.ukf.download(F.F_ROLLOUT_OBS_AER).reshape(self.E, self.m * 4)
        return self._format_obs(self.ukf.download(F.F_ROLLOUT_OBS).reshape(self.E, self.m * 12).astype(self.obs_dtype, copy=False))

    def get_original_reward(self):
        """The rewards of the last step before normalization (after the layout's nan_to_num)."""
        self._need_normalize()
        return self._old_reward.copy()

    def normalizer_state(self):
        """{'obs_mean' [F], 'obs_var' [F], 'obs_count', 'ret_mean', 'ret_var', 'ret_count', 'returns' [E]}: VecNormalize's
        obs_rms, ret_rms and returns, for a checkpoint or an evaluation env (load_normalizer_state)."""
        self._need_normalize()
        return self.ukf.rollout_norm_state()

    def load_normalizer_state(self, state):
        """Restore a normalizer_state() dict; `training` keeps its setting.  The next step normalizes with it."""
        self._need_normalize()
        self.ukf.rollout_load_norm_state(state)

    # -- device-resident consumer (a policy on the same GPU): no host copies, nothing synchronises -------------------
    def device_views(self):
        """Zero-copy torch tensors over the episodic mode's device buffers: 'actions' int32 [E] (INPUT of
        vector_step_device; with a device tasker its output, the actions the step took), 'obs' float64 [E, m*12] ([E, m*4] for obs_returned='aer'), 'reward' float64 [E], 'done' uint8
        [E], 'greedy' int32 [E, taskers], 'truncated' uint8 [E] (done raised by the step limit alone) and 'terminal_obs'
        float64 [E, m*12] ([E, m*4] for 'aer'): with auto-reset, the final observation of each environment's last finished
        episode, valid after a step whose 'done' is set for it (a PPO on the device bootstraps V(terminal_obs) where
        done & truncated).
        With config['episode_stats']: 'episode_stats' float64 [E, EPISODE_STATS_DOUBLES], the record of each environment's
        last finished episode (layout: include/ssa_ukf.h; episode_info turns a row into the infos entry), valid after a
        step whose 'done' is set for it.
        With config['normalize']: 'obs_norm' float32 [E, F] (F = m*12, or m*4 for 'aer'), 'reward_norm' float64 [E] and
        'terminal_obs_norm' float32 [E, F] (with auto-reset, valid like 'terminal_obs').
        The outputs are overwritten by every step; they are valid in stream order on the stream the step runs on."""
        assert self.rng == 'device', "device views exist in the device-resident episodic mode (rng='device')"
        if getattr(self, "_views", None) is None:
            u = self.ukf
            obs = (u.torch_view(F.F_ROLLOUT_OBS_AER).view(self.E, self.m * 4) if self._obs_aer else
                   u.torch_view(F.F_ROLLOUT_OBS).view(self.E, self.m * 12))
            term = u.torch_view(F.F_ROLLOUT_TERMINAL_OBS).view(-1)
            term = term[:self.N * 4].view(self.E, self.m * 4) if self._obs_aer else term.view(self.E, self.m * 12)
            self._views = {"actions": u.torch_view(F.F_ROLLOUT_ACTIONS), "obs": obs,
                           "reward": u.torch_view(F.F_ROLLOUT_REWARD), "done": u.torch_view(F.F_ROLLOUT_DONE),
                           "greedy": u.torch_view(F.F_ROLLOUT_GREEDY), "truncated": u.torch_view(F.F_ROLLOUT_TRUNCATED),
                           "terminal_obs": term}
            if self.episode_stats:
                self._views["episode_stats"] = u.torch_view(F.F_ROLLOUT_EPISODE_STATS)
            if self.normalize:
                self._views.update({"obs_norm": u.torch_view(F.F_ROLLOUT_OBS_NORM),
                                    "reward_norm": u.torch_view(F.F_ROLLOUT_REWARD_NORM),
                                    "terminal_obs_norm": u.torch_view(F.F_ROLLOUT_TERMINAL_OBS_NORM)})
        return self._views

    def vector_step_device(self, stream=None):
        """One vectorised env step whose actions are ALREADY in device_views()['actions'] (written by a device-side
        policy on the same stream) and whose obs / reward / done stay on the device: one CUDA-graph launch, no H2D, no D2H,
        no synchronisation (the reference hands every observation to the learner process through the host, SURVEY 3.4).
        The host mirrors (self.i, self.episodes) are not maintained in this mode."""
        assert self.rng == 'device'
        self.ukf.rollout_step(self.auto_reset, stream=stream, device_io=True, obs_aer=self._obs_aer,
                              obs_f32=self.normalize and self.obs_dtype == np.float32)  # (the normalization's layout)
        return self.device_views()

    # -- device taskers --------------------------------------------------------------------------------------
    def greedy_actions(self, tasker=F.TASKER_VISIBLE_GREEDY):
        """agents.py argmax rules evaluated on the device for every env (valid after a step / reset); where the
        reference would fall back to `env.action_space.sample()` the env's own Discrete space is sampled."""
        if self.rng == 'device':  # already part of the step's output block
            a = self._io["greedy"][:, tasker].astype(np.int64)
        else:
            self.ukf.upload(F.F_STEP_INDEX, self.i)
            self.ukf.env_reduce(step_index=-1)
            a = self.ukf.download(F.F_GREEDY)[:, tasker].astype(np.int64)
        for e in np.where(a < 0)[0]:
            a[e] = self.action_spaces[e].sample()
        return a

    def visible(self):
        return self.ukf.download(F.F_VISIBLE).reshape(self.E, self.m).astype(bool)

    def get_unwrapped(self):
        return [self]

    def close(self):
        if self.ukf is not None:
            self.ukf.close()
            self.ukf = None
