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
vector_step in host mode against 0.45 ms in device mode).
"""
import numpy as np

from . import _lib, dynamics
from .episode import draw_episode
from .gym_shim import seeding, spaces
from .transformations import arcsec2rad, default_eops, deg2rad, gcrs2irts_matrix_b, lla2ecef, load_eop_c04, time_table
from .ukf import BatchedUKF, Q_discrete_white_noise_block

F = _lib


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
        self.seed(seeds)
        if self.rng == 'device':
            if self.reward_type == 'shaped':
                raise ValueError("rng='device' does not support the 'shaped' reward (host-side history); use rng='host'")
            keys = np.array([int(s_) & 0xFFFFFFFFFFFFFFFF for s_ in self.init_seeds], dtype=np.uint64)
            self._io = self.ukf.rollout_config(self.orbits, self.trans_matrix, keys, self.x_sigma, self.z_sigma, self.P_0,
                                               self.update_interval)
            self.z_noise = None  # drawn on the device, step by step
            self._infos = [{} for _ in range(self.E)]
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
        share one launch — and replaces NaN / inf by 0.001 as the reference does."""
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
            return self._format_obs(self._io["obs"].reshape(self.E, self.m * 12).astype(self.obs_dtype, copy=False))
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

    def reset_at(self, e):
        """Reset environment e only (device state of the other environments is untouched)."""
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
    def vector_step(self, actions):
        actions = np.ascontiguousarray(actions, dtype=np.int32).reshape(self.E)
        assert np.all((actions >= 0) & (actions < self.m)), "invalid action"
        if self.rng == 'device':
            return self._device_step(actions)
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

    def _device_step(self, actions):
        """rng='device': the whole step (noise, UKF, reward / done, auto-reset, fresh obs, greedy taskers) is one
        H2D copy of the actions, one CUDA-graph launch and one D2H copy (ssa_ukf_rollout_step).  The returned obs
        is a VIEW of the handle's pinned output block: it is overwritten by the next step."""
        io = self._io
        io["actions"][:] = actions
        f32 = self.obs_dtype == np.float32
        self.ukf.rollout_step(self.auto_reset, obs_f32=f32)
        self.ukf.sync()
        dones = io["done"].astype(bool)
        rewards = io["reward"].copy()
        self.i += 1
        if self.auto_reset:
            self.i[dones] = 0
            self.episodes[dones] += 1
        self.obs = self._format_obs(io["obs_f32" if f32 else "obs"].reshape(self.E, self.m * 12))
        return self.obs, self._format_reward(rewards), dones, self._infos  # E empty dicts, allocated once (4096 dict constructions cost 100 us)

    # -- device-resident consumer (a policy on the same GPU): no host copies, nothing synchronises -------------------
    def device_views(self):
        """Zero-copy torch tensors over the episodic mode's device buffers: 'actions' int32 [E] (INPUT of
        vector_step_device), 'obs' float64 [E, m*12], 'reward' float64 [E], 'done' uint8 [E], 'greedy' int32 [E, taskers].
        The outputs are overwritten by every step; they are valid in stream order on the stream the step runs on."""
        assert self.rng == 'device', "device views exist in the device-resident episodic mode (rng='device')"
        if getattr(self, "_views", None) is None:
            u = self.ukf
            self._views = {"actions": u.torch_view(F.F_ROLLOUT_ACTIONS), "obs": u.torch_view(F.F_ROLLOUT_OBS).view(self.E, self.m * 12),
                           "reward": u.torch_view(F.F_ROLLOUT_REWARD), "done": u.torch_view(F.F_ROLLOUT_DONE),
                           "greedy": u.torch_view(F.F_ROLLOUT_GREEDY)}
        return self._views

    def vector_step_device(self, stream=None):
        """One vectorised env step whose actions are ALREADY in device_views()['actions'] (written by a device-side
        policy on the same stream) and whose obs / reward / done stay on the device: one CUDA-graph launch, no H2D, no D2H,
        no synchronisation (the reference hands every observation to the learner process through the host, SURVEY 3.4).
        The host mirrors (self.i, self.episodes) are not maintained in this mode."""
        assert self.rng == 'device'
        self.ukf.rollout_step(self.auto_reset, stream=stream, device_io=True)
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
