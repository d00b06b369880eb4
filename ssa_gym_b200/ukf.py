"""Host-side mirror of the filter objects of the reference, backed by the CUDA library.

The reference keeps one filterpy `UnscentedKalmanFilter` per RSO (ssa_tasker_simple_2.py:211-218) and
loops over them in Python.  `BatchedUKF` owns ALL filters of all environments as one device-resident
struct-of-arrays and advances them with one fused kernel launch per step through the C ABI
(include/ssa_ukf.h).  Weights, Q and the observer constants are computed here on the host with the
same Python/numpy expressions filterpy and the reference use, so the device receives bit-identical
constants (SURVEY.md H1: sum(Wm) != 1 must be reproduced, not "fixed").
"""
import ctypes

import numpy as np

from . import _lib
from .transformations import lla2ecef, trans_uvw_ecef


def merwe_weights(n=6, alpha=1e-4, beta=2.0, kappa=-3.0):
    """filterpy MerweScaledSigmaPoints._compute_weights, same expression order."""
    lambda_ = alpha ** 2 * (n + kappa) - n
    c = .5 / (n + lambda_)
    Wc = np.full(2 * n + 1, c)
    Wm = np.full(2 * n + 1, c)
    Wc[0] = lambda_ / (n + lambda_) + (1 - alpha ** 2 + beta)
    Wm[0] = lambda_ / (n + lambda_)
    return Wm, Wc, lambda_ + n


def Q_discrete_white_noise_block(dt, var, block_size=3):
    """filterpy.common.Q_discrete_white_noise(dim=2, dt, var, block_size=3, order_by_dim=False) (SS2:110)."""
    Q2 = np.array([[.25 * dt ** 4, .5 * dt ** 3], [.5 * dt ** 3, dt ** 2]], dtype=float)
    out = np.zeros((2 * block_size, 2 * block_size))
    for i in range(2):
        for j in range(2):
            out[i * block_size:(i + 1) * block_size, j * block_size:(j + 1) * block_size] = np.eye(block_size) * Q2[i, j]
    return out * var


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _host_array(ptr, ctype, shape):
    """numpy view of `shape` over host memory the handle owns (its pinned blocks), at a ctypes pointer."""
    n = int(np.prod(shape))
    return np.ctypeslib.as_array(ctypes.cast(ptr, ctypes.POINTER(ctype)), shape=(n,)).reshape(shape)


class _CudaArray:
    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (ptr, False), "version": 2}


def _device_tensor(ptr, shape, dtype, device):
    """Zero-copy torch tensor of `shape` over device memory the handle owns, at address ptr on cuda:device."""
    import torch
    typestr = {np.dtype(np.float64): "<f8", np.dtype(np.float32): "<f4", np.dtype(np.int32): "<i4",
               np.dtype(np.uint8): "|u1"}[np.dtype(dtype)]
    return torch.as_tensor(_CudaArray(ptr, shape, typestr), device=torch.device("cuda", device))


class BatchedUKF:
    """N = n_envs * m unscented Kalman filters resident on one GPU.

    Parameters mirror the reference's env_config (envs/__init__.py:23-28)."""

    def __init__(self, n_envs, m, dt, Q, R, obs_lla, obs_limit_rad, alpha=1e-4, beta=2.0, kappa=-3.0,
                 obs_type="aer", reward_type="jones", n_steps=480, resample_after_predict=True, device=0):
        self.lib = _lib.require_gpu()
        self.n_envs, self.m, self.N = int(n_envs), int(m), int(n_envs) * int(m)
        self.device = int(device)
        Wm, Wc, lam_plus_n = merwe_weights(6, alpha, beta, kappa)
        self.Wm, self.Wc, self.lam_plus_n = Wm, Wc, lam_plus_n
        cfg = _lib.SsaUkfCfg()
        cfg.abi_version = _lib.SSA_UKF_ABI_VERSION
        cfg.n_objects, cfg.n_envs, cfg.m = self.N, self.n_envs, self.m
        cfg.obs_type = {"aer": _lib.OBS_AER, "xyz": _lib.OBS_XYZ}[obs_type]
        cfg.resample_after_predict = 1 if resample_after_predict else 0
        cfg.reward_type = {"jones": _lib.REWARD_JONES, "trinary": _lib.REWARD_TRINARY, "shaped": _lib.REWARD_SHAPED}[reward_type]
        cfg.n_steps = int(n_steps)
        cfg.dt = float(dt)
        cfg.lam_plus_n = float(lam_plus_n)
        Q = np.asarray(Q, dtype=np.float64).reshape(6, 6)
        R = np.asarray(R, dtype=np.float64)
        if R.ndim == 1:  # tests.py:162 passes a 1-D R: `P += noise_cov` broadcasts it over the rows
            R = np.tile(R, (3, 1))
        R = R.reshape(3, 3)
        obs_lla = np.asarray(obs_lla, dtype=np.float64)
        self.obs_lla = obs_lla
        self.obs_itrs = lla2ecef(obs_lla)
        T = trans_uvw_ecef(obs_lla[0], obs_lla[1])
        for i in range(13):
            cfg.Wm[i], cfg.Wc[i] = Wm[i], Wc[i]
        for i, v in enumerate(Q.ravel()):
            cfg.Q[i] = v
        for i, v in enumerate(R.ravel()):
            cfg.R[i] = v
        for i in range(3):
            cfg.obs_itrs[i] = self.obs_itrs[i]
        for i, v in enumerate(np.asarray(T, dtype=np.float64).ravel()):
            cfg.T[i] = v
        cfg.obs_limit = float(obs_limit_rad)
        self.cfg = cfg
        self.Q, self.R, self.T = Q, R, T
        h = ctypes.c_void_p()
        _lib.check(self.lib.ssa_ukf_create(ctypes.byref(cfg), self.device, ctypes.byref(h)), "ssa_ukf_create")
        self.h = h
        self.ld = self.lib.ssa_ukf_ld(h)
        self._shapes = {
            _lib.F_X_TRUE: ((self.N, 6), np.float64), _lib.F_X_FILTER: ((self.N, 6), np.float64),
            _lib.F_P_FILTER: ((self.N, 6, 6), np.float64), _lib.F_OBS: ((self.N, 12), np.float64),
            _lib.F_DELTA_POS: ((self.N,), np.float64), _lib.F_DELTA_VEL: ((self.N,), np.float64),
            _lib.F_SIGMA_POS: ((self.N,), np.float64), _lib.F_SIGMA_VEL: ((self.N,), np.float64),
            _lib.F_TRACE: ((self.N,), np.float64), _lib.F_Z_TRUE: ((self.N, 3), np.float64),
            _lib.F_Y: ((self.N, 3), np.float64), _lib.F_S: ((self.N, 3, 3), np.float64),
            _lib.F_SIGMAS_H: ((self.N, 13, 3), np.float64), _lib.F_Z_NOISE: ((self.N, 3), np.float64),
            _lib.F_VISIBLE: ((self.N,), np.uint8), _lib.F_UPDATED: ((self.N,), np.uint8),
            _lib.F_STATUS: ((self.N,), np.int32), _lib.F_INFLATIONS: ((self.N,), np.int32),
            _lib.F_ACTIONS: ((self.n_envs,), np.int32), _lib.F_REWARD: ((self.n_envs,), np.float64),
            _lib.F_DONE: ((self.n_envs,), np.uint8), _lib.F_GREEDY: ((self.n_envs, _lib.N_TASKERS), np.int32),
            _lib.F_SCORES: ((self.N, 6), np.float64), _lib.F_TRANS_ENV: ((self.n_envs, 3, 3), np.float64),
            _lib.F_STEP_INDEX: ((self.n_envs,), np.int32), _lib.F_ENV_STATS: ((self.n_envs, 4), np.float64),
            _lib.F_DIAG: ((self.N, 2), np.float64), _lib.F_INNOV_FLAGS: ((self.N,), np.uint8),
            _lib.F_CATALOG_STATS: ((5,), np.float64), _lib.F_ROLLOUT_OBS: ((self.N, 12), np.float64),
            _lib.F_ROLLOUT_REWARD: ((self.n_envs,), np.float64), _lib.F_ROLLOUT_ACTIONS: ((self.n_envs,), np.int32),
            _lib.F_ROLLOUT_DONE: ((self.n_envs,), np.uint8), _lib.F_ROLLOUT_GREEDY: ((self.n_envs, _lib.N_TASKERS), np.int32),
            _lib.F_ROLLOUT_OBS_AER: ((self.N, 4), np.float64),
            _lib.F_ROLLOUT_EPISODE_STATS: ((self.n_envs, _lib.EPISODE_STATS_DOUBLES), np.float64),
            _lib.F_ROLLOUT_TERMINAL_OBS: ((self.N, 12), np.float64), _lib.F_ROLLOUT_TRUNCATED: ((self.n_envs,), np.uint8),
        }

    # -- lifetime ---------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "h", None):
            self.lib.ssa_ukf_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- state ------------------------------------------------------------------------------------
    def reset(self, x_true, x_filter, P0, stream=None):
        x_true = np.ascontiguousarray(x_true, dtype=np.float64).reshape(self.N, 6)
        x_filter = np.ascontiguousarray(x_filter, dtype=np.float64).reshape(self.N, 6)
        P0 = np.ascontiguousarray(P0, dtype=np.float64)
        per_obj = 1 if (P0.size == self.N * 36 and P0.size != 36) else 0
        if per_obj:
            P0 = P0.reshape(self.N, 36)
        else:
            P0 = P0.reshape(36)
        _lib.check(self.lib.ssa_ukf_reset(self.h, _ptr(x_true), _ptr(x_filter), _ptr(P0), per_obj, stream), "ssa_ukf_reset")

    def upload(self, field, arr, stream=None):
        shape, dtype = self._shapes[field]
        arr = np.ascontiguousarray(arr, dtype=dtype).reshape(shape)
        _lib.check(self.lib.ssa_ukf_upload(self.h, field, _ptr(arr), arr.nbytes, stream), "ssa_ukf_upload")
        return arr  # keep alive until the stream has consumed it (async H2D)

    def download(self, field, out=None, stream=None):
        shape, dtype = self._shapes[field]
        if out is None:
            out = np.empty(shape, dtype=dtype)
        _lib.check(self.lib.ssa_ukf_download(self.h, field, _ptr(out), out.nbytes, stream), "ssa_ukf_download")
        return out

    def device_ptr(self, field):
        p, n = ctypes.c_void_p(), ctypes.c_size_t()
        _lib.check(self.lib.ssa_ukf_device_ptr(self.h, field, ctypes.byref(p), ctypes.byref(n)), "ssa_ukf_device_ptr")
        return p.value, n.value

    def torch_view(self, field):
        """Zero-copy torch tensor over a handle-owned device buffer (AoS fields keep their host shape;
        SoA fields X_TRUE / X_FILTER / P_FILTER come back as [rows, ld])."""
        ptr, _ = self.device_ptr(field)
        shape, dtype = self._shapes[field]
        if field in (_lib.F_X_TRUE, _lib.F_X_FILTER):
            shape = (6, self.ld)
        elif field == _lib.F_P_FILTER:
            shape = (21, self.ld)
        return _device_tensor(ptr, shape, dtype, self.device)

    # -- the hot path -----------------------------------------------------------------------------
    def step(self, M, flags, stream=None):
        M = np.ascontiguousarray(M, dtype=np.float64).reshape(9) if M is not None else None
        _lib.check(self.lib.ssa_ukf_step(self.h, _ptr(M) if M is not None else None, int(flags), stream), "ssa_ukf_step")

    def step_profile(self, M, flags, stream=None):
        """One step with CUDA events around each kernel; returns ms per kernel [factor, fx, ut, hx, update]."""
        M = np.ascontiguousarray(M, dtype=np.float64).reshape(9)
        ms = (ctypes.c_double * 5)()
        _lib.check(self.lib.ssa_ukf_step_profile(self.h, _ptr(M), int(flags), stream, ms), "ssa_ukf_step_profile")
        return np.array(ms[:])

    def step_host(self, M, flags, z_noise=None, obs_out=None, dpos_out=None, status_out=None, actions=None, stream=None):
        """Asynchronous step with host buffers (pinned numpy arrays): H2D of the inputs, kernels, D2H of the
        results, double-buffered and overlapped across consecutive calls.  Call host_join()+sync() before reading."""
        M = np.ascontiguousarray(M, dtype=np.float64).reshape(9)
        self._keep = (M, z_noise, actions)  # keep host inputs alive until consumed
        _lib.check(self.lib.ssa_ukf_step_host(self.h, _ptr(M), int(flags), _ptr(actions) if actions is not None else None,
                                              _ptr(z_noise) if z_noise is not None else None,
                                              _ptr(obs_out) if obs_out is not None else None,
                                              _ptr(dpos_out) if dpos_out is not None else None,
                                              _ptr(status_out) if status_out is not None else None, stream), "ssa_ukf_step_host")

    def host_join(self, stream=None):
        _lib.check(self.lib.ssa_ukf_host_join(self.h, stream), "ssa_ukf_host_join")

    def host_io(self):
        """The handle's pinned host I/O blocks as numpy views, one dict per pipeline parity:
        inputs 'z_noise' [N,3], 'M' [9], 'actions' [E]; outputs 'obs' [N,12], 'delta_pos' [N], 'status' [N]."""
        if getattr(self, "_io", None) is None:
            N, E = self.N, self.n_envs
            io = []
            for b in range(2):
                ptrs = [ctypes.c_void_p() for _ in range(6)]
                _lib.check(self.lib.ssa_ukf_host_io(self.h, b, *[ctypes.byref(q) for q in ptrs]), "ssa_ukf_host_io")
                io.append({"z_noise": _host_array(ptrs[0], ctypes.c_double, (N, 3)), "M": _host_array(ptrs[1], ctypes.c_double, (9,)),
                           "actions": _host_array(ptrs[2], ctypes.c_int32, (E,)), "obs": _host_array(ptrs[3], ctypes.c_double, (N, 12)),
                           "delta_pos": _host_array(ptrs[4], ctypes.c_double, (N,)), "status": _host_array(ptrs[5], ctypes.c_int32, (N,))})
            self._io = io
            self._parity_out = ctypes.c_int(0)
        return self._io

    def host_stats(self, parity):
        """Reward terms (SSA_F_CATALOG_STATS layout, 5 doubles) of the pinned steps of `parity`: (numpy view of the
        pinned host copy - valid after host_join() + sync -, device pointer of the slot).  Needs catalog_stats() once."""
        hp, dp = ctypes.c_void_p(), ctypes.c_void_p()
        _lib.check(self.lib.ssa_ukf_host_stats(self.h, int(parity), ctypes.byref(hp), ctypes.byref(dp)), "ssa_ukf_host_stats")
        return _host_array(hp, ctypes.c_double, (5,)), dp.value

    def host_stats_torch(self, parity):
        """Zero-copy torch view [5] of the device slot of host_stats(parity) (input of an NCCL gather)."""
        _, dp = self.host_stats(parity)
        return _device_tensor(dp, (5,), np.float64, self.device)

    def step_pinned(self, flags, stream=None):
        """Pipelined step on the pinned blocks of host_io(): fill host_io()[b] of the parity this call will use
        (0, 1, 0, ... from the first call; `next_parity`), call, read host_io()[b] outputs after host_join()+sync.
        One H2D copy, one graph launch, one D2H copy per call.  Returns the parity used."""
        self.host_io()
        _lib.check(self.lib.ssa_ukf_step_pinned(self.h, int(flags), stream, ctypes.byref(self._parity_out)), "ssa_ukf_step_pinned")
        self._next_parity = self._parity_out.value ^ 1
        return self._parity_out.value

    # -- device-resident episodic mode (vectorised reset, counter-based RNG) --------------------------------
    def rollout_config(self, orbits, trans_table, seeds, x_sigma, z_sigma, P0, update_interval=1):
        orbits = np.ascontiguousarray(orbits, dtype=np.float64).reshape(-1, 6)
        table = np.ascontiguousarray(trans_table, dtype=np.float64).reshape(-1, 9)
        seeds = np.ascontiguousarray(seeds, dtype=np.uint64).reshape(self.n_envs)
        xs = np.ascontiguousarray(x_sigma, dtype=np.float64).reshape(6)
        zs = np.ascontiguousarray(z_sigma, dtype=np.float64).reshape(3)
        P0 = np.ascontiguousarray(P0, dtype=np.float64).reshape(36)
        _lib.check(self.lib.ssa_ukf_rollout_config(self.h, _ptr(orbits), len(orbits), _ptr(table), len(table), _ptr(seeds),
                                                   _ptr(xs), _ptr(zs), _ptr(P0), int(update_interval)), "ssa_ukf_rollout_config")
        ptrs = [ctypes.c_void_p() for _ in range(5)]
        _lib.check(self.lib.ssa_ukf_rollout_io(self.h, *[ctypes.byref(q) for q in ptrs]), "ssa_ukf_rollout_io")
        N, E = self.N, self.n_envs
        self.rollout_io = {"actions": _host_array(ptrs[0], ctypes.c_int32, (E,)), "obs": _host_array(ptrs[1], ctypes.c_double, (N, 12)),
                           "reward": _host_array(ptrs[2], ctypes.c_double, (E,)),
                           "greedy": _host_array(ptrs[3], ctypes.c_int32, (E, _lib.N_TASKERS)),
                           "done": _host_array(ptrs[4], ctypes.c_uint8, (E,))}
        h32, d32 = ctypes.c_void_p(), ctypes.c_void_p()
        _lib.check(self.lib.ssa_ukf_rollout_obs_f32(self.h, ctypes.byref(h32), ctypes.byref(d32)), "ssa_ukf_rollout_obs_f32")
        self.rollout_io["obs_f32"] = _host_array(h32, ctypes.c_float, (N, 12))  # filled by rollout_step(obs_f32=True)
        self.rollout_obs_f32_device = d32.value
        ha, da = ctypes.c_void_p(), ctypes.c_void_p()
        _lib.check(self.lib.ssa_ukf_rollout_obs_aer(self.h, ctypes.byref(ha), ctypes.byref(da)), "ssa_ukf_rollout_obs_aer")
        self.rollout_io["obs_aer"] = _host_array(ha, ctypes.c_double, (N, 4))  # filled by rollout_reset and rollout_step(obs_aer=True)
        ht = ctypes.c_void_p()
        _lib.check(self.lib.ssa_ukf_rollout_truncated(self.h, ctypes.byref(ht), None), "ssa_ukf_rollout_truncated")
        self.rollout_io["truncated"] = _host_array(ht, ctypes.c_uint8, (E,))  # done raised by the step limit alone
        self._term_w = 12
        self.rollout_norm_io = None  # (a new configuration runs without normalization, rollout_normalize)
        return self.rollout_io

    def rollout_reset(self, stream=None):
        _lib.check(self.lib.ssa_ukf_rollout_reset(self.h, stream), "ssa_ukf_rollout_reset")

    def rollout_step(self, auto_reset=True, stream=None, device_io=False, obs_f32=False, obs_aer=False):
        """obs_f32: the observations leave the device as float32 (rollout_io['obs_f32']; the float64 block is not copied).
        obs_aer: the step also computes the 'aer' observation [N, 4] (rollout_io['obs_aer'], device field F_ROLLOUT_OBS_AER),
        which leaves the device instead of the float64 block.  The two exclude each other."""
        mode = (1 if auto_reset else 0) | (_lib.ROLLOUT_DEVICE_IO if device_io else 0) | (_lib.ROLLOUT_OBS_F32 if obs_f32 else 0) | \
            (_lib.ROLLOUT_OBS_AER if obs_aer else 0)
        _lib.check(self.lib.ssa_ukf_rollout_step(self.h, mode, stream), "ssa_ukf_rollout_step")
        if auto_reset:
            self._term_w = 4 if obs_aer else 12  # the layout of the final observations this step records

    def rollout_tasker(self, tasker, spoil_p=0.25):
        """Pick every environment's action inside the step graph (a TASKER_* id, include/ssa_ukf.h), TASKER_EXTERNAL for
        the caller's actions.  spoil_p is TASKER_VISIBLE_GREEDY_SPOILED's probability of a random action.  After
        rollout_config (which restores TASKER_EXTERNAL); the taken actions are in rollout_io['actions'] after a step."""
        _lib.check(self.lib.ssa_ukf_rollout_tasker(self.h, int(tasker), float(spoil_p)), "ssa_ukf_rollout_tasker")

    def rollout_episode_stats_enable(self):
        """Accumulate per-episode statistics inside the step graph from the next rollout_reset on (after rollout_config,
        which turns them off again).  Records: rollout_episode_stats, or the device field F_ROLLOUT_EPISODE_STATS."""
        _lib.check(self.lib.ssa_ukf_rollout_episode_stats_enable(self.h), "ssa_ukf_rollout_episode_stats_enable")

    def rollout_episode_stats(self, envs, stream=None):
        """The records [len(envs), EPISODE_STATS_DOUBLES] of the environments `envs` (layout: include/ssa_ukf.h); blocks
        until copied.  A row is that of the episode that ended on the last step whose done flag was set for it."""
        envs = np.ascontiguousarray(envs, dtype=np.int32).reshape(-1)
        out = np.empty((len(envs), _lib.EPISODE_STATS_DOUBLES))
        _lib.check(self.lib.ssa_ukf_rollout_episode_stats_download(self.h, _ptr(envs), len(envs), _ptr(out), stream),
                   "ssa_ukf_rollout_episode_stats_download")
        return out

    def rollout_terminal_obs(self, envs, stream=None):
        """The final observations [len(envs), m*12] ([len(envs), m*4] after steps with obs_aer) of the environments
        `envs`: their observation rows on the last auto-reset step whose done flag was set for them, before the re-draw
        (include/ssa_ukf.h).  Blocks until copied."""
        envs = np.ascontiguousarray(envs, dtype=np.int32).reshape(-1)
        out = np.empty((len(envs), self.m * self._term_w))
        _lib.check(self.lib.ssa_ukf_rollout_terminal_obs_download(self.h, _ptr(envs), len(envs), _ptr(out), stream),
                   "ssa_ukf_rollout_terminal_obs_download")
        return out

    def rollout_reset_envs(self, envs, stream=None):
        """rollout_reset of the environments `envs` only: re-drawn, refreshed, their episode statistics restarted; the
        others keep their state and outputs.  rollout_io is valid after a sync."""
        envs = np.ascontiguousarray(envs, dtype=np.int32).reshape(-1)
        _lib.check(self.lib.ssa_ukf_rollout_reset_envs(self.h, _ptr(envs), len(envs), stream), "ssa_ukf_rollout_reset_envs")

    def rollout_normalize(self, on=True, obs_layout=_lib.NORM_OBS_ROWS, reward_nan_to_num=False, training=True, norm_obs=True,
                          norm_reward=True, clip_obs=10.0, clip_reward=10.0, gamma=0.99, epsilon=1e-8):
        """Stable-Baselines3's VecNormalize inside the step graph (include/ssa_ukf.h, ssa_ukf_rollout_normalize); on=False
        turns it off.  obs_layout (NORM_OBS_*) must match the steps' obs_f32 / obs_aer.  After rollout_config (which
        turns it off).  rollout_norm_io: pinned host views of the normalized obs [E, F] float32 and rewards [E]."""
        if not on:
            _lib.check(self.lib.ssa_ukf_rollout_normalize(self.h, None), "ssa_ukf_rollout_normalize")
            self.rollout_norm_io = None
            return None
        c = _lib.SsaNormCfg(int(bool(norm_obs)), int(bool(norm_reward)), int(bool(training)), int(obs_layout),
                            int(bool(reward_nan_to_num)), float(clip_obs), float(clip_reward), float(gamma), float(epsilon))
        _lib.check(self.lib.ssa_ukf_rollout_normalize(self.h, ctypes.byref(c)), "ssa_ukf_rollout_normalize")
        F = self.m * (4 if obs_layout == _lib.NORM_OBS_AER else 12)
        self.norm_F = F
        E = self.n_envs
        self._shapes[_lib.F_ROLLOUT_OBS_NORM] = ((E, F), np.float32)
        self._shapes[_lib.F_ROLLOUT_TERMINAL_OBS_NORM] = ((E, F), np.float32)
        self._shapes[_lib.F_ROLLOUT_REWARD_NORM] = ((E,), np.float64)
        self._shapes[_lib.F_ROLLOUT_NORM_STATE] = ((4 + E + 3 * F,), np.float64)
        ho, hr = ctypes.c_void_p(), ctypes.c_void_p()
        _lib.check(self.lib.ssa_ukf_rollout_norm_io(self.h, ctypes.byref(ho), ctypes.byref(hr)), "ssa_ukf_rollout_norm_io")
        self.rollout_norm_io = {"obs": _host_array(ho, ctypes.c_float, (E, F)), "reward": _host_array(hr, ctypes.c_double, (E,))}
        return self.rollout_norm_io

    def rollout_norm_state(self, stream=None):
        """The normalization state: {'obs_mean' [F], 'obs_var' [F], 'obs_count', 'ret_mean', 'ret_var', 'ret_count',
        'returns' [E]} (VecNormalize's obs_rms, ret_rms and returns); blocks until copied."""
        F, E = self.norm_F, self.n_envs
        out = np.empty(2 * F + 4 + E)
        _lib.check(self.lib.ssa_ukf_rollout_norm_state_download(self.h, _ptr(out), out.size, stream),
                   "ssa_ukf_rollout_norm_state_download")
        return {"obs_mean": out[:F], "obs_var": out[F:2 * F], "obs_count": float(out[2 * F]), "ret_mean": float(out[2 * F + 1]),
                "ret_var": float(out[2 * F + 2]), "ret_count": float(out[2 * F + 3]), "returns": out[2 * F + 4:]}

    def rollout_load_norm_state(self, state, stream=None):
        """Restore a rollout_norm_state() dict (training keeps its current setting); blocks until copied."""
        F, E = self.norm_F, self.n_envs
        buf = np.concatenate([np.asarray(state["obs_mean"], np.float64).reshape(F), np.asarray(state["obs_var"], np.float64).reshape(F),
                              [state["obs_count"], state["ret_mean"], state["ret_var"], state["ret_count"]],
                              np.asarray(state["returns"], np.float64).reshape(E)])
        _lib.check(self.lib.ssa_ukf_rollout_norm_state_upload(self.h, _ptr(buf), buf.size, stream), "ssa_ukf_rollout_norm_state_upload")

    def rollout_terminal_obs_norm(self, envs, stream=None):
        """The normalized final observations float32 [len(envs), F] of the environments `envs` (as rollout_terminal_obs)."""
        envs = np.ascontiguousarray(envs, dtype=np.int32).reshape(-1)
        out = np.empty((len(envs), self.norm_F), dtype=np.float32)
        _lib.check(self.lib.ssa_ukf_rollout_terminal_obs_norm_download(self.h, _ptr(envs), len(envs), _ptr(out), stream),
                   "ssa_ukf_rollout_terminal_obs_norm_download")
        return out

    @property
    def next_parity(self):
        return getattr(self, "_next_parity", 0)

    def predict(self, stream=None):
        _lib.check(self.lib.ssa_ukf_predict(self.h, stream), "ssa_ukf_predict")

    def update(self, M, all_objects=False, stream=None):
        M = np.ascontiguousarray(M, dtype=np.float64).reshape(9)
        _lib.check(self.lib.ssa_ukf_update(self.h, _ptr(M), 1 if all_objects else 0, stream), "ssa_ukf_update")

    def env_reduce(self, step_index, stream=None):
        _lib.check(self.lib.ssa_ukf_env_reduce(self.h, None, int(step_index), stream), "ssa_ukf_env_reduce")

    def scores(self, stream=None):
        _lib.check(self.lib.ssa_ukf_scores(self.h, stream), "ssa_ukf_scores")
        return self.download(_lib.F_SCORES, stream=stream)

    def snapshot(self, stream=None):
        """Every per-step output of the last step in one device-to-host copy; returns a dict of numpy views into a
        host block that the next snapshot() overwrites."""
        if getattr(self, "_snap", None) is None:
            N = self.N
            nbytes = int(self.lib.ssa_ukf_snapshot_bytes(self.h))
            buf = np.empty(nbytes, dtype=np.uint8)
            d = buf[:N * 118 * 8].view(np.float64).reshape(N, 118)
            st = buf[N * 118 * 8:N * 118 * 8 + 4 * N].view(np.int32)
            u8 = buf[N * 118 * 8 + 4 * N:]
            self._snap = (buf, {"x_true": d[:, 0:6], "x_filter": d[:, 6:12], "P_filter": d[:, 12:48].reshape(N, 6, 6),
                                "obs": d[:, 48:60], "delta_pos": d[:, 60], "delta_vel": d[:, 61], "sigma_pos": d[:, 62],
                                "sigma_vel": d[:, 63], "z_true": d[:, 64:67], "y": d[:, 67:70], "S": d[:, 70:79].reshape(N, 3, 3),
                                "sigmas_h": d[:, 79:118].reshape(N, 13, 3), "status": st, "visible": u8[:N], "updated": u8[N:]})
        buf, views = self._snap
        _lib.check(self.lib.ssa_ukf_snapshot(self.h, _ptr(buf), buf.nbytes, stream), "ssa_ukf_snapshot")
        return views

    def catalog_stats(self, index_offset=0, stream=None):
        """Catalog mode: reduce this shard's reward terms on the device (SSA_F_CATALOG_STATS: max delta_pos, trinary
        count sum, objects, max trace, global index of it); asynchronous, read with download / torch_view."""
        _lib.check(self.lib.ssa_ukf_catalog_stats(self.h, int(index_offset), stream), "ssa_ukf_catalog_stats")

    def diagnostics(self, stream=None):
        """Consistency diagnostics of the current state: (nees [N], nis [N] (NaN where not updated), flags uint8 [N]:
        0x80 valid | bit a: |y_a| < sqrt(S_aa) | bit 3+a: |y_a| < 2 sqrt(S_aa)).  NIS / flags need SSA_STEP_RECORD."""
        _lib.check(self.lib.ssa_ukf_diagnostics(self.h, stream), "ssa_ukf_diagnostics")
        d = self.download(_lib.F_DIAG, stream=stream)
        return d[:, 0].copy(), d[:, 1].copy(), self.download(_lib.F_INNOV_FLAGS, stream=stream)

    def sync(self, stream=None):
        _lib.check(self.lib.ssa_ukf_sync(self.h, stream), "ssa_ukf_sync")

    @property
    def launch_count(self):
        return int(self.lib.ssa_ukf_launch_count(self.h))


def fp64_peak_tflops(device=0, stream=None):
    lib = _lib.require_gpu()
    v = ctypes.c_double()
    _lib.check(lib.ssa_ukf_fp64_peak(int(device), stream, ctypes.byref(v)), "ssa_ukf_fp64_peak")
    return v.value


def innovation_stats(y, valid, nlags=40, device=0):
    """Whiteness statistics of B innovation series on the device (ssa_innovation_stats): y [B, n, 3], valid [B, n] bool.
    Returns (dw [B, 3], acf [B, 3, nlags + 1]): Durbin-Watson over the valid entries in order (SS2:782-832) and the
    autocorrelation with missing='conservative' (SS2:655-668)."""
    lib = _lib.require_gpu()
    y = np.ascontiguousarray(np.nan_to_num(np.asarray(y, dtype=np.float64)))
    valid = np.ascontiguousarray(np.asarray(valid).astype(np.uint8))
    B, n = valid.shape
    assert y.shape == (B, n, 3) and 0 <= nlags < n
    dw = np.empty((B, 3))
    acf = np.empty((B, 3, nlags + 1))
    _lib.check(lib.ssa_innovation_stats(_ptr(y), _ptr(valid), B, n, int(nlags), _ptr(dw), _ptr(acf), int(device)), "ssa_innovation_stats")
    return dw, acf
