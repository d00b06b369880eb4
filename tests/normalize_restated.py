"""Stable-Baselines3's VecNormalize and RunningMeanStd restated in numpy (SB3 is not installed here), expression by
expression, for the normalization tests.  `moments(arr)` computes a batch's (mean, var) over axis 0: numpy's np.mean /
np.var by default, or the fixed-order sums of the device (ssa_norm_moments) to compare the rest bit for bit."""
import numpy as np


def numpy_moments(arr):
    return np.mean(arr, axis=0), np.var(arr, axis=0)


class RunningMeanStd:
    def __init__(self, shape=(), epsilon=1e-4, moments=numpy_moments):
        self.mean = np.zeros(shape, np.float64)
        self.var = np.ones(shape, np.float64)
        self.count = epsilon
        self.moments = moments

    def update(self, arr):
        batch_mean, batch_var = self.moments(arr)
        self.update_from_moments(batch_mean, batch_var, arr.shape[0])

    def update_from_moments(self, batch_mean, batch_var, batch_count):
        delta = batch_mean - self.mean
        tot_count = self.count + batch_count
        new_mean = self.mean + delta * batch_count / tot_count
        m_a = self.var * self.count
        m_b = batch_var * batch_count
        m_2 = m_a + m_b + np.square(delta) * self.count * batch_count / tot_count
        new_var = m_2 / tot_count
        new_count = batch_count + self.count
        self.mean, self.var, self.count = new_mean, new_var, new_count


class VecNormalize:
    """VecNormalize's arithmetic on arrays: step(obs, rewards, dones, terminal) and reset(obs) return what its step_wait /
    reset return (observations cast to float32 at the end, as the device emits them)."""

    def __init__(self, E, F, training=True, norm_obs=True, norm_reward=True, clip_obs=10.0, clip_reward=10.0, gamma=0.99,
                 epsilon=1e-8, moments=numpy_moments):
        self.obs_rms = RunningMeanStd(shape=(F,), moments=moments)
        self.ret_rms = RunningMeanStd(shape=(), moments=moments)
        self.returns = np.zeros(E)
        self.training, self.norm_obs, self.norm_reward = training, norm_obs, norm_reward
        self.clip_obs, self.clip_reward, self.gamma, self.epsilon = clip_obs, clip_reward, gamma, epsilon

    def normalize_obs(self, obs):
        if not self.norm_obs:
            return obs
        return np.clip((obs - self.obs_rms.mean) / np.sqrt(self.obs_rms.var + self.epsilon), -self.clip_obs, self.clip_obs)

    def normalize_reward(self, reward):
        if not self.norm_reward:
            return reward
        return np.clip(reward / np.sqrt(self.ret_rms.var + self.epsilon), -self.clip_reward, self.clip_reward)

    def step(self, obs, rewards, dones, terminal=None):
        """terminal: rows [n_done, F] of the finished environments, or None."""
        if self.training and self.norm_obs:
            self.obs_rms.update(obs)
        out = self.normalize_obs(obs)
        if self.training:
            self.returns = self.returns * self.gamma + rewards
            self.ret_rms.update(self.returns)
        r = self.normalize_reward(rewards)
        term = None if terminal is None else self.normalize_obs(terminal).astype(np.float32)
        self.returns[dones] = 0
        return out.astype(np.float32), r, term

    def reset(self, obs):
        self.returns = np.zeros(len(obs))
        if self.training and self.norm_obs:
            self.obs_rms.update(obs)
        return self.normalize_obs(obs).astype(np.float32)

    def state(self):
        """The saved layout of ssa_ukf_rollout_norm_state_download."""
        F = len(self.obs_rms.mean)
        return np.concatenate([self.obs_rms.mean, self.obs_rms.var, [self.obs_rms.count, self.ret_rms.mean, self.ret_rms.var,
                                                                     self.ret_rms.count], self.returns]).reshape(2 * F + 4 + len(self.returns))
