"""CPU: the running normalization of the episodic mode (ssa_norm_* in csrc/ssa_ukf_core.h, run by k_normalize on the device)
through its host build (tests/twin/normalize_twin.cpp, compiled here with the host twin's flags into a temporary
directory), against a numpy restatement of Stable-Baselines3's VecNormalize / RunningMeanStd (normalize_restated.py).

Given the same batch moments, the merge and the element-wise maps are bit-equal to the restatement, step after step.  The
batch moments use the device's fixed summation order instead of numpy's sequential one; against np.mean / np.var they
agree within the rounding-error bound of the two orders: |d mean| <= (E + L + log2(leaves)) eps mean|x| per column, L the
leaf length.  Edge cases: E = 1, constant columns, 1e20 failed-filter sentinels, NaN, values at the clip, gamma 0 and 1,
the training toggle, resets."""
import atexit
import ctypes
import math
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

import helpers as H
from normalize_restated import VecNormalize, numpy_moments

EPS = np.finfo(np.float64).eps
_LIB = {}


def norm_twin():
    """tests/twin/normalize_twin.cpp built once per process (flags of helpers.build_twin) in a temporary directory."""
    if "lib" not in _LIB:
        d = tempfile.mkdtemp(prefix="ssa_normalize_twin_")
        atexit.register(shutil.rmtree, d, True)
        lib = os.path.join(d, "libnormalize_twin.so")
        gxx = "/usr/bin/g++" if os.path.isfile("/usr/bin/g++") else "g++"
        subprocess.run([gxx, "-O2", "-std=c++17", "-ffp-contract=off", "-mfma", "-mavx2", "-shared", "-fPIC",
                        "-Wno-unknown-pragmas", "-o", lib, os.path.join(H.TWIN_DIR, "normalize_twin.cpp")], check=True)
        L = ctypes.CDLL(lib)
        D, I, P = ctypes.c_double, ctypes.c_int, ctypes.c_void_p
        L.twin_norm_moments.argtypes = [P, ctypes.c_long, I, I, P, P]
        L.twin_norm_merge.argtypes = [P, P, P, D, D, D]
        L.twin_norm_obs.argtypes = [I, P, P, P, D, D, P]
        L.twin_norm_reward.argtypes = [I, P, D, D, D, P]
        L.twin_norm_return.argtypes = [I, P, D, P, I, P]
        L.twin_normalize.argtypes = [I, I, I, P, I, P, P, P, I, I, I, I, D, D, D, D, P, P, P, P]
        _LIB["lib"] = L
    return _LIB["lib"]


def leaf(E):
    return 32 if E <= 32768 else (E + 1023) // 1024


def twin_moments(arr, f32=False):
    """(mean, var) over axis 0 in the device's order (ssa_norm_moments), of a 1-d or 2-d float64 array."""
    a = np.ascontiguousarray(arr, dtype=np.float64)
    E = a.shape[0]
    F = 1 if a.ndim == 1 else a.shape[1]
    mean, var = np.empty(F), np.empty(F)
    m, v = ctypes.c_double(), ctypes.c_double()
    for c in range(F):
        norm_twin().twin_norm_moments(a.ctypes.data + 8 * c, F, E, int(f32), ctypes.byref(m), ctypes.byref(v))
        mean[c], var[c] = m.value, v.value
    return (mean[0], var[0]) if a.ndim == 1 else (mean, var)


class TwinNormalize:
    """twin_normalize over host arrays, with the state in the saved layout (2 F + 4 + E doubles)."""

    def __init__(self, E, F, training=True, norm_obs=True, norm_reward=True, clip_obs=10.0, clip_reward=10.0, gamma=0.99,
                 epsilon=1e-8, f32=False, reward_nan=False):
        self.E, self.F = E, F
        self.state = np.concatenate([np.zeros(F), np.ones(F), [1e-4, 0.0, 1.0, 1e-4], np.zeros(E)])
        self.training, self.norm_obs, self.norm_reward = training, norm_obs, norm_reward
        self.clip_obs, self.clip_reward, self.gamma, self.epsilon = clip_obs, clip_reward, gamma, epsilon
        self.f32, self.reward_nan = f32, reward_nan
        self.term = np.zeros((E, F), np.float32)

    def run(self, mode, obs, done=None, reward=None, term=None):
        E, F = self.E, self.F
        obs = np.ascontiguousarray(obs, dtype=np.float64).reshape(E, F)
        done = np.ascontiguousarray(np.zeros(E) if done is None else done, dtype=np.uint8)
        reward = np.ascontiguousarray(np.zeros(E) if reward is None else reward, dtype=np.float64)
        term_in = None if term is None else np.ascontiguousarray(term, dtype=np.float64).reshape(E, F)
        out, rout = np.zeros((E, F), np.float32), np.zeros(E)
        norm_twin().twin_normalize(mode, E, F, H.p(obs), int(self.f32), None if term_in is None else H.p(term_in), H.p(done),
                                   H.p(reward), int(self.training), int(self.norm_obs), int(self.norm_reward),
                                   int(self.reward_nan), self.clip_obs, self.clip_reward, self.gamma, self.epsilon,
                                   H.p(self.state), H.p(out), H.p(self.term), H.p(rout))
        return out, rout

    def step(self, obs, reward, done, term=None):
        return self.run(0, obs, done, reward, term)

    def reset(self, obs):
        return self.run(1, obs)[0]


def bits(a, b):
    """bit equality; float32 arrays compared through their (exact) float64 values"""
    f = lambda x: np.asarray(x).astype(np.float64) if np.asarray(x).dtype == np.float32 else np.asarray(x)
    return H.bits_equal(f(a), f(b))


def _episode(E, F, steps, seed, scale=None, **kw):
    """A raw stream: rows of widely different column scales, rewards with some NaN, ~10 % done per step."""
    rng = np.random.default_rng(seed)
    scale = np.logspace(-3, 7, F) if scale is None else scale
    for _ in range(steps):
        obs = rng.standard_normal((E, F)) * scale + scale
        reward = rng.standard_normal(E)
        done = rng.random(E) < 0.1
        term = rng.standard_normal((E, F)) * scale
        yield obs, reward, done, term


def _run_both(E, F, steps, seed, twin_kw=None, rest_kw=None, nan_reward=False):
    twin_kw, rest_kw = twin_kw or {}, rest_kw or {}
    tw = TwinNormalize(E, F, reward_nan=nan_reward, **twin_kw)
    f32 = twin_kw.get("f32", False)
    cast = (lambda a: a.astype(np.float32).astype(np.float64)) if f32 else (lambda a: a)
    rest = VecNormalize(E, F, moments=lambda a: twin_moments(a), **rest_kw)
    rng = np.random.default_rng(seed + 1)
    o0 = rng.standard_normal((E, F)) * 1e3
    assert bits(tw.reset(o0), rest.reset(cast(o0)))
    assert bits(tw.state, rest.state())
    for t, (obs, reward, done, term) in enumerate(_episode(E, F, steps, seed)):
        if nan_reward:
            reward[::7] = np.nan
            reward[1::11] = np.inf
        out, r = tw.step(obs, reward, done, term)
        rr = np.nan_to_num(reward, nan=0.5, posinf=0.5, neginf=0.5) if nan_reward else reward
        o_e, r_e, t_e = rest.step(cast(obs), rr, done, cast(term[done]))
        assert bits(out, o_e) and bits(r, r_e), t
        assert bits(tw.term[done], t_e), t
        assert bits(tw.state, rest.state()), t
    return tw, rest


@pytest.mark.parametrize("E,F", [(1, 12), (7, 4), (33, 24), (256, 120), (1000, 40), (40000, 2)])
def test_step_sequence_bit_equal_given_the_same_moments(E, F):
    _run_both(E, F, 6, seed=E + F)


@pytest.mark.parametrize("kw", [dict(gamma=0.0), dict(gamma=1.0), dict(norm_obs=False), dict(norm_reward=False),
                                dict(clip_obs=0.5, clip_reward=0.25), dict(epsilon=0.0), dict(epsilon=1e-2)])
def test_options_bit_equal(kw):
    _run_both(64, 24, 5, seed=3, twin_kw=kw, rest_kw=kw)


def test_float32_rows_and_nan_rewards():
    """obs_dtype float32: the statistics see the float32-rounded rows; non-'flatten' layouts: NaN / inf rewards enter as 0.5."""
    _run_both(100, 24, 5, seed=5, twin_kw=dict(f32=True))
    _run_both(100, 24, 5, seed=6, nan_reward=True)


def test_training_toggle():
    """training=False: nothing moves but returns[done] = 0 (VecNormalize zeroes them whatever training is); back on, the
    updates continue from where they stopped."""
    E, F = 50, 12
    tw, rest = TwinNormalize(E, F), VecNormalize(E, F, moments=twin_moments)
    o0 = np.random.default_rng(9).standard_normal((E, F))
    tw.reset(o0), rest.reset(o0)
    for t, (obs, reward, done, term) in enumerate(_episode(E, F, 9, 10)):
        training = t not in (3, 4, 5)
        tw.training = rest.training = training
        before = tw.state.copy()
        out, r = tw.step(obs, reward, done, term)
        o_e, r_e, t_e = rest.step(obs, reward, done, term[done])
        assert bits(out, o_e) and bits(r, r_e) and bits(tw.term[done], t_e) and bits(tw.state, rest.state()), t
        if not training:
            after = before.copy()
            after[2 * F + 4:][done] = 0.0
            assert bits(tw.state, after), t


def test_reset_envs_refreshes_rows_and_returns_only():
    E, F = 40, 12
    tw = TwinNormalize(E, F)
    rng = np.random.default_rng(4)
    tw.reset(rng.standard_normal((E, F)))
    obs, reward, done, term = next(_episode(E, F, 1, 4))
    tw.step(obs, reward, np.zeros(E, bool))
    state = tw.state.copy()
    mask = np.zeros(E, bool)
    mask[[3, 17]] = True
    fresh = rng.standard_normal((E, F))
    o2, _ = tw.run(2, fresh, done=mask)
    exp = state.copy()
    exp[2 * F + 4:][mask] = 0.0
    assert bits(tw.state, exp)
    m, v = state[:F], state[F:2 * F]
    ref = np.clip((fresh[mask] - m) / np.sqrt(v + 1e-8), -10, 10).astype(np.float32)
    assert bits(o2[mask], ref) and not np.any(o2[~mask])


def test_reset_zeroes_returns_and_updates_obs_statistics():
    E, F = 30, 8
    tw, rest = TwinNormalize(E, F), VecNormalize(E, F, moments=twin_moments)
    for obs, reward, done, term in _episode(E, F, 2, 1):
        tw.step(obs, reward, done), rest.step(obs, reward, done)
    o = np.random.default_rng(2).standard_normal((E, F))
    assert bits(tw.reset(o), rest.reset(o)) and bits(tw.state, rest.state()) and not np.any(tw.state[2 * F + 4:])


def _moment_bound(x, mean_t, var_t):
    """|d mean| and |d var| of the fixed order against np.mean / np.var, within the worst-case bounds of the two sums."""
    E = x.shape[0]
    n_leaves = -(-E // leaf(E))
    c = E + leaf(E) + math.ceil(math.log2(max(n_leaves, 1))) + 4
    mean_n, var_n = numpy_moments(x)
    dm = np.abs(mean_t - mean_n)
    assert np.all(dm <= c * EPS * np.mean(np.abs(x), axis=0)), (dm, np.mean(np.abs(x), axis=0))
    dev = np.abs(x - mean_n)
    bound = c * EPS * np.mean(dev ** 2, axis=0) + 2 * dm * np.mean(dev, axis=0) + dm ** 2
    assert np.all(np.abs(var_t - var_n) <= bound * (1 + 1e-12))


@pytest.mark.parametrize("E", [1, 2, 31, 32, 33, 4096, 40000])
def test_batch_moments_within_bound_of_numpy(E):
    rng = np.random.default_rng(E)
    x = np.concatenate([rng.standard_normal((E, 4)) * [1, 1e-3, 1e6, 3e7] + [0, 5, -1e6, 4e7],
                        rng.lognormal(0, 3, (E, 2))], axis=1)
    mean_t, var_t = twin_moments(x)
    _moment_bound(x, mean_t, var_t)
    if E == 1:
        assert bits(mean_t, x[0]) and not np.any(var_t)


def test_constant_columns_and_sentinels():
    """A constant column has variance 0 and mean the constant (exactly, for a value whose multiples are exact); a column
    with 1e20 failed-filter sentinels stays finite and its normalized values are clipped."""
    E, F = 4096, 3
    x = np.empty((E, F))
    x[:, 0] = 1.5
    x[:, 1] = np.random.default_rng(0).standard_normal(E) * 1e7
    x[::97, 1] = 1e20
    x[:, 2] = -2.0 ** -20
    mean_t, var_t = twin_moments(x)
    assert mean_t[0] == 1.5 and var_t[0] == 0.0 and mean_t[2] == -2.0 ** -20 and var_t[2] == 0.0
    assert np.isfinite(mean_t[1]) and np.isfinite(var_t[1])
    _moment_bound(x, mean_t, var_t)
    tw, rest = TwinNormalize(E, F), VecNormalize(E, F, moments=twin_moments)
    out, rest_out = tw.reset(x), rest.reset(x)
    assert bits(out, rest_out) and np.all(np.abs(out) <= 10) and np.all(np.isfinite(out))


def test_nan_propagates_like_numpy():
    E, F = 64, 3
    x = np.random.default_rng(1).standard_normal((E, F))
    x[5, 1] = np.nan
    tw, rest = TwinNormalize(E, F), VecNormalize(E, F, moments=twin_moments)
    out, rest_out = tw.reset(x), rest.reset(x)
    assert bits(out, rest_out) and np.all(np.isnan(out[:, 1])) and not np.any(np.isnan(out[:, [0, 2]]))
    assert np.isnan(tw.state[1]) and np.isnan(tw.state[F + 1]) and np.isnan(numpy_moments(x)[0][1])


def test_element_maps_and_clip_edges():
    """normalize_obs / normalize_reward / the return update against numpy on edge values: exactly at the clip, beyond it,
    +-inf, NaN, -0.0."""
    L = norm_twin()
    v = np.array([10.0, -10.0, 10.000000000000002, -11.0, np.inf, -np.inf, np.nan, -0.0, 0.0, 3.0, 1e300, -1e-300])
    n = len(v)
    for mean, var, eps, clip in [(0.0, 1.0, 0.0, 10.0), (1.0, 4.0, 1e-8, 0.5), (-3.0, 1e-12, 1e-8, 10.0), (0.0, 0.0, 0.0, 1.0)]:
        out = np.empty(n)
        L.twin_norm_obs(n, H.p(v), H.p(np.full(n, mean)), H.p(np.full(n, var)), eps, clip, H.p(out))
        with np.errstate(all="ignore"):
            exp = np.clip((v - np.full(n, mean)) / np.sqrt(np.full(n, var) + eps), -clip, clip)
        assert bits(out, exp), (mean, var, eps, clip)
        L.twin_norm_reward(n, H.p(v), var, eps, clip, H.p(out))
        with np.errstate(all="ignore"):
            exp = np.clip(v / np.sqrt(var + eps), -clip, clip)
        assert bits(out, exp)
    ret = np.random.default_rng(3).standard_normal(n)
    for gamma in (0.0, 0.99, 1.0):
        for nan in (0, 1):
            out = np.empty(n)
            L.twin_norm_return(n, H.p(ret), gamma, H.p(v), nan, H.p(out))
            r = np.nan_to_num(v, nan=0.5, posinf=0.5, neginf=0.5) if nan else v
            assert bits(out, ret * gamma + r)


def test_merge_bit_equal():
    """update_from_moments on random and extreme moments (count 1e-4 start, large counts, zero variance, 1e40 deltas)."""
    from normalize_restated import RunningMeanStd
    rng = np.random.default_rng(12)
    cases = [(rng.standard_normal() * 10.0 ** rng.integers(-5, 20), abs(rng.standard_normal()) * 10.0 ** rng.integers(-10, 40),
              float(rng.integers(1, 5000))) for _ in range(200)] + [(1e20, 1e40, 4096.0), (0.0, 0.0, 1.0), (-1e-300, 0.0, 3.0)]
    rms = RunningMeanStd(())
    m, v, c = ctypes.c_double(0.0), ctypes.c_double(1.0), ctypes.c_double(1e-4)
    for bm, bv, bc in cases:
        rms.update_from_moments(bm, bv, int(bc))
        norm_twin().twin_norm_merge(ctypes.byref(m), ctypes.byref(v), ctypes.byref(c), bm, bv, bc)
        assert bits(m.value, rms.mean) and bits(v.value, rms.var) and bits(c.value, rms.count)
