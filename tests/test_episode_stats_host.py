"""CPU: the per-episode statistics of the episodic mode (ssa_ep_* in csrc/ssa_ukf_core.h, run by k_ep_row0 / k_ep_step on
the device) through their host build (tests/twin/episode_stats_twin.cpp, compiled here with the host twin's flags into a
temporary directory), on synthetic episodes, against the numpy restatements of the reference's
diagnostics (oracle/diagnostics.py): innovation-bound counts exact, Durbin-Watson statistics within 1e-14 relative, NEES
sums bit-equal to sequential Python sums of twin_diagnostics, NaN values left out, objects with fewer than two entries
left out of the per-object min / max, no-observation episodes NaN.  Also vec_env.episode_info against
D.innovation_bounds."""
import atexit
import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np

import helpers as H
from oracle import diagnostics as D
from ssa_gym_b200 import _lib as F
from ssa_gym_b200.vec_env import episode_info

EPO, EPE, EPR = 12, 20, F.EPISODE_STATS_DOUBLES
_LIB = {}


def stats_twin():
    """tests/twin/episode_stats_twin.cpp built once per process (flags of helpers.build_twin) in a temporary directory."""
    if "lib" not in _LIB:
        d = tempfile.mkdtemp(prefix="ssa_episode_stats_twin_")
        atexit.register(shutil.rmtree, d, True)
        lib = os.path.join(d, "libepisode_stats_twin.so")
        gxx = "/usr/bin/g++" if os.path.isfile("/usr/bin/g++") else "g++"
        subprocess.run([gxx, "-O2", "-std=c++17", "-ffp-contract=off", "-mfma", "-mavx2", "-shared", "-fPIC",
                        "-Wno-unknown-pragmas", "-o", lib, os.path.join(H.TWIN_DIR, "episode_stats_twin.cpp")], check=True)
        _LIB["lib"] = ctypes.CDLL(lib)
    return _LIB["lib"]


class TwinEpisodeStats:
    """Accumulators of E environments of m objects in the device's layouts, advanced by their host build."""

    def __init__(self, E, m):
        self.E, self.m = E, m
        self.obj = np.zeros((E * m, EPO))
        self.env = np.zeros((E, EPE))
        self.rec = np.zeros((E, EPR))

    def row0(self, step_idx, x_true, x, P):
        stats_twin().twin_episode_stats_row0(self.E, self.m, H.p(np.ascontiguousarray(step_idx, dtype=np.int32)),
                                         H.p(_f(x_true)), H.p(_f(x)), H.p(_packed(P)), H.p(self.obj))

    def step(self, step_idx, x_true, x, P, act_eff, updated, y, S, reward, done, status, auto_reset=True):
        stats_twin().twin_episode_stats_step(
            self.E, self.m, H.p(np.ascontiguousarray(step_idx, dtype=np.int32)), H.p(_f(x_true)), H.p(_f(x)), H.p(_packed(P)),
            H.p(np.ascontiguousarray(act_eff, dtype=np.int32)), H.p(np.ascontiguousarray(updated, dtype=np.uint8)),
            H.p(_f(np.nan_to_num(y))), H.p(_f(np.nan_to_num(S))), H.p(_f(reward)),
            H.p(np.ascontiguousarray(done, dtype=np.uint8)), H.p(np.ascontiguousarray(status, dtype=np.int32)),
            int(bool(auto_reset)), H.p(self.obj), H.p(self.env), H.p(self.rec))


def _f(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _packed(P):
    P = np.asarray(P, dtype=np.float64)
    return H.pack_P(P) if P.shape[-2:] == (6, 6) else _f(P)


def twin_nees(x_true, x, P):
    N = len(x_true)
    nees, nis, fl = np.empty(N), np.empty(N), np.empty(N, np.uint8)
    z3, z9, u = np.zeros((N, 3)), np.zeros((N, 9)), np.zeros(N, np.uint8)
    H.twin().twin_diagnostics(N, H.p(_f(x_true)), H.p(_f(x)), H.p(_packed(P)), H.p(z3), H.p(z9), H.p(u), H.p(nees),
                              H.p(nis), H.p(fl))
    return nees


def expected_record(rows, obs, L, ret, status_end, m):
    """The record of one episode from its histories.  rows: [(x_true [m,6], x [m,6], P [m,6,6])] for rows 0 .. L;
    obs: [(object, y [3], S [3,3])] of the tasked updates in order.  Returns (record with NaN where a value is compared
    at tolerance, dict of the values compared at tolerance)."""
    rec = np.full(EPR, np.nan)
    rec[0], rec[1] = L, ret
    nees = np.array([twin_nees(*r) for r in rows])          # [L + 1, m]
    per_obj = []
    for j in range(m):
        s = 0.0
        for v in nees[:, j]:
            if not np.isnan(v):
                s = s + float(v)
        per_obj.append(s)
    tot = 0.0
    for s in per_obj:
        tot = tot + s
    rec[2], rec[3] = tot, float((~np.isnan(nees)).sum())
    rec[6] = len(obs)
    tol = {}
    if obs:
        y = np.array([o[1] for o in obs]); S = np.array([o[2] for o in obs])
        one, two = D.innovation_flags(y, S)
        rec[7:10], rec[10:13] = one.sum(0), two.sum(0)
        ok = S.reshape(-1, 9).any(axis=1)  # (the synthetic singular S are zero matrices: ssa_inv3 reports them)
        nis = D.nis(y[ok], S[ok])
        rec[5] = ok.sum()
        tol["nis_sum"] = nis.sum()
        tol["dw_all"] = D.durbin_watson(y)
        dws = [D.durbin_watson(y[[o[0] == j for o in obs]]) for j in range(m) if sum(o[0] == j for o in obs) >= 2]
        tol["dw_min"] = np.min(dws, axis=0) if dws else np.full(3, np.nan)
        tol["dw_max"] = np.max(dws, axis=0) if dws else np.full(3, np.nan)
        tol["bounds"] = D.innovation_bounds(y, S)
    else:
        rec[5] = 0.0
        rec[7:13] = 0.0
        tol["nis_sum"] = 0.0
        tol["dw_all"] = tol["dw_min"] = tol["dw_max"] = np.full(3, np.nan)
        tol["bounds"] = np.full((2, 3), np.nan)
    rec[22] = float((status_end & F.ST_FAILED != 0).sum())
    return rec, tol


def _close(got, want, rtol):
    got, want = np.asarray(got, float), np.asarray(want, float)
    same_nan = np.array_equal(np.isnan(got), np.isnan(want))
    ok = ~np.isnan(want)
    return same_nan and np.all(np.abs(got[ok] - want[ok]) <= rtol * np.abs(want[ok]))


def _random_spd(rng, n, k, scale):
    A = rng.normal(size=(n, k, k)) * scale[:, None]
    return A @ np.swapaxes(A, 1, 2) + np.eye(k) * (scale ** 2)[None, :] * 0.1


def synthetic_run(E, m, T, seed, auto_reset=True):
    """T steps of E environments with random states, covariances (some not positive definite), innovations (some with a
    singular S), tasked objects (some steps skipped), rewards, done flags and failed objects; the twin's records compared
    with expected_record at every done.  Returns counters of the branches reached."""
    rng = np.random.RandomState(seed)
    acc = TwinEpisodeStats(E, m)
    N = E * m
    sc6 = np.array([1e5] * 3 + [1e2] * 3)
    sc3 = np.array([1e-5, 1e-5, 1e3])

    def draw_state():
        xt = rng.normal(size=(N, 6)) * 7e6
        x = xt + rng.normal(size=(N, 6)) * sc6
        P = _random_spd(rng, N, 6, np.tile(sc6, (N, 1)).reshape(N, 6)[0])
        bad = rng.rand(N) < 0.05  # not positive definite: NaN NEES
        P[bad, 2, 2] = -P[bad, 2, 2]
        return xt, x, P

    step_idx = np.zeros(E, np.int32)
    hist = [{"rows": [], "obs": [], "ret": 0.0} for _ in range(E)]
    seen = {"records": 0, "obs0": 0, "obs1": 0, "obs2+": 0, "nan_nees": 0, "nan_nis": 0, "skipped": 0, "failed": 0,
            "dw_lt2": 0}
    for t in range(T):
        xt, x, P = draw_state()
        acc.row0(step_idx, xt, x, P)
        for e in range(E):
            if step_idx[e] == 0:
                sl = slice(e * m, (e + 1) * m)
                hist[e] = {"rows": [(xt[sl], x[sl], P[sl])], "obs": [], "ret": 0.0}
        xt, x, P = draw_state()   # the state after this step's predict / update
        step_idx = step_idx + 1
        act = rng.randint(0, m, size=E).astype(np.int32)
        act[rng.rand(E) < 0.2] = -1
        updated = (rng.rand(N) < 0.7).astype(np.uint8)
        y = rng.normal(size=(N, 3)) * sc3 * rng.choice([0.5, 1.0, 3.0], size=(N, 1))
        S = _random_spd(rng, N, 3, sc3)
        sing = rng.rand(N) < 0.05
        S[sing] = 0.0
        reward = rng.normal(size=E)
        status = np.where(rng.rand(N) < 0.03, F.ST_FAILED | F.ST_NAN, 0).astype(np.int32)
        done = (rng.rand(E) < 0.15) | (step_idx >= 12)
        acc.step(step_idx, xt, x, P, act, updated, y, S, reward, done, status, auto_reset)
        for e in range(E):
            sl = slice(e * m, (e + 1) * m)
            hist[e]["rows"].append((xt[sl], x[sl], P[sl]))
            a = act[e]
            seen["skipped"] += a < 0
            if a >= 0 and updated[e * m + a]:
                hist[e]["obs"].append((a, y[e * m + a], S[e * m + a]))
            hist[e]["ret"] = hist[e]["ret"] + float(reward[e])
            if not done[e]:
                continue
            h = hist[e]
            want, tol = expected_record(h["rows"], h["obs"], step_idx[e], h["ret"], status[sl], m)
            got = acc.rec[e]
            exact = ~np.isnan(want)
            assert H.bits_equal(got[exact], want[exact]), (t, e, got, want)
            assert _close(got[4], tol["nis_sum"], 1e-9), (got[4], tol["nis_sum"])
            assert _close(got[13:16], tol["dw_all"], 1e-14) and _close(got[16:19], tol["dw_min"], 1e-14) and \
                _close(got[19:22], tol["dw_max"], 1e-14), (got[13:22], tol)
            info = episode_info(got)
            assert np.array_equal(info["innovation_bounds"], tol["bounds"], equal_nan=True)
            assert info["l"] == step_idx[e] and info["r"] == h["ret"] and info["observations"] == len(h["obs"])
            counts = np.bincount([o[0] for o in h["obs"]], minlength=m)
            seen["records"] += 1
            seen["obs0" if not h["obs"] else "obs1" if counts.max() == 1 else "obs2+"] += 1
            seen["dw_lt2"] += bool(h["obs"]) and np.any((counts == 1))
            seen["nan_nees"] += int(want[3] < (len(h["rows"]) * m))
            seen["nan_nis"] += int(want[5] < want[6])
            seen["failed"] += int(want[22] > 0)
        if auto_reset:
            step_idx[done] = 0
    return seen


def test_records_equal_oracle_diagnostics_with_auto_reset():
    seen = synthetic_run(E=7, m=4, T=60, seed=1)
    assert seen["records"] > 30 and all(v > 0 for v in seen.values()), seen


def test_records_without_auto_reset_cover_the_episode_so_far():
    """Without auto-reset a finished environment keeps its accumulators: the record of every later step covers rows
    0 .. i of the one episode."""
    seen = synthetic_run(E=5, m=3, T=25, seed=2, auto_reset=False)
    assert seen["records"] > 50, seen


def test_dw_push_is_the_innovation_stats_order():
    """One long series through ssa_ep_observe: the Durbin-Watson state equals D.durbin_watson within 1e-14 and a
    series of one entry gives num = 0 (statistic 0) while an object with one entry stays out of min / max."""
    E, m, T = 1, 2, 300
    rng = np.random.RandomState(5)
    acc = TwinEpisodeStats(E, m)
    P = np.broadcast_to(np.diag([1e10] * 3 + [1e4] * 3), (m, 6, 6))
    xt = rng.normal(size=(m, 6)); x = xt.copy()
    acc.row0([0], xt, x, P)
    ys = []
    for i in range(1, T + 1):
        a = 0 if i < T else 1   # object 1: one entry
        y = rng.normal(size=(m, 3)) * [1e-5, 1e-5, 1e3] + [3e-6, 0.0, -200.0]
        S = np.broadcast_to(np.diag([1e-10, 1e-10, 1e6]), (m, 3, 3)).reshape(m, 9)
        ys.append(y[a])
        acc.step([i], xt, x, P, [a], np.ones(m, np.uint8), y, S, [0.5], [i == T], np.zeros(m, np.int32))
    ys = np.array(ys)
    rec = acc.rec[0]
    assert _close(rec[13:16], D.durbin_watson(ys), 1e-14)
    assert _close(rec[16:19], D.durbin_watson(ys[:-1]), 1e-14) and _close(rec[19:22], D.durbin_watson(ys[:-1]), 1e-14)
    assert rec[0] == T and rec[1] == 0.5 * T and rec[6] == T and rec[3] == 2 * (T + 1) and rec[2] == 0.0
    # the accumulators were cleared for the next episode
    assert not acc.env.any() and not acc.obj.any()
