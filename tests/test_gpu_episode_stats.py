"""-m gpu: per-episode statistics of the device-resident episodic mode (VecSSATaskerEnv(rng='device', episode_stats=True),
ssa_ukf_rollout_episode_stats_*), EXACT against the host twin on every launch path.

StatsTwin extends helpers.EpisodicTwin: it steps the twin with SSA_STEP_RECORD and applies the host build of the shared
accumulator functions (tests/twin/episode_stats_twin.cpp: twin_episode_stats_row0 / _step) to the same states, so every
record of every finished episode must be bit-equal to the device's. It also keeps each episode's histories (rows 0 .. L
of every object, the tasked innovations), against which the records are checked with the reference's formulas: the
Durbin-Watson columns bit-equal to ssa_innovation_stats on the recorded innovation series, ANEES and NIS close to
oracle/diagnostics.py's nees / nis, the innovation bounds equal to its innovation_bounds. The statistics change nothing
else: observations, rewards, dones and greedy picks equal those of an environment without them, whose step graph
launches the kernels it launched before."""
import collections

import numpy as np
import pytest

import helpers as H
from oracle import diagnostics as D
from ssa_gym_b200 import _lib as F
from ssa_gym_b200.ukf import innovation_stats
from ssa_gym_b200.vec_env import VecSSATaskerEnv, episode_info
from test_episode_stats_host import TwinEpisodeStats, twin_nees
from test_gpu_env_reduce_paths import SWITCHES, _cfg, launch_path  # noqa: F401  (launch_path: fixture)

pytestmark = pytest.mark.gpu
E = 45
FLAGS = F.STEP_TRUTH | F.STEP_PREDICT | F.STEP_UPDATE_ACT | F.STEP_EPILOGUE | F.STEP_M_PER_ENV | F.STEP_RECORD


class StatsTwin(H.EpisodicTwin):
    """EpisodicTwin with the per-episode statistics: `acc` holds the twin's accumulators and records, `hist[e]` the
    histories of environment e's current episode, `finished` the (environment, record, histories) of every episode whose
    done flag was raised on the last step."""

    def __init__(self, vec, cfg, auto_reset=True):
        super().__init__(vec, cfg)
        self.auto_reset = auto_reset
        self.acc = TwinEpisodeStats(self.E, self.m)
        self.hist = [None] * self.E
        self.finished = []
        self.seen = collections.Counter()

    def reset(self):
        out = super().reset()
        self.acc = TwinEpisodeStats(self.E, self.m)
        return out

    def _rows(self, e):
        st, sl = self.st, slice(e * self.m, (e + 1) * self.m)
        return st.x_true[sl].copy(), st.x[sl].copy(), st.P[sl].copy()

    def step(self, actions):
        E, m, st = self.E, self.m, self.st
        self.acc.row0(self.step_idx, st.x_true, st.x, st.P)
        for e in np.where(self.step_idx == 0)[0]:
            self.hist[e] = {"rows": [self._rows(e)], "obs": []}
        zn = np.zeros((self.N, 3))
        H.twin().twin_env_noise(E, m, H.p(self.keys), H.p(self.episode), H.p(self.step_idx), H.p(self.sig), H.p(zn))
        nxt = self.step_idx + 1
        a_eff = np.where(nxt % self.update_interval == 0, actions, -1).astype(np.int32)
        self.seen["skipped"] += int((a_eff < 0).sum())
        H.cpu_step("twin", self.cfg, st, self.table[np.minimum(nxt, self.n - 1)].reshape(E, 9), FLAGS, actions=a_eff,
                   z_noise=zn)
        self.step_idx[:] = nxt
        reward, done, self.greedy = H.emu_env_reduce(st, E, m, self.step_idx, self.reward_type, self.n, self.shannon)
        self.acc.step(self.step_idx, st.x_true, st.x, st.P, a_eff, st.updated, st.y, st.S.reshape(-1, 9), reward, done,
                      st.status, self.auto_reset)
        self.finished = []
        for e in range(E):
            h = self.hist[e]
            h["rows"].append(self._rows(e))
            a = int(a_eff[e])
            if a >= 0 and st.updated[e * m + a]:
                h["obs"].append((a, st.y[e * m + a].copy(), st.S[e * m + a].copy()))
            if done[e]:
                self.finished.append((e, self.acc.rec[e].copy(), {"rows": list(h["rows"]), "obs": list(h["obs"])}))
        if self.auto_reset and done.any():
            self._draw(done)
            self._refresh(done)
        return st.obs.copy(), reward, done, self.greedy.copy()


def check_against_formulas(rec, hist, m, seen, device=0):
    """One record against the reference's formulas on the episode's histories; counts the branches it shows."""
    L = len(hist["rows"]) - 1
    assert rec[0] == L and rec[6] == len(hist["obs"])
    nees = np.array([twin_nees(*r) for r in hist["rows"]])   # [L + 1, m]
    ok = ~np.isnan(nees)
    seen["nan_nees"] += int((~ok).any())
    assert rec[3] == ok.sum()
    info = episode_info(rec)
    if ok.any():
        # up to the summation order, the mean of the finite twin_diagnostics values (env.anees() of the drop-in env)
        assert abs(info["anees"] - np.nanmean(nees)) <= 1e-12 * abs(np.nanmean(nees)), (info["anees"], np.nanmean(nees))
        # against the reference's explicit inverse: the conditioning-aware bound of the drop-in env's diagnostics test
        sel = ok.ravel()
        xt = np.concatenate([r[0] for r in hist["rows"]])[sel]; x = np.concatenate([r[1] for r in hist["rows"]])[sel]
        P = np.concatenate([r[2] for r in hist["rows"]])[sel]
        ref = D.nees(xt, x, P)
        cond = np.array([np.linalg.cond(p_) for p_ in P])
        assert abs(info["anees"] - ref.mean()) <= np.mean(1e-15 * cond * np.abs(ref) + 1e-12) + 1e-12 * abs(ref.mean())
    else:
        assert np.isnan(info["anees"])
    counts = np.bincount([o[0] for o in hist["obs"]], minlength=m)
    seen["obs0" if not hist["obs"] else "obs1" if counts.max() == 1 else "obs2+"] += 1
    seen["some_object_once"] += int((counts == 1).any())
    seen["failed"] += int(rec[22] > 0)
    if not hist["obs"]:
        assert np.isnan(info["nis"]) and np.isnan(info["innovation_bounds"]).all() and np.isnan(rec[13:22]).all()
        return
    y = np.array([o[1] for o in hist["obs"]]); S = np.array([o[2] for o in hist["obs"]])
    nis = D.nis(y, S)
    condS = np.array([np.linalg.cond(s_) for s_ in S])
    assert abs(info["nis"] - np.nanmean(nis)) <= np.mean(1e-14 * condS * np.abs(nis) + 1e-12) + 1e-12 * abs(np.nanmean(nis))
    assert np.array_equal(info["innovation_bounds"], D.innovation_bounds(y, S))
    # Durbin-Watson: ssa_innovation_stats on the overall series and on every object's own series of this episode
    series = np.zeros((1 + m, L, 3)); valid = np.zeros((1 + m, L), bool)
    for t, (a, yy, _) in enumerate(hist["obs"]):
        series[0, t] = series[1 + a, t] = yy
        valid[0, t] = valid[1 + a, t] = True
    dw, _ = innovation_stats(series, valid, 0, device)
    assert H.bits_equal(rec[13:16], dw[0])
    per = dw[1:][valid[1:].sum(1) >= 2]
    lo = np.min(per, axis=0) if len(per) else np.full(3, np.nan)
    hi = np.max(per, axis=0) if len(per) else np.full(3, np.nan)
    assert H.bits_equal(rec[16:19], lo) and H.bits_equal(rec[19:22], hi)
    assert np.array_equal(info["durbin_watson"], np.round(np.vstack([dw[0], lo, hi]), 3), equal_nan=True)


def stats_vs_twin(cfg, total_steps, E=E, seed0=500, action_seed=11, auto_reset=True):
    """VecSSATaskerEnv(episode_stats=True) against StatsTwin and against a statistics-off environment with the same seeds
    and actions; returns the branch counters."""
    seeds = list(range(seed0, seed0 + E))
    vec = VecSSATaskerEnv(dict(cfg, episode_stats=True), E, seeds=seeds, rng="device", auto_reset=auto_reset)
    off = VecSSATaskerEnv(cfg, E, seeds=seeds, rng="device", auto_reset=auto_reset)
    emu = StatsTwin(vec, cfg, auto_reset)
    emu.reset()
    assert H.bits_equal(vec.obs, off.obs)
    rng = np.random.RandomState(action_seed)
    for t in range(total_steps):
        a = rng.randint(0, emu.m, size=E) if t % 2 == 0 else vec.greedy_actions(F.TASKER_VISIBLE_GREEDY)
        a = np.asarray(a, dtype=np.int32)
        o_v, r_v, d_v, infos = vec.vector_step(a)
        g_v = vec._io["greedy"].copy()
        o_o, r_o, d_o, _ = off.vector_step(a)
        assert H.bits_equal(o_v, o_o) and H.bits_equal(r_v, r_o) and np.array_equal(d_v, d_o), t
        assert np.array_equal(g_v, off._io["greedy"]), t
        _, r_e, d_e, g_e = emu.step(a)
        assert np.array_equal(d_v, d_e) and H.bits_equal(r_v, r_e) and np.array_equal(g_v, g_e), t
        fin = [f[0] for f in emu.finished]
        assert fin == np.flatnonzero(d_v).tolist()
        assert all(("episode" in infos[e]) == bool(d_v[e]) for e in range(E)), t
        if fin:
            recs = vec.ukf.rollout_episode_stats(fin)
            for k, (e, rec_e, hist) in enumerate(emu.finished):
                assert H.bits_equal(recs[k], rec_e), (t, e, recs[k], rec_e)
                assert infos[e]["episode"]["r"] == rec_e[1] and infos[e]["episode"]["l"] == rec_e[0]
                check_against_formulas(rec_e, hist, emu.m, emu.seen)
                emu.seen["records"] += 1
    vec.close()
    off.close()
    return emu.seen


@pytest.mark.parametrize("update_interval", [1, 2])
@pytest.mark.parametrize("m", [10, 70])
@pytest.mark.parametrize("switch", ["default"] + sorted(SWITCHES))
def test_episode_records_equal_twin_on_every_launch_path(launch_path, switch, m, update_interval):  # noqa: F811
    if switch != "default":
        launch_path(SWITCHES[switch])
    cfg = _cfg(rso_count=m, steps=7, reward_type="jones", update_interval=update_interval, obs_limit=10 if m == 70 else -90)
    seen = stats_vs_twin(cfg, 30)
    assert seen["records"] >= E and seen["obs1"] + seen["obs2+"] > 0, seen
    assert seen["some_object_once"] > 0, seen
    if m == 10 and update_interval == 1:  # (three observation steps of 7-step episodes rarely task one object twice)
        assert seen["obs2+"] > 0, seen
    if update_interval > 1:
        assert seen["skipped"] > 0, seen


def test_episode_records_without_auto_reset():
    """done stays set: the record is rewritten every step and covers the episode so far."""
    cfg = _cfg(rso_count=10, steps=5, reward_type="trinary", update_interval=1)
    seen = stats_vs_twin(cfg, 12, auto_reset=False)
    assert seen["records"] >= 7 * E and seen["obs2+"] > 0, seen


@pytest.mark.parametrize("over,need", [
    # a P_0 that is not positive definite: row 0's NEES is NaN and left out (the filters recover through the
    # inflation of robust_cholesky); episodes without any observation (a high mask over two objects)
    ({"P_0": np.diag([1e10, 1e10, 1e10, 1e4, 1e4, 0.0]), "rso_count": 2, "obs_limit": 45}, {"nan_nees", "obs0"}),
])
def test_episode_record_branches(over, need):
    cfg = _cfg(steps=9, reward_type="jones", update_interval=1, **over)
    seen = stats_vs_twin(cfg, 25)
    assert all(seen[k] > 0 for k in need), seen


def test_device_view_launch_counts_and_refusals():
    """device_views()['episode_stats'] rows equal the downloaded records; a statistics-off step graph launches as many
    kernels as that of a handle that never enabled them (a rollout_config turns them off), two fewer than a
    statistics-on one; rng='host' refuses episode_stats and a download before enable is SSA_EINVAL."""
    import torch
    cfg = _cfg(rso_count=6, steps=7, reward_type="jones", update_interval=2)
    seeds = list(range(300, 300 + E))
    vh = VecSSATaskerEnv(dict(cfg, episode_stats=True), E, seeds=seeds, rng="device")
    vd = VecSSATaskerEnv(dict(cfg, episode_stats=True), E, seeds=seeds, rng="device")
    views = vd.device_views()
    assert tuple(views["episode_stats"].shape) == (E, F.EPISODE_STATS_DOUBLES)
    rng = np.random.RandomState(5)
    n_done = 0
    for t in range(30):
        a = rng.randint(0, 6, size=E).astype(np.int32)
        _, _, dh, _ = vh.vector_step(a)
        views["actions"].copy_(torch.from_numpy(a))
        vd.vector_step_device()
        torch.cuda.synchronize()
        assert np.array_equal(views["done"].cpu().numpy().astype(bool), dh), t
        de = np.flatnonzero(dh)
        if len(de):
            assert H.bits_equal(views["episode_stats"].cpu().numpy()[de], vh.ukf.rollout_episode_stats(de)), t
            n_done += len(de)
    assert n_done >= E

    def per_step(v):
        c0 = v.ukf.launch_count
        v.vector_step(np.zeros(E, np.int32))
        c1 = v.ukf.launch_count
        v.vector_step(np.zeros(E, np.int32))
        return c1 - c0, v.ukf.launch_count - c1

    never = VecSSATaskerEnv(cfg, E, seeds=seeds, rng="device")
    again = VecSSATaskerEnv(dict(cfg, episode_stats=True), E, seeds=seeds, rng="device")
    base = per_step(never)
    assert per_step(again) == (base[0] + 2, base[1] + 2)
    again._io = again.ukf.rollout_config(again.orbits, again.trans_matrix, np.array(again.init_seeds, dtype=np.uint64),
                                         again.x_sigma, again.z_sigma, again.P_0, again.update_interval)
    again.episode_stats = False
    again.vector_reset()
    assert per_step(again) == base
    u = again.ukf
    out = np.empty((1, F.EPISODE_STATS_DOUBLES))
    rc = u.lib.ssa_ukf_rollout_episode_stats_download(u.h, H.p(np.zeros(1, np.int32)), 1, H.p(out), None)
    assert rc == F.SSA_EINVAL and b"not enabled" in u.lib.ssa_ukf_last_error()
    with pytest.raises(F.SsaUkfError):
        u.rollout_episode_stats([0])
    with pytest.raises(ValueError):
        VecSSATaskerEnv(dict(cfg, episode_stats=True), 4, rng="host")
    for v in (vh, vd, never, again):
        v.close()
