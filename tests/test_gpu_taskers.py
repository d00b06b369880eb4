"""-m gpu: device taskers (VecSSATaskerEnv.set_tasker, ssa_ukf_rollout_tasker): the nine agents of agents.py picked
inside the episodic step graph.

Every tasker on every launch path equals the host twin with the restated pick (tests/tasker_restated.py) at every
step: taken actions, observations, rewards, dones and greedy columns.  A tasker run replayed as external actions is
bit-identical, episode records included; a tasker step launches the kernels of an external step; the random agents
have the reference's distributions; bad arguments are refused."""
import numpy as np
import pytest
import torch
from scipy import stats

import helpers as H
import tasker_restated as R
import ssa_gym_b200
from ssa_gym_b200 import _lib as F
from ssa_gym_b200 import agents
from ssa_gym_b200.transformations import gcrs2irts_matrix_approx, time_table
from ssa_gym_b200.vec_env import VecSSATaskerEnv
from test_gpu_env_reduce_paths import SWITCHES, launch_path  # noqa: F401  (launch_path: fixture)

pytestmark = pytest.mark.gpu
E = 45
AGENTS = [agents.agent_naive_greedy, agents.agent_visible_greedy, agents.agent_pos_error_greedy,
          agents.agent_vel_error_greedy, agents.agent_visible_greedy_aer, agents.agent_shannon,
          agents.agent_naive_random, agents.agent_visible_random, agents.agent_visible_greedy_spoiled]


def _cfg(**over):
    cfg = dict(ssa_gym_b200.env_config)
    cfg.update(over)
    cfg["trans_matrix"] = gcrs2irts_matrix_approx(time_table(cfg["t_0"], cfg["time_step"], cfg["steps"]))
    return cfg


def _vec(cfg, n=E, seed0=500, **kw):
    return VecSSATaskerEnv(cfg, n, seeds=list(range(seed0, seed0 + n)), rng="device", **kw)


def tasker_vs_twin(tasker, m, update_interval, steps=24, p=0.25):
    """Run tasker `tasker` on the device and in the twin (15-degree mask, 'jones', 6-step episodes) and demand
    equality at every step; returns the twin's counters."""
    cfg = _cfg(rso_count=m, steps=6, reward_type="jones", update_interval=update_interval, obs_limit=15)
    vec = _vec(cfg)
    vec.set_tasker(AGENTS[tasker], p)
    emu = R.TaskerTwin(vec, cfg, tasker, p)
    N = E * m
    obs_e, g_e = emu.reset()
    assert H.bits_equal(vec.obs.reshape(N, 12), obs_e) and np.array_equal(vec._io["greedy"], g_e)
    for t in range(steps):
        obs_v, r_v, d_v, _ = vec.vector_step()
        obs_e, r_e, d_e, g_e = emu.step()
        assert np.array_equal(vec.last_actions, emu.last_actions), (t, np.where(vec.last_actions != emu.last_actions))
        assert np.array_equal(d_v, d_e), t
        assert H.bits_equal(r_v, r_e), t
        assert H.bits_equal(obs_v.reshape(N, 12), obs_e), t
        assert np.array_equal(vec._io["greedy"], g_e), (t, np.where(vec._io["greedy"] != g_e))
        assert np.array_equal(vec.i, emu.step_idx), t
    st, u = emu.st, vec.ukf
    assert H.bits_equal(u.download(F.F_X_FILTER), st.x) and H.bits_equal(H.pack_P(u.download(F.F_P_FILTER)), H.pack_P(st.P))
    assert np.array_equal(u.download(F.F_VISIBLE).reshape(-1), st.visible.reshape(-1))
    vec.close()
    return emu.seen


def _require(seen, tasker, m, update_interval, steps=24):
    assert seen["resets"] >= E, seen
    if update_interval == 2:
        assert seen["skipped"] > 0, seen  # picks on steps update_interval skips
    if m == 10 and tasker != F.TASKER_NAIVE_GREEDY:  # the 15-degree mask leaves environments without candidates
        assert seen["fallback"] > 0 and seen["only_object_0"] > 0 and seen["none_visible"] > 0, seen
    if tasker == F.TASKER_NAIVE_RANDOM:
        assert seen["fallback"] == E * steps, seen
    if tasker == F.TASKER_VISIBLE_GREEDY_SPOILED:
        assert seen["spoiled"] > 0, seen  # candidate steps that took the fallback


@pytest.mark.parametrize("m,update_interval", [(10, 1), (10, 2), (70, 1), (70, 2)])
@pytest.mark.parametrize("tasker", range(len(AGENTS)))
def test_tasker_equals_twin(launch_path, tasker, m, update_interval):
    seen = tasker_vs_twin(tasker, m, update_interval)
    _require(seen, tasker, m, update_interval)


@pytest.mark.parametrize("tasker", range(len(AGENTS)))
@pytest.mark.parametrize("switch", sorted(SWITCHES))
def test_tasker_launch_path_equals_twin(launch_path, switch, tasker):
    """Each launch-path switch, each tasker; m = 10 / update_interval 1 and m = 70 / update_interval 2 alternate."""
    launch_path(SWITCHES[switch])
    m, ui = (10, 1) if (tasker + sorted(SWITCHES).index(switch)) % 2 == 0 else (70, 2)
    seen = tasker_vs_twin(tasker, m, ui)
    _require(seen, tasker, m, ui)


def test_replay_as_external_actions_is_bit_identical():
    """A tasker run fed back as external actions to an env with the same seeds gives the same run, bit for bit,
    episode statistics records included."""
    cfg = _cfg(rso_count=10, steps=6, reward_type="shaped", update_interval=2, obs_limit=15, episode_stats=True)
    a, b = _vec(cfg), _vec(cfg)
    a.set_tasker("visible_greedy_spoiled", 0.3)
    n_done = 0
    for t in range(30):
        oa, ra, da, ia = a.vector_step()
        ob, rb, db, ib = b.vector_step(a.last_actions)
        assert np.array_equal(b.last_actions, a.last_actions), t
        assert H.bits_equal(oa, ob) and H.bits_equal(ra, rb) and np.array_equal(da, db), t
        assert np.array_equal(a._io["greedy"], b._io["greedy"]), t
        for e in np.flatnonzero(da):
            assert H.bits_equal(np.array(ia[e]["episode"]["r"]), np.array(ib[e]["episode"]["r"]))
        n_done += int(da.sum())
    ea, eb = a.ukf.rollout_episode_stats(range(E)), b.ukf.rollout_episode_stats(range(E))
    assert n_done >= E and H.bits_equal(ea, eb)
    a.close(); b.close()


def test_device_loop_equals_host_loop():
    """vector_step_device with a tasker: device_views()['actions'] holds the taken actions, and the run equals the
    vector_step run of an env with the same seeds."""
    cfg = _cfg(rso_count=10, steps=6, reward_type="jones", update_interval=1, obs_limit=15)
    a, b = _vec(cfg), _vec(cfg)
    a.set_tasker(agents.agent_visible_random)
    b.set_tasker(agents.agent_visible_random)
    for t in range(20):
        oa, ra, da, _ = a.vector_step()
        v = b.vector_step_device()
        torch.cuda.synchronize()
        assert np.array_equal(v["actions"].cpu().numpy(), a.last_actions), t
        assert H.bits_equal(v["obs"].cpu().numpy(), oa) and H.bits_equal(v["reward"].cpu().numpy(), ra), t
        assert np.array_equal(v["done"].cpu().numpy().astype(bool), da), t
    a.close(); b.close()


def test_launch_counts_and_return_to_external():
    cfg = _cfg(rso_count=10, steps=6, reward_type="jones", update_interval=1, obs_limit=15, episode_stats=True)
    vec = _vec(cfg)
    u, m = vec.ukf, vec.m
    rng = np.random.RandomState(4)

    def launches(step):
        l0 = u.launch_count
        step()
        return u.launch_count - l0

    ext = launches(lambda: vec.vector_step(rng.randint(0, m, size=E)))
    vec.set_tasker(agents.agent_naive_random)
    tsk = launches(vec.vector_step)
    assert tsk == ext and tsk > 0
    # back to the caller's actions: the H2D of the actions takes effect again
    vec.set_tasker(None)
    for _ in range(3):
        want = rng.randint(0, m, size=E)
        vec.vector_step(want)
        assert np.array_equal(vec.last_actions, want)
        assert np.array_equal(u.download(F.F_ROLLOUT_ACTIONS), want)
    # rollout_config returns the handle to external actions
    u.rollout_tasker(F.TASKER_NAIVE_RANDOM)
    keys = np.array(vec.init_seeds, dtype=np.uint64)
    io = u.rollout_config(vec.orbits, vec.trans_matrix, keys, vec.x_sigma, vec.z_sigma, vec.P_0, 1)
    u.rollout_reset()
    for _ in range(3):
        want = rng.randint(0, m, size=E).astype(np.int32)
        io["actions"][:] = want
        u.rollout_step(True)
        u.sync()
        assert np.array_equal(io["actions"], want) and np.array_equal(u.download(F.F_ROLLOUT_ACTIONS), want)
    vec.close()


# ---- distributions (fixed seeds: deterministic) --------------------------------------------------------------------
def _run_recorded(agent, p=0.25, n=256, steps=60):
    """(actions, visibility, greedy) at every step of a tasker run: the visibility and greedy rows the pick read."""
    cfg = _cfg(rso_count=10, steps=6, reward_type="jones", update_interval=1, obs_limit=15)
    vec = _vec(cfg, n=n, seed0=900)
    vec.set_tasker(agent, p)
    acts, vis, gre = [], [], []
    for _ in range(steps):
        vis.append(vec.visible())
        gre.append(vec._io["greedy"].copy())
        vec.vector_step()
        acts.append(vec.last_actions.copy())
    vec.close()
    return np.array(acts), np.array(vis), np.array(gre)


def test_naive_random_is_uniform():
    acts, _, _ = _run_recorded(agents.agent_naive_random)
    counts = np.bincount(acts.reshape(-1), minlength=10)
    assert stats.chisquare(counts).pvalue > 1e-3, counts


def test_visible_random_picks_visible_objects_uniformly():
    acts, vis, _ = _run_recorded(agents.agent_visible_random)
    cells = {}
    n_cand = 0
    for a, v in zip(acts.reshape(-1), vis.reshape(-1, 10)):
        idx = R.candidates(v)
        if idx is None:
            continue
        n_cand += 1
        assert v[a], (a, v)
        k = len(idx)
        cells.setdefault(k, np.zeros(k, np.int64))[int(np.searchsorted(idx, a))] += 1
    assert n_cand > 1000
    chi2, dof = 0.0, 0
    for k, c in cells.items():
        if c.sum() >= 5 * k:  # (expected count >= 5 per cell)
            chi2 += stats.chisquare(c).statistic
            dof += k - 1
    assert dof >= 10 and stats.chi2.sf(chi2, dof) > 1e-3, (chi2, dof, cells)


def test_spoiled_fallback_share():
    p, m = 0.25, 10
    acts, vis, gre = _run_recorded(agents.agent_visible_greedy_spoiled, p)
    cand = np.array([R.candidates(v) is not None for v in vis.reshape(-1, m)])
    took_other = acts.reshape(-1)[cand] != gre.reshape(-1, F.N_TASKERS)[cand, F.TASKER_VISIBLE_GREEDY]
    n, k = int(cand.sum()), int(took_other.sum())
    assert n > 1000
    # a fallback differs from the greedy pick with probability (m - 1) / m
    assert stats.binomtest(k, n, p * (m - 1) / m).pvalue > 1e-3, (k, n)


# ---- refusals ------------------------------------------------------------------------------------------------------
def test_refusals():
    cfg = _cfg(rso_count=10, steps=6, reward_type="jones", update_interval=1)
    host = VecSSATaskerEnv(cfg, 4, seeds=[1, 2, 3, 4])
    with pytest.raises(ValueError):
        host.set_tasker(agents.agent_visible_greedy)
    with pytest.raises(F.SsaUkfError, match="EINVAL"):  # before rollout_config
        host.ukf.rollout_tasker(F.TASKER_VISIBLE_GREEDY)
    host.close()
    vec = _vec(cfg, n=4)
    for t, p in ((-2, 0.25), (9, 0.25), (F.TASKER_VISIBLE_GREEDY_SPOILED, float("nan")),
                 (F.TASKER_VISIBLE_GREEDY_SPOILED, float("inf")), (F.TASKER_VISIBLE_GREEDY_SPOILED, -0.1),
                 (F.TASKER_VISIBLE_GREEDY_SPOILED, 1.1)):
        with pytest.raises(F.SsaUkfError, match="EINVAL"):
            vec.ukf.rollout_tasker(t, p)
    for p in (0.0, 1.0):
        vec.ukf.rollout_tasker(F.TASKER_VISIBLE_GREEDY_SPOILED, p)
    vec.ukf.rollout_tasker(F.TASKER_EXTERNAL)
    with pytest.raises(ValueError):
        vec.set_tasker(lambda obs, env: 0)
    with pytest.raises(ValueError):
        vec.set_tasker("no_such_agent")
    with pytest.raises(ValueError):  # external actions are required without a tasker
        vec.vector_step()
    vec.set_tasker("shannon")
    with pytest.raises(ValueError):
        vec.vector_step(np.zeros(4, np.int64))
    vec.vector_step()
    vec.close()
