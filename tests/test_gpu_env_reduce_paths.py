"""-m gpu: the per-environment reductions (ssa_env_reduce_kernel, k_env_refresh, ssa_det_kernel) on every launch path
of the episodic mode, and agent_shannon in the host-RNG mode, EXACT against the host twin.

Every configuration runs E = 45 environments (not a multiple of 4: the last CTA of the warp-per-environment kernel has
idle warps) through at least E auto-resets and compares, at every step, observations, rewards, dones, all six greedy
columns and the step counters, and at the end the filter state, status, inflation counts, updated and visible flags
(helpers.episodic_vs_twin).  The m values cover one and two objects per lane of the warp path (m = 10, 40, 64), the
warp / CTA boundary (64 / 65) and a CTA whose threads stride over the objects twice (130)."""
import numpy as np
import pytest

import helpers as H
import ssa_gym_b200
from ssa_gym_b200 import _lib as F
from ssa_gym_b200.transformations import gcrs2irts_matrix_approx, time_table
from ssa_gym_b200.vec_env import VecSSATaskerEnv

pytestmark = pytest.mark.gpu
E = 45
SWITCHES = {"det_kernel": {"SSA_UKF_DET_KERNEL": "1"}, "refresh_chain": {"SSA_UKF_REFRESH_CHAIN": "1"},
            "no_graph": {"SSA_UKF_GRAPH": "0"}, "split": {"SSA_UKF_KERNEL": "split"},
            "tile2": {"SSA_UKF_KERNEL": "tile2"}, "team": {"SSA_UKF_KERNEL": "team"}, "act_split": {"SSA_UKF_ACT": "split"}}
PATH_VARS = sorted({k for v in SWITCHES.values() for k in v})


def _cfg(**over):
    cfg = dict(ssa_gym_b200.env_config)
    cfg.update(over)
    cfg["trans_matrix"] = gcrs2irts_matrix_approx(time_table(cfg["t_0"], cfg["time_step"], cfg["steps"]))
    return cfg


@pytest.fixture
def launch_path(monkeypatch):
    """Sets the launch-path variables of one configuration (the handle reads them once, at its creation)."""
    for k in PATH_VARS:
        monkeypatch.delenv(k, raising=False)

    def use(env):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
    return use


@pytest.mark.parametrize("m,over", [
    (10, {"steps": 6, "reward_type": "jones", "update_interval": 1}),
    (40, {"steps": 8, "reward_type": "trinary", "update_interval": 2}),
    (64, {"steps": 7, "reward_type": "jones", "update_interval": 2, "obs_limit": 10}),
    (65, {"steps": 8, "reward_type": "trinary", "update_interval": 1}),
    (130, {"steps": 6, "reward_type": "jones", "update_interval": 1, "obs_limit": 10}),
])
def test_default_path_equals_twin(launch_path, m, over):
    seen = H.episodic_vs_twin(_cfg(rso_count=m, **over), E, 40)
    assert seen["resets"] >= E, seen


@pytest.mark.parametrize("update_interval", [1, 2])
def test_sparse_visibility_equals_twin(launch_path, update_interval):
    """A 30-degree mask over 4 objects: environments that see nothing and environments that see only object 0 (the
    `not np.any(idx)` quirk of agents.py:37) at many steps."""
    seen = H.episodic_vs_twin(_cfg(rso_count=4, steps=7, reward_type="trinary", update_interval=update_interval,
                                   obs_limit=30), E, 40)
    assert seen["resets"] >= E and seen["none_visible"] > 0 and seen["only_object_0"] > 0, seen


@pytest.mark.parametrize("m", [10, 70])
@pytest.mark.parametrize("switch", sorted(SWITCHES))
def test_launch_path_equals_twin(launch_path, switch, m):
    """Each launch-path switch against the twin (and therefore against the default path, which equals the twin)."""
    launch_path(SWITCHES[switch])
    over = {"steps": 6, "reward_type": "jones", "update_interval": 1} if m == 10 else \
        {"steps": 7, "reward_type": "trinary", "update_interval": 2, "obs_limit": 10}
    seen = H.episodic_vs_twin(_cfg(rso_count=m, **over), E, 40)
    assert seen["resets"] >= E, seen


# ---- host-RNG mode: greedy_actions / env_reduce at one step index ------------------------------------------------
def _host_state(u):
    class S:
        pass
    s = S()
    s.dpos, s.dvel, s.trace = u.download(F.F_DELTA_POS), u.download(F.F_DELTA_VEL), u.download(F.F_TRACE)
    s.visible, s.P = u.download(F.F_VISIBLE), u.download(F.F_P_FILTER)
    return s


@pytest.mark.parametrize("m", [10, 70])
def test_greedy_actions_repeatable_and_exact_in_host_mode(m):
    """VecSSATaskerEnv(rng='host'): greedy_actions of every tasker, called twice at one step in different orders and
    after reset_at, returns the same device picks, and every pick equals the twin emulation (agent_shannon: the
    determinant history keyed to the step index, restarted at step 0 of a re-drawn environment)."""
    cfg = _cfg(rso_count=m, steps=7, reward_type="jones", obs_limit=10)
    vec = VecSSATaskerEnv(cfg, E, seeds=list(range(700, 700 + E)))
    u = vec.ukf
    hist = H.ShannonHistory(E, m)
    rng = np.random.RandomState(2)
    n_resets = 0
    for t in range(30):
        order = [F.TASKER_SHANNON] + list(range(F.N_TASKERS)) + [F.TASKER_SHANNON]
        picks = []
        for k in (order if t % 2 else order[::-1]):
            vec.greedy_actions(k)
            picks.append(u.download(F.F_GREEDY))
        assert all(np.array_equal(g, picks[0]) for g in picks), t
        _, _, g_e = H.emu_env_reduce(_host_state(u), E, m, vec.i, cfg["reward_type"], cfg["steps"], hist)
        assert np.array_equal(picks[0], g_e), (t, np.where(picks[0] != g_e))
        _, _, d, _ = vec.vector_step(rng.randint(0, m, size=E))
        n_resets += int(d.sum())
        if t % 5 == 4:  # an explicit reset: the re-drawn environment starts its history again
            vec.reset_at(t % E)
    assert n_resets >= E
    vec.close()
