"""-m gpu: the kernels each launch-path switch selects, as the handle's launch counter sees them.

The tests of bit-exactness show that every path computes the same values; these pin down WHICH path ran.  Every value
of SSA_UKF_KERNEL (unset and unknown values select the tile kernels), and SSA_UKF_ACT=split, runs five flag
combinations through every catalog entry point: ssa_ukf_step (as plain launches and as a cached graph),
ssa_ukf_step_host and ssa_ukf_step_pinned (plain launches and a captured graph).  A captured graph adds the launches it
holds, so each entry point must add the same count per call.  The episodic step is counted on every switch of
test_gpu_env_reduce_paths.SWITCHES, with and without auto-reset, at m = 10 (the warp-per-environment reduction) and
m = 70 (the CTA-per-environment one, after ssa_det_kernel)."""
import numpy as np
import pytest

import helpers as H
from ssa_gym_b200 import _lib as F
from ssa_gym_b200.ukf import BatchedUKF
from ssa_gym_b200.vec_env import VecSSATaskerEnv
from test_gpu_env_reduce_paths import SWITCHES, _cfg

pytestmark = pytest.mark.gpu

LAUNCH_VARS = ("SSA_UKF_KERNEL", "SSA_UKF_ACT", "SSA_UKF_STEP_GRAPH", "SSA_UKF_GRAPH", "SSA_UKF_CHUNK", "SSA_UKF_PDL",
               "SSA_UKF_STAGED_MAX", "SSA_UKF_DET_KERNEL", "SSA_UKF_REFRESH_CHAIN")

FULL = F.STEP_TRUTH | F.STEP_PREDICT | F.STEP_UPDATE_ALL | F.STEP_EPILOGUE
FLAGS = {"full": FULL, "rl": F.STEP_TRUTH | F.STEP_PREDICT | F.STEP_UPDATE_ACT | F.STEP_EPILOGUE,
         "predict": F.STEP_TRUTH | F.STEP_PREDICT, "epilogue": F.STEP_EPILOGUE, "full_stats": FULL | F.STEP_CATALOG_STATS}

# launches per step: tile = k_factor, k_predict_tile, k_refactor, k_update_tile (k_hx + k_update where k_update_tile
# does not apply); tile2 folds the factorisations into the tile kernels; fused is one k_step_tile per full catalog step;
# split is k_factor, k_fx, k_ut, k_hx, k_update; team is one ssa_step_kernel, without the reward-term reduction.
# SSA_STEP_CATALOG_STATS adds its two reduction kernels.
TILE = {"full": 4, "rl": 4, "predict": 3, "epilogue": 2, "full_stats": 6}
STEP_LAUNCHES = {
    "unset": ({}, TILE),
    "unknown": ({"SSA_UKF_KERNEL": "no-such-kernel"}, TILE),
    "tile": ({"SSA_UKF_KERNEL": "tile"}, TILE),
    "tile2": ({"SSA_UKF_KERNEL": "tile2"}, {"full": 2, "rl": 2, "predict": 2, "epilogue": 2, "full_stats": 4}),
    "fused": ({"SSA_UKF_KERNEL": "fused"}, {"full": 1, "rl": 4, "predict": 3, "epilogue": 2, "full_stats": 3}),
    "split": ({"SSA_UKF_KERNEL": "split"}, {"full": 5, "rl": 5, "predict": 3, "epilogue": 2, "full_stats": 7}),
    "team": ({"SSA_UKF_KERNEL": "team"}, {"full": 1, "rl": 1, "predict": 1, "epilogue": 1, "full_stats": 1}),
    "act_split": ({"SSA_UKF_ACT": "split"}, {"full": 4, "rl": 5, "predict": 3, "epilogue": 2, "full_stats": 6}),
}
ENTRY_POINTS = {"step": {"SSA_UKF_STEP_GRAPH": "0"}, "step_graph": {"SSA_UKF_STEP_GRAPH": "1"}, "step_host": {},
                "step_pinned": {"SSA_UKF_GRAPH": "0"}, "step_pinned_graph": {"SSA_UKF_GRAPH": "1"}}

# launches per episodic step, (auto-reset, no auto-reset), at m = 10 and m = 70: k_env_begin, the step's kernels
# (RL flags), the reward / done reduction (1, or ssa_det_kernel + 1), then with auto-reset k_env_refresh, or, on the
# refresh chain and the team kernel, k_env_reset + the gated epilogue + the reduction again
ROLLOUT_LAUNCHES = {
    "default": {10: (7, 6), 70: (8, 7)},
    "det_kernel": {10: (8, 7), 70: (8, 7)},
    "refresh_chain": {10: (10, 6), 70: (12, 7)},
    "no_graph": {10: (7, 6), 70: (8, 7)},
    "split": {10: (8, 7), 70: (9, 8)},
    "tile2": {10: (5, 4), 70: (6, 5)},
    "team": {10: (6, 3), 70: (8, 4)},
    "act_split": {10: (8, 7), 70: (9, 8)},
}


@pytest.fixture
def launch_env(monkeypatch):
    """Clears every launch switch, then sets those given (the handle reads them once, at its creation)."""
    for k in LAUNCH_VARS:
        monkeypatch.delenv(k, raising=False)

    def use(*envs):
        for env in envs:
            for k, v in env.items():
                monkeypatch.setenv(k, v)
    return use


def _catalog_handle(E=8, m=16):
    N = E * m
    cat, x, P0, _ = H.c2_inputs(N, 1)
    cfg = H.make_cfg(N, E=E, m=m)
    ukf = BatchedUKF(n_envs=E, m=m, dt=20.0, Q=np.array(cfg.Q).reshape(6, 6), R=np.array(cfg.R).reshape(3, 3),
                     obs_lla=[np.radians(H.OBSERVER_DEG[0]), np.radians(H.OBSERVER_DEG[1]), H.OBSERVER_DEG[2]],
                     obs_limit_rad=np.radians(-90.0))
    ukf.reset(cat, x, P0)
    ukf.upload(F.F_ACTIONS, np.arange(E, dtype=np.int32) % m)
    ukf.catalog_stats()  # (SSA_STEP_CATALOG_STATS needs it once)
    return ukf


@pytest.mark.parametrize("entry", sorted(ENTRY_POINTS))
@pytest.mark.parametrize("switch", sorted(STEP_LAUNCHES))
def test_catalog_step_launches(launch_env, switch, entry):
    env, table = STEP_LAUNCHES[switch]
    launch_env(env, ENTRY_POINTS[entry])
    ukf = _catalog_handle()
    M = H.CEL2TER06AXY
    if entry.startswith("step_pinned"):
        io = ukf.host_io()
        for b in range(2):
            io[b]["M"][:] = M.reshape(9)
            io[b]["actions"][:] = np.arange(ukf.n_envs, dtype=np.int32) % ukf.m
    call = {"step": lambda f: ukf.step(M, f), "step_graph": lambda f: ukf.step(M, f),
            "step_host": lambda f: ukf.step_host(M, f), "step_pinned": ukf.step_pinned,
            "step_pinned_graph": ukf.step_pinned}[entry]
    for name, flags in FLAGS.items():
        for rep in range(3):  # (the first call of a graph path captures, the next ones replay; both parities)
            l0 = ukf.launch_count
            call(flags)
            assert ukf.launch_count - l0 == table[name], (name, rep)
    ukf.host_join()
    ukf.sync()
    ukf.close()


@pytest.mark.parametrize("m", [10, 70])
@pytest.mark.parametrize("switch", sorted(ROLLOUT_LAUNCHES))
def test_rollout_step_launches(launch_env, switch, m):
    launch_env(SWITCHES.get(switch, {}))
    E = 6
    vec = VecSSATaskerEnv(_cfg(rso_count=m, steps=6, reward_type="jones", update_interval=1), E,
                          seeds=list(range(300, 300 + E)), rng="device")
    u = vec.ukf
    want = ROLLOUT_LAUNCHES[switch][m]
    for auto_reset in (0, 1, 1, 1, 1, 1, 1, 1):  # (auto-reset steps past the episode's end re-draw environments)
        l0 = u.launch_count
        u.rollout_step(auto_reset=bool(auto_reset))
        assert u.launch_count - l0 == want[1 - auto_reset], auto_reset
    u.sync()
    vec.close()
