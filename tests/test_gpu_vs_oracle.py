"""-m gpu: the CUDA path against the INDEPENDENT oracle (oracle/ukf_oracle.c: reference operation order, libm),
through the C ABI, on the same seeded inputs — plus the operator callables and the reward.py score terms.
Tolerances are the ones derived in tests/test_oracle_golden.py; bit-exactness (against the host twin of the
device arithmetic) is in tests/test_gpu_bitexact.py."""
import numpy as np
import pytest

import helpers as H
from ssa_gym_b200 import _lib as F
from ssa_gym_b200 import dynamics
from ssa_gym_b200.ukf import BatchedUKF

pytestmark = pytest.mark.gpu
FULL = F.STEP_TRUTH | F.STEP_PREDICT | F.STEP_UPDATE_ALL | F.STEP_EPILOGUE | F.STEP_RECORD


def _ukf(N, **kw):
    cfg = H.make_cfg(N, **kw)
    return cfg, BatchedUKF(n_envs=kw.get("E") or 1, m=kw.get("m") or N, dt=20.0, Q=np.array(cfg.Q).reshape(6, 6),
                           R=np.array(cfg.R).reshape(3, 3),
                           obs_lla=[np.radians(H.OBSERVER_DEG[0]), np.radians(H.OBSERVER_DEG[1]), H.OBSERVER_DEG[2]],
                           obs_limit_rad=np.radians(kw.get("obs_limit_deg", -90.0)), reward_type=kw.get("reward_type", "jones"),
                           n_steps=kw.get("n_steps", 480))


def test_operator_callables_run_on_device_and_match_oracle():
    cat, x, _, _ = H.c2_inputs(4096)
    o, _ = H.lib_fx("oracle", x, 20.0)
    g = dynamics.fx_xyz_farnocchia(x, 20.0)
    rn = np.linalg.norm(o[:, :3], axis=1)[:, None]
    assert np.max(np.abs(g[:, :3] - o[:, :3]) / rn) < 1e-12                      # states: 1e-9 relative attained
    cfg = H.make_cfg(8)
    lla = np.array([np.radians(H.OBSERVER_DEG[0]), np.radians(H.OBSERVER_DEG[1]), H.OBSERVER_DEG[2]])
    z = dynamics.hx_aer_erfa(x, H.CEL2TER06AXY, lla, np.array(cfg.obs_itrs))
    zo = H.lib_hx("oracle", x, H.CEL2TER06AXY, np.array(cfg.obs_itrs), np.array(cfg.T))
    assert np.max(np.abs(z[:, :2] - zo[:, :2])) < 1e-12 and np.max(np.abs(z[:, 2] - zo[:, 2]) / zo[:, 2]) < 1e-14
    assert np.allclose(dynamics.fx_xyz_farnocchia(H.X6, 20.0),
                       [3.4051146353071168e+07, 2.3987757265636690e+07, 6.5213375290091345e+06, -1.9874091167254180e+03,
                        2.1478682154692128e+03, 9.1318892628514527e+02], rtol=1e-14)
    assert np.allclose(dynamics.residual_z_aer(np.array([np.radians(0.001), np.radians(10), 5.0]),
                                               np.array([np.radians(359.99), np.radians(-10), 7.0])),
                       [1.9198621771934277e-04, 3.4906585039886590e-01, -2.0], rtol=1e-12)
    assert np.allclose(dynamics.mean_z_uvw(np.array([[6.2, .1, 1e7], [.1, .12, 1.0001e7], [.05, .08, .9999e7]]), np.array([.5, .25, .25])),
                       [6.2790484981683656e+00, 1.0032788718535418e-01, 9.9665302565392759e+06], rtol=1e-13)
    U = dynamics.robust_cholesky(np.diag([1e10] * 3 + [1e4] * 3) * 3e-8)
    assert np.allclose(U.T @ U, np.diag([1e10] * 3 + [1e4] * 3) * 3e-8, rtol=1e-14)
    with pytest.raises(np.linalg.LinAlgError):
        dynamics.robust_cholesky(-np.eye(6) * 1e30)


def test_fused_step_c2_against_oracle():
    N = 20000
    cat, x, P0, zn = H.c2_inputs(N, 2)
    cfg, ukf = _ukf(N)
    ukf.reset(cat, x, P0)
    so = H.HostState(cat, x, P0)
    for s in range(2):
        ukf.upload(F.F_Z_NOISE, zn[s]); ukf.step(H.CEL2TER06AXY, FULL)
        H.cpu_step("oracle", cfg, so, H.CEL2TER06AXY, FULL, z_noise=zn[s])
        if s == 0:
            xg, xtg = ukf.download(F.F_X_FILTER), ukf.download(F.F_X_TRUE)
            rn = np.linalg.norm(so.x_true[:, :3], axis=1)[:, None]
            assert np.max(np.abs(xtg[:, :3] - so.x_true[:, :3]) / rn) < 1e-11       # truth: plain fx parity
            e = np.abs(xg[:, :3] - so.x[:, :3]) / rn
            assert np.median(e) < 1e-7 and e.max() < 1e-3                            # UT mean: conditioning bound
            assert np.array_equal(ukf.download(F.F_VISIBLE), so.visible)            # integer work: exact
            assert np.array_equal(ukf.download(F.F_UPDATED), so.updated)
            assert np.array_equal(ukf.download(F.F_STATUS), so.status)
            zt = ukf.download(F.F_Z_TRUE)
            assert np.max(np.abs(zt[:, :2] - so.z_true[:, :2])) < 1e-11 and np.max(np.abs(zt[:, 2] - so.z_true[:, 2]) / so.z_true[:, 2]) < 1e-12
        # covariance, innovation covariance, innovation: dimensionless (P by sqrt(P_ii P_jj), S likewise, y in sigmas).
        # The bounds are the conditioning of the reference's own filter, not a choice: against exact arithmetic its
        # double-precision run is off by 1e-4 (median) in a covariance after the first 1-arcsec update and by O(1) in the
        # worst element (tests/test_exact_truth.py); two faithful builds of its formulas differ by the same amounts.
        Pg, Sg, yg = ukf.download(F.F_P_FILTER), ukf.download(F.F_S), ukf.download(F.F_Y)
        d = np.sqrt(np.abs(np.einsum("nii->ni", so.P)))
        eP = np.abs(Pg - so.P) / (d[:, :, None] * d[:, None, :])
        dS = np.sqrt(np.einsum("nii->ni", so.S))
        eS, ey = np.abs(Sg - so.S) / (dS[:, :, None] * dS[:, None, :]), np.abs(yg - so.y) / dS
        lim = {0: (1e-5, 3e-2, 1e-6, 1e-4), 1: (1e-3, 1e-1, 1e-3, 1e-2)}[s]
        assert np.median(eP) < lim[0] and np.quantile(eP, 0.99) < lim[1], (s, np.median(eP), np.quantile(eP, 0.99))
        assert np.median(eS) < lim[2] and np.median(ey) < lim[3], (s, np.median(eS), np.median(ey))
        # K is not an output; x = x_pred + K y pins it: the updated state within the same envelope
        xg_s = ukf.download(F.F_X_FILTER)
        ex = np.abs(xg_s[:, :3] - so.x[:, :3]) / np.linalg.norm(so.x_true[:, :3], axis=1)[:, None]
        assert np.median(ex) < (1e-7 if s == 0 else 1e-6), (s, np.median(ex))
    assert (ukf.download(F.F_STATUS) & 1).sum() == 0
    assert abs(np.median(ukf.download(F.F_DELTA_POS)) / np.median(so.dpos) - 1) < 0.05
    ukf.close()


def test_env_reduce_and_scores():
    """Per-environment reductions (reward/done, greedy taskers) against numpy on the downloaded arrays: integer
    outputs bit-exact incl. first-maximum ties and the `np.any(visible)` index-0 quirk, agent_shannon against the twin
    emulation of its determinant history (repeated calls at one step index give the same picks); reward.py terms."""
    E, m = 257, 10
    N = E * m
    cat, x, P0, zn = H.c2_inputs(N, 3)
    for reward_type in ("jones", "trinary"):
        cfg, ukf = _ukf(N, E=E, m=m, obs_limit_deg=20.0, reward_type=reward_type, n_steps=50)
        ukf.reset(cat, x, P0)
        rng = np.random.RandomState(9)
        for s in range(3):
            ukf.upload(F.F_ACTIONS, rng.randint(0, m, E).astype(np.int32)); ukf.upload(F.F_Z_NOISE, zn[s])
            ukf.step(H.CEL2TER06AXY, F.STEP_TRUTH | F.STEP_PREDICT | F.STEP_UPDATE_ACT | F.STEP_EPILOGUE)
        hist = H.ShannonHistory(E, m)    # agent_shannon's determinant history in the device's arithmetic
        ukf.env_reduce(step_index=3)     # first call: no previous covariance -> every log-determinant ratio is 0
        g0 = ukf.download(F.F_GREEDY)
        vis0 = ukf.download(F.F_VISIBLE).reshape(E, m).astype(bool)
        sh0 = hist.scores(ukf.download(F.F_P_FILTER), np.full(E, 3))
        assert np.all(sh0 == 0.0)
        for e in range(E):
            v = np.where(vis0[e])[0]
            assert g0[e, F.TASKER_SHANNON] == (v[0] if np.any(v) else -1)
        ukf.env_reduce(step_index=3)     # again at the same step: the same picks
        assert np.array_equal(ukf.download(F.F_GREEDY), g0)
        for s in range(3, 5):
            ukf.upload(F.F_ACTIONS, rng.randint(0, m, E).astype(np.int32)); ukf.upload(F.F_Z_NOISE, zn[s % 3])
            ukf.step(H.CEL2TER06AXY, F.STEP_TRUTH | F.STEP_PREDICT | F.STEP_UPDATE_ACT | F.STEP_EPILOGUE)
        ukf.env_reduce(step_index=5)     # the ratio is between the two steps the reduction ran at (3 and 5)
        g5 = ukf.download(F.F_GREEDY)
        ukf.env_reduce(step_index=5)
        ukf.sync()
        assert np.array_equal(ukf.download(F.F_GREEDY), g5)
        dpos, dvel, tr = (ukf.download(f).reshape(E, m) for f in (F.F_DELTA_POS, F.F_DELTA_VEL, F.F_TRACE))
        vis = ukf.download(F.F_VISIBLE).reshape(E, m).astype(bool)
        greedy, rew, done = ukf.download(F.F_GREEDY), ukf.download(F.F_REWARD), ukf.download(F.F_DONE)
        P = ukf.download(F.F_P_FILTER).reshape(E, m, 6, 6)
        sh = hist.scores(P, np.full(E, 5))
        for e in range(E):
            assert greedy[e, F.TASKER_NAIVE_GREEDY] == np.argmax([np.trace(Pj) for Pj in P[e]])
            v = np.where(vis[e])[0]
            if not np.any(v):
                assert np.all(greedy[e, 1:] == -1)
            else:
                assert greedy[e, F.TASKER_VISIBLE_GREEDY] == v[np.argmax([np.trace(Pj) for Pj in P[e][v]])]
                assert greedy[e, F.TASKER_POS_ERROR_GREEDY] == v[np.argmax(dpos[e, v])]
                assert greedy[e, F.TASKER_VEL_ERROR_GREEDY] == v[np.argmax(dvel[e, v])]
                # agent_visible_greedy_aer (agents.py:57-63): the 'aer' observation's trace column after nan_to_num
                assert greedy[e, F.TASKER_VISIBLE_GREEDY_AER] == v[np.argmax(np.nan_to_num(tr[e, v], nan=0.001, posinf=0.001, neginf=0.001))]
                # agent_shannon (agents.py:15-26): argmax log(det P_5 / det P_3) in the device's arithmetic, exact
                # (ssa_det6_sym against exact determinants: tests/test_det_exact.py)
                assert greedy[e, F.TASKER_SHANNON] == H.first_visible_argmax(sh[e], vis[e]), (e, sh[e], vis[e])
            if reward_type == "trinary":
                assert rew[e] == np.mean(((dpos[e] < 1e4) * 1 + (dpos[e] < 1e7) * 1)) / 2 and done[e] == 0
            else:
                mx = np.max(dpos[e])
                assert (rew[e], done[e]) == ((0.0, 1) if mx > 5e6 else (1.0, 1) if mx < 3e4 else (0.0, 0))
        assert np.array_equal(tr, np.array([[np.trace(Pj) for Pj in Pe] for Pe in P]))   # trace order: bit-exact
        if reward_type == "jones":
            from oracle import dynamics_restated as D
            sc = ukf.scores().reshape(E, m, 6)
            # the determinant columns: bit-equal to the restatement of ssa_scores_kernel, which
            # tests/test_det_exact.py bounds against exact determinants
            det6, det3 = H.scores_det_restated(P.reshape(N, 6, 6))
            assert H.bits_equal(sc[:, :, 3].ravel(), det6) and H.bits_equal(sc[:, :, 4].ravel(), det3)
            for e in range(0, E, 37):
                for j in range(m):
                    assert np.isclose(sc[e, j, 0], D.score_scaled_trace_P(P[e, j]), rtol=1e-14)
                    assert sc[e, j, 1] == D.score_trace_P(P[e, j])
                    assert np.isclose(sc[e, j, 3], D.score_det_P(P[e, j]), rtol=1e-6)
                    assert np.isclose(sc[e, j, 4], D.score_det_pos_P(P[e, j]), rtol=1e-8)
                    assert np.isclose(sc[e, j, 2], D.score_scaled_det_P(P[e, j], dt=20.0), rtol=1e-6)
        ukf.close()
