"""The determinants behind agent_shannon and the reward.py score terms against EXACT determinants.

Every IEEE double is an exact rational, so Gaussian elimination over fractions.Fraction gives the exact determinant of
the matrix the kernel was handed.  `ssa_det6_sym` (unpivoted symmetric elimination, ssa_ukf_core.h) runs here through
the host twin, bit-equal to the device by construction; the `ssa_scores_kernel` determinants through their numpy
restatement (helpers.scores_det_restated, bit-equal to the device: tests/test_gpu_vs_oracle.py).  The yardstick is
numpy's own LAPACK determinant, what the reference's agent_shannon calls.

Measured on 8 572 covariances per mode (every 7th object-snapshot of 3 000 C2 objects over 60 steps): ssa_det6_sym is
off by at most 0.6 (catalog) and 2.9 (RL) times eps * cond(correlation matrix), np.linalg.det by up to 11 and 116."""
import numpy as np
import pytest

import helpers as H
from ssa_gym_b200 import _lib as F
from test_stress_c5 import singular_covariances

EPS = 2.0 ** -52


def _twin_covariances(mode, N=1200, steps=60, snaps=(1, 2, 5, 10, 20, 40, 60)):
    """Covariances of a twin run: catalog mode (every object updated) or RL mode (one tasked object per 10)."""
    cat, x, P0, zn = H.c2_inputs(N, steps)
    cfg = H.make_cfg(N) if mode == "catalog" else H.make_cfg(N, E=N // 10, m=10)
    st = H.HostState(cat, x, P0)
    rng = np.random.RandomState(5)
    out = []
    for s in range(1, steps + 1):
        if mode == "catalog":
            flags, act = F.STEP_TRUTH | F.STEP_PREDICT | F.STEP_UPDATE_ALL | F.STEP_EPILOGUE, None
        else:
            flags, act = F.STEP_TRUTH | F.STEP_PREDICT | F.STEP_UPDATE_ACT | F.STEP_EPILOGUE, rng.randint(0, 10, N // 10)
        H.cpu_step("twin", cfg, st, H.CEL2TER06AXY, flags, actions=act, z_noise=zn[s - 1])
        if s in snaps:
            out.append(st.P[::3].copy())
    assert (st.status & 1).sum() == 0
    return np.concatenate(out)


def _errors(P, dets):
    ex = [H.exact_det(A) for A in P]
    return np.array([[H.rel_err_exact(d[i], ex[i]) for i in range(len(P))] for d in dets])


@pytest.mark.parametrize("mode", ["catalog", "rl"])
def test_det6_sym_against_exact_on_filter_covariances(mode):
    P = _twin_covariances(mode)
    e_sym, e_np = _errors(P, [H.twin_det6(P), np.linalg.det(P)])
    k = H.corr_cond(P)
    # per matrix: within a conditioning bound (measured max 2.9 eps * cond; numpy's LU reaches 116)
    assert np.all(e_sym <= 16 * EPS * k), (np.max(e_sym / (EPS * k)), np.argmax(e_sym / (EPS * k)))
    # as a population: no further from the exact value than numpy's determinant
    assert e_sym.max() <= 2 * e_np.max() and np.median(e_sym) <= 2 * np.median(e_np), (e_sym.max(), e_np.max())
    assert np.median(e_sym) < 1e-14 and e_sym.max() < 1e-8


def test_det6_sym_against_exact_on_edge_covariances():
    P0 = np.diag([1e10] * 3 + [1e4] * 3)
    fail = np.diag([1e20] * 3 + [1e12] * 3)  # the filter-failure sentinels (SSA_XFAIL_POS / SSA_XFAIL_VEL)
    for A in (P0, fail, P0 * 1e-12, np.diag([3.0, 5.0, 7.0, 11.0, 13.0, 1e-300])):
        d = H.twin_det6(A[None])[0]
        assert H.rel_err_exact(d, H.exact_det(A)) <= 3 * EPS, A.diagonal()  # six products, each rounded once
    # exactly singular: a repeated row and column, a zero row and column -> exactly 0
    S = P0.copy(); S[1] = S[0]; S[:, 1] = S[:, 0]
    Z = P0.copy(); Z[4] = 0.0; Z[:, 4] = 0.0
    assert np.array_equal(H.twin_det6(np.stack([S, Z])), [0.0, 0.0])
    assert H.exact_det(S) == 0 and H.exact_det(Z) == 0

    # the stress covariances of test_stress_c5 (tiny, rank deficient, indefinite, hopeless); non-finite ones have no
    # exact determinant: NaN / inf in, NaN / inf out
    S = singular_covariances(600)
    fin = np.isfinite(S).all((1, 2))
    assert not np.isfinite(H.twin_det6(S[~fin])).any()
    P, cls = S[fin], (np.arange(600) % 6)[fin]
    e_sym, e_np = _errors(P, [H.twin_det6(P), np.linalg.det(P)])
    spd = cls <= 1
    k = H.corr_cond(P[spd])
    assert np.all(e_sym[spd] <= 16 * EPS * k)
    assert np.all(e_sym[cls == 2] == 0)  # rank deficient: exactly 0, as the exact determinant
    for c in (3, 4):  # indefinite: the unpivoted elimination loses what numpy's pivoted LU loses, within a factor 2
        assert e_sym[cls == c].max() <= 2 * e_np[cls == c].max(), (c, e_sym[cls == c].max(), e_np[cls == c].max())


def test_scores_kernel_determinants_against_exact():
    """score_det_P (pivoted 6x6 elimination) and score_det_pos_P (3x3 cofactor formula) of ssa_scores_kernel, through
    the restatement the GPU test pins bit for bit, against the exact determinants of the same matrices."""
    P = np.concatenate([_twin_covariances("catalog", N=600, snaps=(1, 5, 20, 60)),
                        _twin_covariances("rl", N=600, snaps=(1, 5, 20, 60))])
    det6, det3 = H.scores_det_restated(P)
    e6, e6np = _errors(P, [det6, np.linalg.det(P)])
    k6 = H.corr_cond(P)
    assert np.all(e6 <= 16 * EPS * k6) and e6.max() <= 2 * e6np.max(), (np.max(e6 / (EPS * k6)), e6.max(), e6np.max())
    B = P[:, :3, :3]
    e3, e3np = _errors(B, [det3, np.linalg.det(B)])
    k3 = H.corr_cond(B)
    # the cofactor formula cancels where LU does not: it may be off by more than numpy, not beyond the conditioning
    assert np.all(e3 <= 64 * EPS * k3), np.max(e3 / (EPS * k3))
    assert np.median(e3) < 1e-13 and e3.max() < 1e-9, (np.median(e3), e3.max(), e3np.max())
