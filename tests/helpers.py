"""Shared test infrastructure: loads the oracle (oracle/liboracle.so), the host twin
(tests/twin/libssa_twin.so) and the product (ssa_gym_b200) and runs the same batch step through each."""
import ctypes
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from ssa_gym_b200 import _lib  # noqa: E402
from ssa_gym_b200.transformations import arcsec2rad, lla2ecef, trans_uvw_ecef  # noqa: E402
from ssa_gym_b200.ukf import Q_discrete_white_noise_block, merwe_weights  # noqa: E402

VP = ctypes.c_void_p
TWIN_DIR = os.path.join(ROOT, "tests", "twin")
TWIN_LIB = os.path.join(TWIN_DIR, "libssa_twin.so")
ORACLE_DIR = os.path.join(ROOT, "oracle")
ORACLE_LIB = os.path.join(ORACLE_DIR, "liboracle.so")
GOLDEN = os.path.join(ROOT, "tests", "golden")

# SOFA cookbook matrix quoted by the reference (tests.py:107-109), used as a fixed trans_matrix
CEL2TER06AXY = np.array([[+0.973104317697536, +0.230363826239128, -0.000703163481769],
                         [-0.230363800456036, +0.973104570632801, +0.000118545368117],
                         [+0.000711560162594, +0.000046626402444, +0.999999745754024]])
OBSERVER_DEG = (38.828198, -77.305352, 20.0)  # envs/__init__.py:24
X6 = np.array([34090858.3, 23944774.4, 6503066.82, -1983.785080, 2150.41744, 913.881611])  # tests.py:130


def _newer(src_list, target):
    if not os.path.isfile(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in src_list if os.path.isfile(s))


def build_twin():
    csrc = os.path.join(ROOT, "ssa_gym_b200", "csrc")
    deps = [os.path.join(TWIN_DIR, "twin.cpp")] + [os.path.join(csrc, h) for h in
                                                    ("ssa_math.h", "ssa_orbit.h", "ssa_meas.h", "ssa_ukf_core.h")]
    if _newer(deps, TWIN_LIB):
        gxx = "/usr/bin/g++" if os.path.isfile("/usr/bin/g++") else "g++"
        cmd = [gxx, "-O2", "-std=c++17", "-ffp-contract=off", "-mfma", "-mavx2", "-fopenmp", "-shared", "-fPIC",
               "-Wno-unknown-pragmas", "-o", TWIN_LIB, os.path.join(TWIN_DIR, "twin.cpp")]
        subprocess.run(cmd, check=True, cwd=TWIN_DIR)
    return TWIN_LIB


def build_oracle():
    deps = [os.path.join(ORACLE_DIR, "ukf_oracle.c"), os.path.join(ROOT, "include", "ssa_ukf.h")]
    if _newer(deps, ORACLE_LIB):
        subprocess.run(["make", "-C", ORACLE_DIR, "-s"], check=True)
    return ORACLE_LIB


_cache = {}


def twin():
    if "twin" not in _cache:
        _cache["twin"] = ctypes.CDLL(build_twin())
    return _cache["twin"]


def oracle():
    if "oracle" not in _cache:
        _cache["oracle"] = ctypes.CDLL(build_oracle())
    return _cache["oracle"]


def p(a):
    return None if a is None else a.ctypes.data_as(VP)


def make_cfg(N, E=None, m=None, dt=20.0, alpha=1e-4, beta=2.0, kappa=-3.0, q_sigma=0.000025, R=None,
             observer_deg=OBSERVER_DEG, obs_limit_deg=-90.0, obs_type="aer", resample=True, reward_type="jones",
             n_steps=480):
    """ssa_ukf_cfg with the reference's default env_config (envs/__init__.py:23-28)."""
    if E is None:
        E, m = 1, N
    Wm, Wc, lam = merwe_weights(6, alpha, beta, kappa)
    c = _lib.SsaUkfCfg()
    c.abi_version = 1
    c.n_objects, c.n_envs, c.m = N, E, m
    c.obs_type = {"aer": 0, "xyz": 1}[obs_type]
    c.resample_after_predict = 1 if resample else 0
    c.reward_type = {"jones": 0, "trinary": 1, "shaped": 2}[reward_type]
    c.n_steps = n_steps
    c.dt, c.lam_plus_n = dt, lam
    for i in range(13):
        c.Wm[i], c.Wc[i] = Wm[i], Wc[i]
    Q = Q_discrete_white_noise_block(dt, q_sigma ** 2)
    for i, v in enumerate(Q.ravel()):
        c.Q[i] = v
    if R is None:
        R = np.diag([arcsec2rad ** 2] * 2 + [1e3 ** 2])
    R = np.asarray(R, dtype=float)
    if R.ndim == 1:
        R = np.tile(R, (3, 1))
    for i, v in enumerate(R.ravel()):
        c.R[i] = v
    lla = np.array([np.radians(observer_deg[0]), np.radians(observer_deg[1]), observer_deg[2]])
    oi = lla2ecef(lla)
    T = trans_uvw_ecef(lla[0], lla[1])
    for i in range(3):
        c.obs_itrs[i] = oi[i]
    for i, v in enumerate(np.asarray(T, dtype=float).ravel()):
        c.T[i] = v
    c.obs_limit = np.radians(obs_limit_deg)
    return c


IU = np.triu_indices(6)


def pack_P(Pfull):
    return np.ascontiguousarray(np.asarray(Pfull).reshape(-1, 6, 6)[:, IU[0], IU[1]])


def unpack_P(Ppacked):
    Pp = np.asarray(Ppacked).reshape(-1, 21)
    out = np.zeros((len(Pp), 6, 6))
    out[:, IU[0], IU[1]] = Pp
    out[:, IU[1], IU[0]] = Pp
    return out


class HostState:
    """Arrays of one batch in the reference's host layout (P full [N,6,6])."""

    def __init__(self, x_true, x, P):
        N = len(x_true)
        self.N = N
        self.x_true = np.ascontiguousarray(x_true, dtype=np.float64).copy()
        self.x = np.ascontiguousarray(x, dtype=np.float64).copy()
        P = np.asarray(P, dtype=np.float64)
        self.P = np.ascontiguousarray(np.broadcast_to(P, (N, 6, 6))).copy()
        self.status = np.zeros(N, np.int32)
        self.infl = np.zeros(N, np.int32)
        self.obs = np.zeros((N, 12))
        self.dpos, self.dvel, self.spos, self.svel, self.trace = (np.zeros(N) for _ in range(5))
        self.z_true = np.full((N, 3), np.nan)
        self.y = np.full((N, 3), np.nan)
        self.S = np.full((N, 3, 3), np.nan)
        self.sigmas_h = np.zeros((N, 13, 3))
        self.visible = np.zeros(N, np.uint8)
        self.updated = np.zeros(N, np.uint8)


def cpu_step(which, cfg, st, M, flags, actions=None, z_noise=None):
    """One batch step through the oracle ('oracle', P full) or the host twin ('twin', P packed)."""
    M = np.ascontiguousarray(M, dtype=np.float64)
    act = None if actions is None else np.ascontiguousarray(actions, dtype=np.int32)
    zn = None if z_noise is None else np.ascontiguousarray(z_noise, dtype=np.float64)
    if which == "oracle":
        fn, P = oracle().oracle_step, st.P
    else:
        fn, P = twin().twin_step, pack_P(st.P)
    fn(ctypes.byref(cfg), p(M), ctypes.c_int(flags), p(st.x_true), p(st.x), p(P), p(st.status), p(st.infl), p(act), p(zn),
       p(st.obs), p(st.dpos), p(st.dvel), p(st.spos), p(st.svel), p(st.trace), p(st.z_true), p(st.y), p(st.S),
       p(st.sigmas_h), p(st.visible), p(st.updated))
    if which != "oracle":
        st.P = unpack_P(P)
    return st


def lib_fx(which, x, dt):
    x = np.ascontiguousarray(x, dtype=np.float64).reshape(-1, 6)
    out = np.empty_like(x)
    exc = np.zeros(len(x), np.int32)
    if which == "gpu":
        _lib.check(_lib.require_gpu().ssa_unit_fx(p(x), float(dt), p(out), p(exc), len(x), 0), "ssa_unit_fx")
    else:
        L, name = (oracle(), "oracle_fx") if which == "oracle" else (twin(), "twin_fx")
        getattr(L, name)(p(x), ctypes.c_double(dt), p(out), p(exc), ctypes.c_int(len(x)))
    return out, exc


def lib_hx(which, x, M, obs_itrs, T):
    x = np.ascontiguousarray(x, dtype=np.float64).reshape(-1, 6)
    M = np.ascontiguousarray(M, dtype=np.float64)
    oi = np.ascontiguousarray(obs_itrs, dtype=np.float64)
    T = np.ascontiguousarray(T, dtype=np.float64)
    out = np.empty((len(x), 3))
    if which == "gpu":
        _lib.check(_lib.require_gpu().ssa_unit_hx_aer(p(x), 6, p(M), p(oi), p(T), p(out), len(x), 0), "ssa_unit_hx_aer")
    else:
        L, name = (oracle(), "oracle_hx_aer") if which == "oracle" else (twin(), "twin_hx_aer")
        getattr(L, name)(p(x), p(M), p(oi), p(T), p(out), ctypes.c_int(len(x)))
    return out


MATH_OPS = ["sin", "cos", "tan", "atan", "asin", "acos", "exp", "log", "sinh", "cosh", "tanh", "atanh", "asinh",
            "acosh", "pow23", "atan2", "pymod"]


def lib_math(which, op, a, b=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    b = None if b is None else np.ascontiguousarray(b, dtype=np.float64)
    out = np.empty_like(a)
    if which == "gpu":
        _lib.check(_lib.require_gpu().ssa_unit_math(MATH_OPS.index(op), p(a), p(b), p(out), a.size, 0), "ssa_unit_math")
    else:
        fn = getattr(twin(), "twin_" + op)
        if b is None:
            fn(p(a), p(out), ctypes.c_int(a.size))
        else:
            fn(p(a), p(b), p(out), ctypes.c_int(a.size))
    return out


def c2_inputs(N=20000, steps=1, catalog=None):
    """SURVEY 8(d) C2 inputs: x_filter = x_true + RandomState(0).normal * x_sigma, P0, z_noise from RandomState(1)."""
    from ssa_gym_b200.catalog import synthetic_catalog
    cat = synthetic_catalog(N, 0) if catalog is None else np.asarray(catalog)[:N]
    x = cat + np.random.RandomState(0).normal(size=(N, 6)) * np.array([1e5] * 3 + [1e2] * 3)
    P0 = np.diag([1e10] * 3 + [1e4] * 3)
    zn = np.random.RandomState(1).normal(size=(steps, N, 3)) * np.array([arcsec2rad, arcsec2rad, 1e3])
    return cat, x, P0, zn


def bits_equal(a, b):
    """Bit-for-bit equality of float arrays.  NaNs must sit in the same places; their sign/payload is not
    compared (an x86 SSE operation generates the 'indefinite' NaN 0xFFF8..., an sm_100a one 0x7FF8...)."""
    a = np.ascontiguousarray(a)
    b = np.ascontiguousarray(b)
    if a.shape != b.shape:
        return False
    if a.dtype.kind == "f":
        na, nb = np.isnan(a), np.isnan(b)
        if not np.array_equal(na, nb):
            return False
        return np.array_equal(np.where(na, 0.0, a).view(np.uint64), np.where(nb, 0.0, b).view(np.uint64))
    return np.array_equal(a, b)


def gpu_available():
    try:
        return _lib.load().ssa_ukf_device_count() > 0
    except Exception:
        return False


class TwinBackedUKF:
    """Same interface as ssa_gym_b200.ukf.BatchedUKF, executed by the host twin (tests only).  Lets the tests run
    the SAME environment code once on the GPU and once on the twin and demand equality of whole episodes."""

    def __init__(self, n_envs, m, dt, Q, R, obs_lla, obs_limit_rad, alpha=1e-4, beta=2.0, kappa=-3.0, obs_type="aer",
                 reward_type="jones", n_steps=480, resample_after_predict=True, device=0):
        from ssa_gym_b200 import _lib as F
        self.F = F
        self.N, self.m, self.n_envs = n_envs * m, m, n_envs
        Wm, Wc, lam = merwe_weights(6, alpha, beta, kappa)
        c = _lib.SsaUkfCfg()
        c.abi_version, c.n_objects, c.n_envs, c.m = 1, self.N, n_envs, m
        c.obs_type = {"aer": 0, "xyz": 1}[obs_type]
        c.resample_after_predict = 1 if resample_after_predict else 0
        c.reward_type, c.n_steps, c.dt, c.lam_plus_n = 0, n_steps, dt, lam
        for i in range(13):
            c.Wm[i], c.Wc[i] = Wm[i], Wc[i]
        for i, v in enumerate(np.asarray(Q, dtype=float).ravel()):
            c.Q[i] = v
        R = np.asarray(R, dtype=float)
        if R.ndim == 1:
            R = np.tile(R, (3, 1))
        for i, v in enumerate(R.ravel()):
            c.R[i] = v
        lla = np.asarray(obs_lla, dtype=float)
        for i, v in enumerate(lla2ecef(lla)):
            c.obs_itrs[i] = v
        for i, v in enumerate(np.asarray(trans_uvw_ecef(lla[0], lla[1]), dtype=float).ravel()):
            c.T[i] = v
        c.obs_limit = obs_limit_rad
        self.cfg = c
        self.st = None
        self.actions = np.zeros(n_envs, np.int32)
        self.z_noise = np.zeros((self.N, 3))

    def reset(self, x_true, x_filter, P0, stream=None):
        self.st = HostState(np.reshape(x_true, (self.N, 6)), np.reshape(x_filter, (self.N, 6)), P0)

    def upload(self, field, arr, stream=None):
        F = self.F
        if field == F.F_ACTIONS:
            self.actions = np.ascontiguousarray(arr, dtype=np.int32).reshape(self.n_envs)
        elif field == F.F_Z_NOISE:
            self.z_noise = np.ascontiguousarray(arr, dtype=np.float64).reshape(self.N, 3)
        else:
            raise NotImplementedError

    def step(self, M, flags, stream=None):
        cpu_step("twin", self.cfg, self.st, np.asarray(M, dtype=float).reshape(3, 3), flags, actions=self.actions,
                 z_noise=self.z_noise)

    def download(self, field, out=None, stream=None):
        F, st = self.F, self.st
        m = {F.F_X_TRUE: st.x_true, F.F_X_FILTER: st.x, F.F_P_FILTER: st.P, F.F_OBS: st.obs, F.F_DELTA_POS: st.dpos,
             F.F_DELTA_VEL: st.dvel, F.F_SIGMA_POS: st.spos, F.F_SIGMA_VEL: st.svel, F.F_TRACE: st.trace,
             F.F_Z_TRUE: st.z_true, F.F_Y: st.y, F.F_S: st.S, F.F_SIGMAS_H: st.sigmas_h, F.F_VISIBLE: st.visible,
             F.F_UPDATED: st.updated, F.F_STATUS: st.status, F.F_INFLATIONS: st.infl}
        return m[field].copy()

    def snapshot(self, stream=None):
        st = self.st
        return {"x_true": st.x_true.copy(), "x_filter": st.x.copy(), "P_filter": st.P.copy(), "obs": st.obs.copy(),
                "delta_pos": st.dpos.copy(), "delta_vel": st.dvel.copy(), "sigma_pos": st.spos.copy(),
                "sigma_vel": st.svel.copy(), "z_true": st.z_true.copy(), "y": st.y.copy(), "S": st.S.copy(),
                "sigmas_h": st.sigmas_h.copy(), "status": st.status.copy(), "visible": st.visible.copy(),
                "updated": st.updated.copy()}

    def sync(self, stream=None):
        pass

    def close(self):
        pass


# ---- agent_shannon and the per-environment reductions in the device's arithmetic ---------------------------------
def twin_det6(P):
    """ssa_det6_sym of each covariance (full [N,6,6] or packed [N,21]) through the host twin: bit-equal to the device."""
    P = np.asarray(P, dtype=np.float64)
    Pp = np.ascontiguousarray(pack_P(P) if P.shape[-2:] == (6, 6) else P.reshape(-1, 21))
    out = np.empty(len(Pp))
    twin().twin_det6_sym(p(Pp), p(out), len(Pp))
    return out


def twin_log_ratio(det, prev):
    """ssa_log(ssa_div(det, prev)) elementwise (numpy's log is not bit-equal to ssa_log, test_math_accuracy.py)."""
    det = np.ascontiguousarray(det, dtype=np.float64)
    prev = np.ascontiguousarray(np.broadcast_to(prev, det.shape), dtype=np.float64)
    out = np.empty_like(det)
    twin().twin_log_ratio(p(det), p(prev), p(out), det.size)
    return out


class ShannonHistory:
    """The determinant history of SSA_TASKER_SHANNON (include/ssa_ukf.h) for E environments of m objects: `last` is
    det P at step `step[e]`, `prev` the denominator of that step's ratio.  A larger step shifts the history, the same
    step re-reads it, step 0 / a smaller step / no history (step -1) restarts it with ratio 1."""

    def __init__(self, E, m):
        self.E, self.m = E, m
        self.prev, self.last = np.zeros((E, m)), np.zeros((E, m))
        self.step = np.full(E, -1, np.int64)

    def scores(self, P, steps, sel=None):
        """log(det P / det P_prev) [E, m] at the per-env step indices `steps`; only the environments in `sel` (bool
        [E], default all) are evaluated and move their history, the others' rows are NaN."""
        E, m = self.E, self.m
        sel = np.ones(E, bool) if sel is None else np.asarray(sel, bool)
        steps = np.asarray(steps, dtype=np.int64)
        det = twin_det6(P).reshape(E, m)
        restart = (steps <= 0) | (self.step < 0) | (steps < self.step)
        shift = ~restart & (steps > self.step)
        prev = np.where(restart[:, None], det, np.where(shift[:, None], self.last, self.prev))
        last = np.where(restart[:, None] | shift[:, None], det, self.last)
        out = np.full((E, m), np.nan)
        out[sel] = twin_log_ratio(det[sel], prev[sel])
        self.prev[sel], self.last[sel], self.step[sel] = prev[sel], last[sel], steps[sel]
        return out


def first_visible_argmax(score, vis):
    """The visible-* rule of ssa_env_reduce_kernel for one environment: the first maximum of `score` among the visible
    objects, a NaN score ordered like +inf (np.argmax: NaN wins); -1 where agents.py:37 `not np.any(idx)` samples."""
    idx = np.where(vis)[0]
    if not np.any(idx):
        return -1
    s = np.asarray(score, dtype=np.float64)[idx]
    return int(idx[np.argmax(np.where(np.isnan(s), np.inf, s))])


def emu_env_reduce(st, E, m, step_idx, reward_type, n_steps, shannon=None, sel=None):
    """numpy restatement of ssa_env_reduce_kernel (SS2:324-354, agents.py:7-81) on twin outputs.  `shannon` is the
    ShannonHistory that the call advances (its column stays -1 without one); `sel` restricts the Shannon history to
    the environments a refresh re-evaluates."""
    dpos = st.dpos.reshape(E, m); dvel = st.dvel.reshape(E, m); tr = st.trace.reshape(E, m)
    vis = st.visible.reshape(E, m).astype(bool)
    max_dpos = dpos.max(1)
    tri = ((dpos < 1e4).astype(int) + (dpos < 1e7).astype(int)).sum(1)
    trinary = (tri.astype(float) / float(m)) / 2.0
    reward = np.zeros(E); done = np.zeros(E, bool)
    if reward_type == "jones":
        hi, lo = max_dpos > 5e6, max_dpos < 3e4
        done |= hi | lo
        reward[lo & ~hi] = 1.0
    else:
        reward = trinary
    done |= (np.asarray(step_idx) + 1 >= n_steps)
    greedy = np.full((E, _lib.N_TASKERS), -1, np.int32)
    greedy[:, _lib.TASKER_NAIVE_GREEDY] = tr.argmax(1)
    sh = shannon.scores(st.P, step_idx, sel) if shannon is not None else None
    for e in range(E):
        greedy[e, _lib.TASKER_VISIBLE_GREEDY] = first_visible_argmax(tr[e], vis[e])
        greedy[e, _lib.TASKER_POS_ERROR_GREEDY] = first_visible_argmax(dpos[e], vis[e])
        greedy[e, _lib.TASKER_VEL_ERROR_GREEDY] = first_visible_argmax(dvel[e], vis[e])
        greedy[e, _lib.TASKER_VISIBLE_GREEDY_AER] = first_visible_argmax(
            np.nan_to_num(tr[e], nan=0.001, posinf=0.001, neginf=0.001), vis[e])
        if sh is not None:
            greedy[e, _lib.TASKER_SHANNON] = first_visible_argmax(sh[e], vis[e])
    return reward, done, greedy


_REFRESHED = ("obs", "dpos", "dvel", "spos", "svel", "trace", "visible", "updated")


class EpisodicTwin:
    """Step-by-step host statement of the device-resident episodic mode (ssa_ukf_rollout_reset / ssa_ukf_rollout_step)
    of a VecSSATaskerEnv(rng='device'): the same counter-based draws (twin_env_reset / twin_env_noise), twin_step with
    the env's trans_matrix row, numpy reward / done / greedy taskers including agent_shannon's determinant history.
    After an auto-reset only the re-drawn environments are refreshed: the others keep this step's outputs."""

    def __init__(self, vec, cfg):
        self.E, self.m, self.n = vec.E, vec.m, vec.n
        self.N = self.E * self.m
        self.reward_type, self.update_interval = cfg["reward_type"], cfg["update_interval"]
        self.keys = np.array(vec.init_seeds, dtype=np.uint64)
        self.table = np.ascontiguousarray(vec.trans_matrix).reshape(self.n, 9)
        self.sig = np.concatenate([vec.x_sigma, vec.z_sigma, vec.P_0[np.triu_indices(6)]])
        self.orbits = np.ascontiguousarray(vec.orbits, dtype=np.float64)
        self.cfg = make_cfg(self.N, E=self.E, m=self.m, dt=cfg["time_step"], alpha=cfg["alpha"], beta=cfg["beta"],
                            kappa=cfg["kappa"], q_sigma=cfg["q_sigma"], R=vec.R, observer_deg=cfg["observer"],
                            obs_limit_deg=cfg["obs_limit"], n_steps=self.n)
        self.episode = np.zeros(self.E, np.uint32)
        self.step_idx = np.zeros(self.E, np.int32)
        self.shannon = ShannonHistory(self.E, self.m)
        self.st = None

    def _draw(self, done):
        N, tw = self.N, twin()
        xt, xf, Pp = np.zeros((N, 6)), np.zeros((N, 6)), np.zeros((N, 21))
        status, infl = np.zeros(N, np.int32), np.zeros(N, np.int32)
        d8 = None if done is None else np.ascontiguousarray(done, dtype=np.uint8)
        tw.twin_env_reset(self.E, self.m, p(self.keys), p(self.episode), p(self.step_idx), p(d8), p(self.orbits),
                          len(self.orbits), p(self.sig), p(xt), p(xf), p(Pp), p(status), p(infl))
        if self.st is None:
            self.st = HostState(xt, xf, unpack_P(Pp))
            return
        rows = np.repeat(np.asarray(done, bool), self.m)
        st = self.st
        st.x_true[rows] = xt[rows]; st.x[rows] = xf[rows]; st.P[rows] = unpack_P(Pp)[rows]
        st.status[rows] = 0; st.infl[rows] = 0

    def _refresh(self, envs):
        """obs / errors / visibility of the fresh objects of `envs` (bool [E]) and their greedy taskers."""
        st, rows = self.st, np.repeat(envs, self.m)
        keep = {k: getattr(st, k).copy() for k in _REFRESHED}
        cpu_step("twin", self.cfg, st, self.table[np.minimum(self.step_idx, self.n - 1)].reshape(self.E, 9),
                 _lib.STEP_EPILOGUE | _lib.STEP_M_PER_ENV)
        for k, v in keep.items():
            getattr(st, k)[~rows] = v[~rows]
        _, _, g = emu_env_reduce(st, self.E, self.m, self.step_idx, self.reward_type, self.n, self.shannon, envs)
        self.greedy[envs] = g[envs]

    def reset(self):
        """rollout_reset: every environment drawn, step index 0; returns obs [N, 12] and greedy [E, taskers]."""
        self._draw(None)
        self.greedy = np.full((self.E, _lib.N_TASKERS), -1, np.int32)
        self._refresh(np.ones(self.E, bool))
        return self.st.obs.copy(), self.greedy.copy()

    def step(self, actions, auto_reset=True):
        """rollout_step; returns obs [N, 12], reward [E], done [E], greedy [E, taskers] as the device's output block."""
        E, m, st = self.E, self.m, self.st
        zn = np.zeros((self.N, 3))
        twin().twin_env_noise(E, m, p(self.keys), p(self.episode), p(self.step_idx), p(self.sig), p(zn))
        nxt = self.step_idx + 1
        a_eff = np.where(nxt % self.update_interval == 0, actions, -1).astype(np.int32)
        cpu_step("twin", self.cfg, st, self.table[np.minimum(nxt, self.n - 1)].reshape(E, 9),
                 _lib.STEP_TRUTH | _lib.STEP_PREDICT | _lib.STEP_UPDATE_ACT | _lib.STEP_EPILOGUE | _lib.STEP_M_PER_ENV,
                 actions=a_eff, z_noise=zn)
        self.step_idx[:] = nxt
        reward, done, self.greedy = emu_env_reduce(st, E, m, self.step_idx, self.reward_type, self.n, self.shannon)
        if auto_reset and done.any():
            self._draw(done)
            self._refresh(done)
        return st.obs.copy(), reward, done, self.greedy.copy()


def episodic_vs_twin(cfg, E, total_steps, seed0=500, action_seed=11):
    """Run VecSSATaskerEnv(cfg, E, rng='device') and EpisodicTwin side by side (actions alternate between random and
    the device's visible-greedy picks) and demand equality at every step: observations, rewards, dones and all six
    greedy columns exact, vec.i equal to the step counters; at the end x, x_true, P, status, inflation counts, updated
    and visible.  Returns counters of what the run went through (auto-resets, environments with nothing / only
    object 0 visible after a step)."""
    from ssa_gym_b200.vec_env import VecSSATaskerEnv
    vec = VecSSATaskerEnv(cfg, E, seeds=list(range(seed0, seed0 + E)), rng="device")
    emu = EpisodicTwin(vec, cfg)
    E, m, N = emu.E, emu.m, emu.N
    obs_e, g_e = emu.reset()
    assert bits_equal(vec.obs.reshape(N, 12), obs_e)
    assert np.array_equal(vec._io["greedy"], g_e), (vec._io["greedy"], g_e)
    rng = np.random.RandomState(action_seed)
    seen = {"resets": 0, "none_visible": 0, "only_object_0": 0}
    for t in range(total_steps):
        a = vec.greedy_actions(_lib.TASKER_VISIBLE_GREEDY) if t % 2 else rng.randint(0, m, size=E)
        a = np.asarray(a, dtype=np.int32)
        obs_v, r_v, d_v, _ = vec.vector_step(a)
        obs_e, r_e, d_e, g_e = emu.step(a)
        assert np.array_equal(d_v, d_e), (t, d_v, d_e)
        assert bits_equal(r_v, r_e), (t, r_v, r_e)
        assert bits_equal(obs_v.reshape(N, 12), obs_e), t
        g_v = vec._io["greedy"]
        for k in range(_lib.N_TASKERS):
            assert np.array_equal(g_v[:, k], g_e[:, k]), (t, k, np.where(g_v[:, k] != g_e[:, k])[0], g_v[:, k], g_e[:, k])
        assert np.array_equal(vec.i, emu.step_idx), t
        vis = emu.st.visible.reshape(E, m).astype(bool)
        seen["resets"] += int(d_e.sum())
        seen["none_visible"] += int((~vis.any(1)).sum())
        seen["only_object_0"] += int((vis[:, 0] & ~vis[:, 1:].any(1)).sum())
    st, u = emu.st, vec.ukf
    assert bits_equal(u.download(_lib.F_X_FILTER), st.x) and bits_equal(u.download(_lib.F_X_TRUE), st.x_true)
    assert bits_equal(pack_P(u.download(_lib.F_P_FILTER)), pack_P(st.P))
    for f, a in ((_lib.F_STATUS, st.status), (_lib.F_INFLATIONS, st.infl), (_lib.F_UPDATED, st.updated),
                 (_lib.F_VISIBLE, st.visible)):
        assert np.array_equal(u.download(f).reshape(a.shape), a), f
    vec.close()
    return seen


def scores_det_restated(P):
    """score_det_P and score_det_pos_P of ssa_scores_kernel restated in its operation order (plain IEEE double
    operations, the library is built with -fmad=false): the 3x3 cofactor formula of the position block and a 6x6
    Gaussian elimination with partial pivoting.  Bit-equal to the device; returns (det6 [N], det3 [N])."""
    P = np.asarray(P, dtype=np.float64).reshape(-1, 6, 6)
    det6, det3 = np.empty(len(P)), np.empty(len(P))
    for n in range(len(P)):
        a = [[float(P[n][min(i, j)][max(i, j)]) for j in range(6)] for i in range(6)]  # the upper triangle, mirrored
        m00, m01, m02, m11, m12, m22 = a[0][0], a[0][1], a[0][2], a[1][1], a[1][2], a[2][2]
        det3[n] = m00 * (m11 * m22 - m12 * m12) - m01 * (m01 * m22 - m12 * m02) + m02 * (m01 * m12 - m11 * m02)
        det = 1.0
        for c in range(6):
            pv = c
            for i in range(c + 1, 6):
                if abs(a[i][c]) > abs(a[pv][c]):
                    pv = i
            if pv != c:
                a[c], a[pv] = a[pv], a[c]
                det = -det
            det *= a[c][c]
            if a[c][c] == 0.0:
                break
            rp = 1.0 / a[c][c]
            for i in range(c + 1, 6):
                lf = a[i][c] * rp
                for j in range(c + 1, 6):
                    a[i][j] -= lf * a[c][j]
        det6[n] = det
    return det6, det3


def exact_det(A):
    """Exact determinant (fractions.Fraction) of a square float matrix: every double is an exact rational."""
    from fractions import Fraction
    a = [[Fraction(float(v)) for v in row] for row in np.asarray(A)]
    n, det = len(a), Fraction(1)
    for c in range(n):
        pv = next((r for r in range(c, n) if a[r][c] != 0), None)
        if pv is None:
            return Fraction(0)
        if pv != c:
            a[c], a[pv] = a[pv], a[c]
            det = -det
        det *= a[c][c]
        for r in range(c + 1, n):
            lf = a[r][c] / a[c][c]
            if lf:
                for k in range(c, n):
                    a[r][k] -= lf * a[c][k]
    return det


def rel_err_exact(value, exact):
    """|value - exact| / |exact| computed exactly, rounded once to float (0 / inf when exact is 0)."""
    from fractions import Fraction
    if exact == 0:
        return 0.0 if value == 0 else np.inf
    if not np.isfinite(value):
        return np.inf
    return float(abs(Fraction(float(value)) - exact) / abs(exact))


def corr_cond(P):
    """Condition number of the correlation matrices of P [N, k, k] (scale-free conditioning of a determinant)."""
    P = np.asarray(P, dtype=np.float64)
    d = np.sqrt(np.abs(np.einsum("nii->ni", P)))
    return np.linalg.cond(P / (d[:, :, None] * d[:, None, :]))
