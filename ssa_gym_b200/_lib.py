"""ctypes binding of libssa_ukf.so (include/ssa_ukf.h).  Fails loudly: there is no CPU fallback.

Loading the library does not need a GPU (the test suite checks that every symbol of the header is
exported on a CPU-only box); creating a handle or calling a unit entry point does.
"""
import ctypes
import os

from . import _build

c_double_p = ctypes.POINTER(ctypes.c_double)
c_void_p = ctypes.c_void_p

SSA_UKF_ABI_VERSION = 1
SSA_OK, SSA_EINVAL, SSA_ECUDA, SSA_ENOMEM, SSA_ENODEV = 0, -1, -2, -3, -4
OBS_AER, OBS_XYZ = 0, 1
REWARD_JONES, REWARD_TRINARY, REWARD_SHAPED = 0, 1, 2
ST_FAILED, ST_LINALG, ST_NAN, ST_FXEXC, ST_TRUTHEXC, ST_IN_UPDATE = 0x1, 0x2, 0x4, 0x8, 0x10, 0x20
STEP_TRUTH, STEP_PREDICT, STEP_UPDATE_ALL, STEP_UPDATE_ACT, STEP_EPILOGUE, STEP_RECORD = 0x1, 0x2, 0x4, 0x8, 0x10, 0x20
STEP_M_PER_ENV = 0x40
STEP_NO_D2H = 0x80
STEP_CATALOG_STATS = 0x100
N_TASKERS = 6
(TASKER_NAIVE_GREEDY, TASKER_VISIBLE_GREEDY, TASKER_POS_ERROR_GREEDY, TASKER_VEL_ERROR_GREEDY, TASKER_VISIBLE_GREEDY_AER,
 TASKER_SHANNON) = range(6)
TASKER_EXTERNAL = -1  # episodic mode only (ssa_ukf_rollout_tasker): the caller's actions, and the random agents
TASKER_NAIVE_RANDOM, TASKER_VISIBLE_RANDOM, TASKER_VISIBLE_GREEDY_SPOILED = 6, 7, 8

(F_X_TRUE, F_X_FILTER, F_P_FILTER, F_OBS, F_DELTA_POS, F_DELTA_VEL, F_SIGMA_POS, F_SIGMA_VEL, F_TRACE,
 F_Z_TRUE, F_Y, F_S, F_SIGMAS_H, F_Z_NOISE, F_VISIBLE, F_STATUS, F_INFLATIONS, F_ACTIONS, F_REWARD, F_DONE,
 F_GREEDY, F_SCORES, F_UPDATED, F_TRANS_ENV, F_STEP_INDEX, F_ENV_STATS, F_DIAG, F_INNOV_FLAGS, F_CATALOG_STATS,
 F_ROLLOUT_OBS, F_ROLLOUT_REWARD, F_ROLLOUT_ACTIONS, F_ROLLOUT_DONE, F_ROLLOUT_GREEDY, F_ROLLOUT_OBS_AER,
 F_ROLLOUT_EPISODE_STATS, F_ROLLOUT_TERMINAL_OBS, F_ROLLOUT_TRUNCATED, F_ROLLOUT_OBS_NORM, F_ROLLOUT_REWARD_NORM,
 F_ROLLOUT_TERMINAL_OBS_NORM, F_ROLLOUT_NORM_STATE) = range(42)
ROLLOUT_DEVICE_IO = 2
ROLLOUT_OBS_F32 = 4
ROLLOUT_OBS_AER = 8
EPISODE_STATS_DOUBLES = 23
NORM_OBS_ROWS, NORM_OBS_ROWS_F32, NORM_OBS_AER = 0, 1, 2


class SsaUkfCfg(ctypes.Structure):
    """Mirror of `struct ssa_ukf_cfg` (include/ssa_ukf.h)."""
    _fields_ = [
        ("abi_version", ctypes.c_int32), ("n_objects", ctypes.c_int32), ("n_envs", ctypes.c_int32),
        ("m", ctypes.c_int32), ("obs_type", ctypes.c_int32), ("resample_after_predict", ctypes.c_int32),
        ("reward_type", ctypes.c_int32), ("n_steps", ctypes.c_int32),
        ("dt", ctypes.c_double), ("lam_plus_n", ctypes.c_double),
        ("Wm", ctypes.c_double * 13), ("Wc", ctypes.c_double * 13),
        ("Q", ctypes.c_double * 36), ("R", ctypes.c_double * 9),
        ("obs_itrs", ctypes.c_double * 3), ("T", ctypes.c_double * 9), ("obs_limit", ctypes.c_double),
    ]


class SsaNormCfg(ctypes.Structure):
    """Mirror of `struct ssa_norm_cfg` (include/ssa_ukf.h)."""
    _fields_ = [
        ("norm_obs", ctypes.c_int32), ("norm_reward", ctypes.c_int32), ("training", ctypes.c_int32),
        ("obs_layout", ctypes.c_int32), ("reward_nan_to_num", ctypes.c_int32),
        ("clip_obs", ctypes.c_double), ("clip_reward", ctypes.c_double), ("gamma", ctypes.c_double), ("epsilon", ctypes.c_double),
    ]


# every symbol include/ssa_ukf.h declares: name -> (restype, argtypes)
_I, _L, _D = ctypes.c_int, ctypes.c_long, ctypes.c_double
_SZ = ctypes.c_size_t
PROTOTYPES = {
    "ssa_ukf_abi_version": (_I, []),
    "ssa_ukf_last_error": (ctypes.c_char_p, []),
    "ssa_ukf_device_count": (_I, []),
    "ssa_ukf_create": (_I, [ctypes.POINTER(SsaUkfCfg), _I, ctypes.POINTER(c_void_p)]),
    "ssa_ukf_destroy": (_I, [c_void_p]),
    "ssa_ukf_ld": (_L, [c_void_p]),
    "ssa_ukf_reset": (_I, [c_void_p, c_void_p, c_void_p, c_void_p, _I, c_void_p]),
    "ssa_ukf_upload": (_I, [c_void_p, _I, c_void_p, _SZ, c_void_p]),
    "ssa_ukf_download": (_I, [c_void_p, _I, c_void_p, _SZ, c_void_p]),
    "ssa_ukf_device_ptr": (_I, [c_void_p, _I, ctypes.POINTER(c_void_p), ctypes.POINTER(_SZ)]),
    "ssa_ukf_step": (_I, [c_void_p, c_void_p, _I, c_void_p]),
    "ssa_ukf_step_profile": (_I, [c_void_p, c_void_p, _I, c_void_p, c_double_p]),
    "ssa_ukf_step_host": (_I, [c_void_p, c_void_p, _I, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "ssa_ukf_host_join": (_I, [c_void_p, c_void_p]),
    "ssa_ukf_host_io": (_I, [c_void_p, _I] + [c_void_p] * 6),
    "ssa_ukf_host_stats": (_I, [c_void_p, _I, c_void_p, c_void_p]),
    "ssa_ukf_step_pinned": (_I, [c_void_p, _I, c_void_p, c_void_p]),
    "ssa_ukf_rollout_config": (_I, [c_void_p, c_void_p, _I, c_void_p, _I, c_void_p, c_void_p, c_void_p, c_void_p, _I]),
    "ssa_ukf_rollout_io": (_I, [c_void_p] + [c_void_p] * 5),
    "ssa_ukf_rollout_reset": (_I, [c_void_p, c_void_p]),
    "ssa_ukf_rollout_step": (_I, [c_void_p, _I, c_void_p]),
    "ssa_ukf_rollout_tasker": (_I, [c_void_p, _I, _D]),
    "ssa_ukf_rollout_obs_f32": (_I, [c_void_p, c_void_p, c_void_p]),
    "ssa_ukf_rollout_obs_aer": (_I, [c_void_p, c_void_p, c_void_p]),
    "ssa_ukf_rollout_episode_stats_enable": (_I, [c_void_p]),
    "ssa_ukf_rollout_episode_stats_download": (_I, [c_void_p, c_void_p, _I, c_void_p, c_void_p]),
    "ssa_ukf_rollout_truncated": (_I, [c_void_p, c_void_p, c_void_p]),
    "ssa_ukf_rollout_terminal_obs_download": (_I, [c_void_p, c_void_p, _I, c_void_p, c_void_p]),
    "ssa_ukf_rollout_reset_envs": (_I, [c_void_p, c_void_p, _I, c_void_p]),
    "ssa_ukf_rollout_normalize": (_I, [c_void_p, ctypes.POINTER(SsaNormCfg)]),
    "ssa_ukf_rollout_norm_io": (_I, [c_void_p, c_void_p, c_void_p]),
    "ssa_ukf_rollout_norm_state_download": (_I, [c_void_p, c_void_p, _SZ, c_void_p]),
    "ssa_ukf_rollout_norm_state_upload": (_I, [c_void_p, c_void_p, _SZ, c_void_p]),
    "ssa_ukf_rollout_terminal_obs_norm_download": (_I, [c_void_p, c_void_p, _I, c_void_p, c_void_p]),
    "ssa_trans_matrix_table": (_I, [_I, _I, _I, _D, _D, _I, c_void_p, _I, c_void_p]),
    "ssa_ukf_predict": (_I, [c_void_p, c_void_p]),
    "ssa_ukf_update": (_I, [c_void_p, c_void_p, _I, c_void_p]),
    "ssa_ukf_env_reduce": (_I, [c_void_p, c_void_p, _I, c_void_p]),
    "ssa_ukf_scores": (_I, [c_void_p, c_void_p]),
    "ssa_ukf_diagnostics": (_I, [c_void_p, c_void_p]),
    "ssa_ukf_catalog_stats": (_I, [c_void_p, _L, c_void_p]),
    "ssa_innovation_stats": (_I, [c_void_p, c_void_p, _I, _I, _I, c_void_p, c_void_p, _I]),
    "ssa_ukf_snapshot_bytes": (ctypes.c_size_t, [c_void_p]),
    "ssa_ukf_snapshot": (_I, [c_void_p, c_void_p, ctypes.c_size_t, c_void_p]),
    "ssa_orbit_gen_eval": (_I, [c_void_p, _I, c_void_p, _I, _D, c_void_p, c_void_p, _D, _D, _I, _I, c_void_p, c_void_p, c_void_p, _I]),
    "ssa_ukf_sync": (_I, [c_void_p, c_void_p]),
    "ssa_ukf_launch_count": (_L, [c_void_p]),
    "ssa_ukf_fp64_peak": (_I, [_I, c_void_p, c_double_p]),
    "ssa_unit_math": (_I, [_I, c_void_p, c_void_p, c_void_p, _I, _I]),
    "ssa_unit_fx": (_I, [c_void_p, _D, c_void_p, c_void_p, _I, _I]),
    "ssa_unit_hx_aer": (_I, [c_void_p, _I, c_void_p, c_void_p, c_void_p, c_void_p, _I, _I]),
    "ssa_unit_aer": (_I, [_I, c_void_p, c_void_p, c_void_p, _I, _I]),
    "ssa_unit_robust_chol": (_I, [c_void_p, _D, c_void_p, c_void_p, _I, _I]),
    "ssa_unit_inv3": (_I, [c_void_p, c_void_p, c_void_p, _I, _I]),
}

_lib = None


class SsaUkfError(RuntimeError):
    pass


def load():
    """Load (building if the .so is missing and nvcc is present) and type the C ABI."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("SSA_UKF_LIB") or _build.LIB  # SSA_UKF_LIB: alternative in-tree build (tuning experiments)
    if not os.path.isfile(path):
        path = _build.build()
    try:
        lib = ctypes.CDLL(path)
    except OSError as e:  # e.g. libcudart missing
        raise SsaUkfError(f"cannot load {path}: {e}.  The UKF hot path has no CPU fallback.") from e
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the header and the library disagree
        fn.restype = res
        fn.argtypes = args
    if lib.ssa_ukf_abi_version() != SSA_UKF_ABI_VERSION:
        raise SsaUkfError("libssa_ukf.so ABI version mismatch")
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        msg = load().ssa_ukf_last_error().decode("utf8", "replace")
        names = {SSA_EINVAL: "EINVAL", SSA_ECUDA: "ECUDA", SSA_ENOMEM: "ENOMEM", SSA_ENODEV: "ENODEV"}
        raise SsaUkfError(f"{what} failed with {names.get(rc, rc)}: {msg}")


def require_gpu():
    """Raise if no CUDA device is visible (used by every product entry point)."""
    lib = load()
    if lib.ssa_ukf_device_count() <= 0:
        raise SsaUkfError("no CUDA device visible: ssa_gym_b200 runs the UKF hot path only on the GPU "
                          "(no CPU fallback by design)")
    return lib
