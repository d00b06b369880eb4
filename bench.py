#!/usr/bin/env python
"""bench.py — the headline metric of BASELINE.json on B200: RSO UKF predict+update per second.

A "step" = one pass of the hot path (truth fx + UKF predict + UKF update + obs/error epilogue) over the whole
catalog.  Default workload = BASELINE.json configs[3] (SURVEY.md 8d "C4"): a 1 000 000-object synthetic catalog,
every object predicted and updated once per step, sharded in contiguous blocks over the N ranks (STRONG scaling:
the catalog is fixed, N = 1 holds all of it on one GPU); every step also reduces the shard's reward terms on the
device (ssa_ukf_catalog_stats) and all-gathers them over NCCL — both inside the timed CUDA events.  Objects never
couple (SURVEY 8e), so that gather is the only collective.  Rank 0 prints ONE JSON line; C2 (the 20 000-orbit
catalog) and C3 (4 096 vectorised environments) are measured briefly on rank 0 and reported under `extra`.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c4|c2|c3] [--impl reference] [--dump-outputs DIR]

`--impl reference` times the CPU oracle port of the reference's algorithm (oracle/ukf_oracle.c, OpenMP over all
host cores) on a bounded sample of the same workload — the reference itself is pure Python around filterpy and
cannot be built or installed offline (DESIGN.md "Reference arm").

`--dump-outputs DIR` writes what the last timed step returned as DIR/<name>.npy.  Every input is drawn from fixed seeds,
so two builds run with the same arguments can be compared output for output.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# Algorithmic cost per unit (one object: truth fx + predict + update + epilogue) under SURVEY 8(d)'s counting convention
# (add/mul/cmp = 1, fma = 2, div = sqrt = 10, sin = cos = 40, atan2 = 80, asin = 70, mod = 10).
#   * SURVEY 8(d), the reference's literal sequence — the figure `roofline.frac` uses: fx 1.85 kflop; unit 39 kflop
#     = 14 fx 25.9 k + 2 Cholesky 0.64 k + 2 sigma draws 0.14 k + unscented transform 0.85 k + update 11 k + epilogue 0.1 k.
#     Per kernel: k_predict_tile = 14 fx + 1 sigma draw + UT = 26.8 k; k_update_tile = 1 sigma draw + update + epilogue = 11.2 k;
#     k_factor / k_refactor = 0.32 k each.
#   * the algorithm AS IMPLEMENTED here (secondary key `frac_as_implemented`): streamlined fx 0.86 kflop (6 divisions,
#     6 square roots, 1 atan2, 5.5 sincos), update without the redundant residual evaluations 6.9 kflop, factorisations + UT
#     1.7 kflop => 20.6 kflop.
FLOP_FX_REF = 1.85e3
FLOP_PER_UNIT_REF = 39.0e3
FLOP_PREDICT_TILE_REF = 14 * FLOP_FX_REF + 0.07e3 + 0.85e3
FLOP_UPDATE_TILE_REF = 11.0e3 + 0.07e3 + 0.1e3
FLOP_FX = 0.86e3
FLOP_PER_UNIT = 14 * FLOP_FX + 6.9e3 + 1.7e3
# Algorithmic bytes.  SURVEY 8(d): 920 B per object-step (full 6x6 covariance: read x 48 + P 288 + x_true 48 + z_noise 24,
# write x 48 + P 288 + x_true 48 + obs 96 + 4 error scalars 32).  The packed-covariance layout used here moves 698 B:
# read x 48 + P 168 + xt 48 + z_noise 24 + status 4; write x 48 + P 168 + xt 48 + obs 96 + 5 scalars 40 + status 4 + flags 2.
BYTES_PER_UNIT_REF = 920
BYTES_PER_UNIT = 48 + 168 + 48 + 24 + 4 + 48 + 168 + 48 + 96 + 40 + 4 + 2
BYTES_PREDICT_TILE = (48 + 48 + 168) * 2   # k_predict_tile: reads xt, x, U; writes xt, x, P (packed) = 528 B / object
N_CATALOG = 1_000_000
CEL2TER06AXY = [+0.973104317697536, +0.230363826239128, -0.000703163481769,
                -0.230363800456036, +0.973104570632801, +0.000118545368117,
                +0.000711560162594, +0.000046626402444, +0.999999745754024]


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c4", choices=["c2", "c4", "c3"])
    ap.add_argument("--envs", type=int, default=4096, help="c3: parallel environments per GPU")
    ap.add_argument("--collector", default="greedy", choices=["greedy", "mlp"], help="c3: 'mlp' = stub PPO rollout collector on the device (1 GPU)")
    ap.add_argument("--gather", action="store_true", help="c3, N>1: also all_gather rewards and observations over NCCL every step (a learner on one device)")
    ap.add_argument("--rng", default="device", choices=["device", "host"], help="c3: episodic RNG mode of VecSSATaskerEnv")
    ap.add_argument("--obs-dtype", default="float64", choices=["float64", "float32"],
                    help="c3 (device rng): dtype of the observations handed to the host (float32: SSA_ROLLOUT_OBS_F32, half the D2H bytes)")
    ap.add_argument("--objects", type=int, default=0, help="override the catalog size (c4: whole job, c2: per rank)")
    ap.add_argument("--no-extra", action="store_true", help="skip the short C2 / C3 measurements reported under `extra`")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (float32 / float64; "
                         f"c2 / c4: rank 0's shard, a fixed sample of at most {DUMP_MAX_OBJECTS} objects) to compare builds")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    return a


# --dump-outputs of c2 / c4: rows of a fixed RandomState(0) sample of the shard, in index order (528 B per object)
DUMP_MAX_OBJECTS = 65536


def write_outputs(out_dir, arrays):
    """Save each array as out_dir/<name>.npy; float32 and float64 stay as they are, anything else becomes float64."""
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in arrays.items():
        arr = np.asarray(arr)
        if arr.dtype not in (np.float32, np.float64):
            arr = arr.astype(np.float64)
        np.save(os.path.join(out_dir, name + ".npy"), arr)


def dump_catalog_outputs(out_dir, ukf, gathered):
    """The per-object results of the last timed step of this rank's shard (a sample of DUMP_MAX_OBJECTS objects when the
    shard is larger) and, c4, the reward terms gathered from every rank [world, 5]."""
    from ssa_gym_b200 import _lib as F
    n = ukf.N
    rows = np.arange(n) if n <= DUMP_MAX_OBJECTS else np.sort(np.random.RandomState(0).choice(n, DUMP_MAX_OBJECTS, replace=False))
    fields = {"x_true": F.F_X_TRUE, "x_filter": F.F_X_FILTER, "P_filter": F.F_P_FILTER, "obs": F.F_OBS,
              "delta_pos": F.F_DELTA_POS, "delta_vel": F.F_DELTA_VEL, "sigma_pos": F.F_SIGMA_POS, "sigma_vel": F.F_SIGMA_VEL,
              "trace": F.F_TRACE, "status": F.F_STATUS, "inflations": F.F_INFLATIONS}
    out = {name: ukf.download(f)[rows] for name, f in fields.items()}
    if gathered is not None:
        out["catalog_stats"] = gathered.cpu().numpy().reshape(-1, 5)
    write_outputs(out_dir, out)


def workload_inputs(n_objects, rank, steps, lo=0, hi=None):
    """Synthetic inputs of SURVEY 8(d).  n_objects <= 20000: C2 (the 20 000-orbit catalog, every rank the same
    workload).  Larger: C4, the catalog tiled to n_objects with RandomState(2) jitter; [lo, hi) selects a rank's
    contiguous shard of it (every rank draws the same whole-catalog streams and slices, so the job's inputs do not
    depend on the number of ranks)."""
    from ssa_gym_b200.catalog import synthetic_catalog, tiled_catalog
    from ssa_gym_b200.transformations import arcsec2rad
    hi = n_objects if hi is None else hi
    if n_objects <= 20000:
        cat = synthetic_catalog(n_objects, seed=0)
    else:
        cat = tiled_catalog(n_objects, synthetic_catalog(20000, 0), seed=2)
    x = cat + np.random.RandomState(1000).normal(size=(n_objects, 6)) * np.array([1e5] * 3 + [1e2] * 3)
    P0 = np.diag([1e10] * 3 + [1e4] * 3)
    rs = np.random.RandomState(2000)
    zn = np.empty((steps, hi - lo, 3))
    for s_ in range(steps):  # slice by slice: the whole-catalog slice is only a temporary
        zn[s_] = rs.normal(size=(n_objects, 3))[lo:hi] * np.array([arcsec2rad, arcsec2rad, 1e3])
    return np.ascontiguousarray(cat[lo:hi]), np.ascontiguousarray(x[lo:hi]), P0, zn


class ClockSampler:
    """SM clock and throttle reasons DURING the timed regions.  NVML (nvidia_ml_py) is polled every ~2 ms from a
    thread because the timed region of a C2 run lasts only milliseconds; `nvidia-smi` (the recipe's query) is the
    fallback when NVML cannot be loaded."""

    def __init__(self, index):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self._t = None
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n = self.nvml
        sm = n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(self.h, n.NVML_CLOCK_SM)
        try:
            r = n.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception:
            r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        names = []
        for name, bit in (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("hw_thermal_slowdown", 0x40),
                          ("sw_thermal_slowdown", 0x20), ("hw_power_brake_slowdown", 0x80)):
            if r & bit:
                names.append(name)
        return float(sm), float(mx), names

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._stop.is_set():
            try:
                if self.nvml is not None:
                    self.rows.append(self._sample_nvml())
                    self._stop.wait(0.002)
                    continue
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    c = [v.strip() for v in out.split(",")]
                    names = [nm for nm, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[3:7])
                             if v.lower().startswith("active")]
                    self.rows.append((float(c[0]), float(c[1]), names))
            except Exception:
                pass
            self._stop.wait(0.1)

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=6)
        sm = [r[0] for r in self.rows]
        mx = [r[1] for r in self.rows]
        reasons = sorted({n for r in self.rows for n in r[2]})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def oracle_lib():
    import subprocess as sp
    lib = os.path.join(ROOT, "oracle", "liboracle.so")
    src = os.path.join(ROOT, "oracle", "ukf_oracle.c")
    if not os.path.isfile(lib) or os.path.getmtime(src) > os.path.getmtime(lib):
        sp.run(["make", "-C", os.path.join(ROOT, "oracle"), "-s"], check=True)
    return ctypes.CDLL(lib)


def run_oracle_steps(cfg, cat, x, P0, zn, n_steps, budget_s=None):
    """Time the CPU oracle (all host threads) on the workload.  Returns (units/s, steps run, threads)."""
    L = oracle_lib()
    L.oracle_num_threads.restype = ctypes.c_int
    L.oracle_set_threads(ctypes.c_int(os.cpu_count() or 1))  # torchrun exports OMP_NUM_THREADS=1: use all host threads
    N = len(cat)
    vp = ctypes.c_void_p
    ptr = lambda a: a.ctypes.data_as(vp)
    xt, xf = cat.copy(), x.copy()
    P = np.ascontiguousarray(np.broadcast_to(P0, (N, 6, 6))).copy()
    status, infl = np.zeros(N, np.int32), np.zeros(N, np.int32)
    obs = np.zeros((N, 12))
    sc = [np.zeros(N) for _ in range(5)]
    vis, upd = np.zeros(N, np.uint8), np.zeros(N, np.uint8)
    M = np.array(CEL2TER06AXY)
    flags = 0x1 | 0x2 | 0x4 | 0x10

    def one(s):
        L.oracle_step(ctypes.byref(cfg), ptr(M), ctypes.c_int(flags), ptr(xt), ptr(xf), ptr(P), ptr(status), ptr(infl), None,
                      ptr(zn[s % len(zn)]), ptr(obs), ptr(sc[0]), ptr(sc[1]), ptr(sc[2]), ptr(sc[3]), ptr(sc[4]),
                      None, None, None, None, ptr(vis), ptr(upd))
    one(0)  # warm-up (page-in, thread pool)
    t0 = time.perf_counter()
    done = 0
    for s in range(n_steps):
        one(s + 1)
        done += 1
        if budget_s is not None and time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return N * done / dt, done, L.oracle_num_threads(), dt


def make_cfg(N):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from ssa_gym_b200 import _lib
    from ssa_gym_b200.transformations import arcsec2rad, lla2ecef, trans_uvw_ecef
    from ssa_gym_b200.ukf import Q_discrete_white_noise_block, merwe_weights
    Wm, Wc, lam = merwe_weights()
    c = _lib.SsaUkfCfg()
    c.abi_version, c.n_objects, c.n_envs, c.m = 1, N, 1, N
    c.obs_type, c.resample_after_predict, c.reward_type, c.n_steps = 0, 1, 0, 480
    c.dt, c.lam_plus_n = 20.0, lam
    for i in range(13):
        c.Wm[i], c.Wc[i] = Wm[i], Wc[i]
    for i, v in enumerate(Q_discrete_white_noise_block(20.0, 0.000025 ** 2).ravel()):
        c.Q[i] = v
    for i, v in enumerate(np.diag([arcsec2rad ** 2] * 2 + [1e3 ** 2]).ravel()):
        c.R[i] = v
    lla = np.array([np.radians(38.828198), np.radians(-77.305352), 20.0])
    for i, v in enumerate(lla2ecef(lla)):
        c.obs_itrs[i] = v
    for i, v in enumerate(np.asarray(trans_uvw_ecef(lla[0], lla[1]), dtype=float).ravel()):
        c.T[i] = v
    c.obs_limit = np.radians(-90.0)
    return c


def c3_measure(a, rank, local_rank, world, steps, warmup, gather, dump_dir=None):
    """BASELINE.json config 3: E parallel environments x default RSO count, one vectorised env step per call, actions
    from the device-side greedy tasker, obs [E, m*12] fp64 handed to the host every step (the RLlib rollout shape).
    Metric: env-steps per second through the public API (VecSSATaskerEnv.vector_step), i.e. end to end by
    construction: every step copies the actions host->device and obs / reward / done device->host.  Returns the
    JSON line as a dict (rank 0) or None; dump_dir: rank 0 writes the last timed step's obs / reward / done there."""
    import torch
    import torch.distributed as dist
    from ssa_gym_b200 import env_config, _lib as F
    from ssa_gym_b200.catalog import synthetic_catalog
    from ssa_gym_b200.transformations import gcrs2irts_matrix_approx, time_table
    from ssa_gym_b200.ukf import fp64_peak_tflops
    from ssa_gym_b200.vec_env import VecSSATaskerEnv
    E = a.envs
    cfg = dict(env_config)
    cfg["orbits"] = synthetic_catalog(20000, 0)
    cfg["trans_matrix"] = gcrs2irts_matrix_approx(time_table(cfg["t_0"], cfg["time_step"], cfg["steps"]))
    m = cfg["rso_count"]
    obs_dtype = getattr(a, "obs_dtype", "float64")
    obs_bytes = 4 if obs_dtype == "float32" else 8
    cfg["obs_dtype"] = obs_dtype
    t0 = time.perf_counter()
    env = VecSSATaskerEnv(cfg, E, seeds=[rank * E + e for e in range(E)], device=local_rank, rng=a.rng)
    t_construct = time.perf_counter() - t0
    stream = torch.cuda.current_stream()
    sp = ctypes.c_void_p(stream.cuda_stream)
    multi = world > 1 and gather is not None

    def barrier():
        if multi:
            dist.barrier()
        torch.cuda.synchronize()

    # N > 1: what a learner on one device needs (SURVEY 8e) - per-env rewards and observations of every rank, gathered
    # with one NCCL all_gather each from the episodic mode's device output block, asynchronously every step
    rew_view = env.ukf.torch_view(F.F_ROLLOUT_REWARD) if (multi and a.rng == "device" and gather) else None
    obs_view = env.ukf.torch_view(F.F_ROLLOUT_OBS) if rew_view is not None else None
    g_rew = torch.zeros(world * E, dtype=torch.float64, device="cuda") if rew_view is not None else None
    g_obs = torch.zeros((world * E * m, 12), dtype=torch.float64, device="cuda") if rew_view is not None else None
    works = []
    n_done = 0
    for w in range(max(warmup, 3)):
        _, _, d, _ = env.vector_step(env.greedy_actions())
    peak_tf = fp64_peak_tflops(local_rank, sp)
    sampler = ClockSampler(local_rank)
    launches0 = env.ukf.launch_count
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    tw0 = time.perf_counter()
    r = None
    for s in range(steps):
        obs, r, d, _ = env.vector_step(env.greedy_actions())
        n_done += int(d.sum())
        if rew_view is not None:
            works.append(dist.all_gather_into_tensor(g_rew, rew_view, async_op=True))
            works.append(dist.all_gather_into_tensor(g_obs, obs_view, async_op=True))
    for w_ in works:
        w_.wait()
    e1.record(stream)
    barrier()
    t_wall = time.perf_counter() - tw0
    clocks = sampler.stop()
    if dump_dir and rank == 0:
        write_outputs(dump_dir, {"obs": obs, "reward": r, "done": d})
    ms = e0.elapsed_time(e1)
    launches = env.ukf.launch_count - launches0
    nw = world if multi else 1
    if multi:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    val = E * nw * steps / (ms * 1e-3)
    flop_env_step = m * (14 * FLOP_FX_REF + 1.7e3) + 11.0e3   # m predicts (14 fx + factorisations / UT) + one update, SURVEY 8(d)
    line = None
    if rank == 0:
        line = {"metric": "env-steps per second (vectorised ssa_tasker_simple_2, RL mode)", "value": val, "unit": "env-steps/s",
                "n_gpus": nw, "steps": steps, "warmup": max(warmup, 3), "ms_per_step": ms / steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": f"C3: {E} parallel envs x {m} RSOs per GPU, vector_step + device greedy tasker, {obs_dtype} obs to host",
                           "obs_dtype": obs_dtype, "envs_per_gpu": E, "rso_count": m, "episode_steps": cfg["steps"], "rng": a.rng, "reward_type": cfg["reward_type"],
                           "l2": f"inputs/outputs larger than nothing to flush: every step moves {E * m * 12 * obs_bytes} B of fresh obs over PCIe"},
                "object_predicts_per_s": val * m,
                "e2e": {"value": val, "unit": "env-steps/s", "h2d_bytes_per_step": 4 * E,
                        "d2h_bytes_per_step": E * m * 12 * obs_bytes + E * 8 + E * 16 + E, "ms_per_step": ms / steps,
                        "api": "VecSSATaskerEnv.vector_step (ssa_ukf_rollout_step)" if a.rng == "device" else "VecSSATaskerEnv.vector_step"},
                "roofline": {"bound": "fp64", "kernel": "whole env step", "achieved": val / nw * flop_env_step / 1e12, "peak": peak_tf,
                             "unit": "TFLOP/s", "frac": val / nw * flop_env_step / 1e12 / peak_tf, "traffic": None,
                             "note": "RL-mode step = m predicts + 1 update per env (SURVEY 8d: 287 kflop at m = 10); at E*m = 40960 "
                                     "objects the step is launch/latency and PCIe bound, not FP64 bound"},
                "gpu_launches": int(launches), "clocks": clocks,
                "extra": {"episodes_finished_in_timed_region": n_done, "construct_and_first_reset_s": t_construct,
                          "nccl_gather_per_step": (None if rew_view is None else
                                                   {"reward_bytes_per_rank": 8 * E, "obs_bytes_per_rank": 96 * E * m,
                                                    "gathered_reward_matches_rank0": bool(np.array_equal(g_rew[:E].cpu().numpy(), r))}),
                          "wall_s_timed_region": t_wall}}
    env.close() if hasattr(env, "close") else None
    return line


def c3_collector_measure(a, local_rank, steps, warmup, fragment=32):
    """BASELINE.json config 3 with a PPO-shaped consumer ON THE DEVICE (SURVEY 8d C3: RLlib is absent, so a stub MLP rollout
    collector stands in; rl_agents/RLLib_PPO_training.py:15-48: default fcnet 2 x 256 tanh, rollout_fragment_length = 32).
    Every vector step: the policy reads the observations [E, m*12] where the step left them (float64 -> float32 cast, no
    normalisation, like the reference feeds them), samples one action per environment, writes them into the env's device
    action buffer, the env steps (ONE graph launch, no H2D / D2H, nothing synchronises), reward / done are appended to
    the fragment; every 32 steps the fragment [32, E, ...] is handed over as a sample batch (kept on the device, where a
    learner would consume it)."""
    import torch
    from ssa_gym_b200 import env_config
    from ssa_gym_b200.catalog import synthetic_catalog
    from ssa_gym_b200.transformations import gcrs2irts_matrix_approx, time_table
    from ssa_gym_b200.vec_env import VecSSATaskerEnv
    E = a.envs
    cfg = dict(env_config)
    cfg["orbits"] = synthetic_catalog(20000, 0)
    cfg["trans_matrix"] = gcrs2irts_matrix_approx(time_table(cfg["t_0"], cfg["time_step"], cfg["steps"]))
    m = cfg["rso_count"]
    env = VecSSATaskerEnv(cfg, E, seeds=list(range(E)), device=local_rank, rng="device")
    dev = torch.device("cuda", local_rank)
    torch.manual_seed(0)
    policy = torch.nn.Sequential(torch.nn.Linear(m * 12, 256), torch.nn.Tanh(), torch.nn.Linear(256, 256), torch.nn.Tanh(),
                                 torch.nn.Linear(256, m + 1)).to(dev)   # m action logits + the value head
    v = env.device_views()
    stream = torch.cuda.current_stream()
    sp = ctypes.c_void_p(stream.cuda_stream)
    frag = {"obs": torch.empty((fragment, E, m * 12), dtype=torch.float32, device=dev),
            "actions": torch.empty((fragment, E), dtype=torch.int32, device=dev),
            "logp": torch.empty((fragment, E), dtype=torch.float32, device=dev),
            "vf": torch.empty((fragment, E), dtype=torch.float32, device=dev),
            "rewards": torch.empty((fragment, E), dtype=torch.float32, device=dev),
            "dones": torch.empty((fragment, E), dtype=torch.uint8, device=dev)}
    batches = 0

    def one(t):
        k = t % fragment
        with torch.no_grad():
            obs32 = v["obs"].to(torch.float32)
            out = policy(obs32)
            logp_all = torch.log_softmax(out[:, :m], dim=1)
            act = torch.multinomial(logp_all.exp(), 1).squeeze(1)
            frag["obs"][k].copy_(obs32)
            frag["actions"][k].copy_(act)
            frag["logp"][k].copy_(logp_all.gather(1, act[:, None]).squeeze(1))
            frag["vf"][k].copy_(out[:, m])
            v["actions"].copy_(act)
        env.vector_step_device(stream=sp)
        frag["rewards"][k].copy_(v["reward"])
        frag["dones"][k].copy_(v["done"])

    for w in range(max(warmup, 3)):
        one(w)
    torch.cuda.synchronize()
    l0 = env.ukf.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tw0 = time.perf_counter()
    e0.record(stream)
    sample_batch = None
    for t in range(steps):
        one(t)
        if (t + 1) % fragment == 0:   # hand the fragment over: [32 * E] timesteps, stays on the device
            sample_batch = {k_: x_.reshape((fragment * E,) + tuple(x_.shape[2:])).clone() for k_, x_ in frag.items()}
            batches += 1
    e1.record(stream)
    torch.cuda.synchronize()
    t_wall = time.perf_counter() - tw0
    ms = e0.elapsed_time(e1)
    n_done = int(frag["dones"].sum().item())
    ok = bool(torch.isfinite(frag["rewards"]).all().item()) and (sample_batch is None or sample_batch["obs"].shape == (fragment * E, m * 12))
    out = {"workload": f"C3: {E} envs x {m} RSOs, stub-MLP PPO rollout collector on the device (2 x 256 tanh, fragment {fragment}), "
                       f"device-resident obs / actions (no host copies)",
           "value": E * steps / (ms * 1e-3), "unit": "env-steps/s", "ms_per_step": ms / steps, "steps": steps,
           "object_predicts_per_s": E * m * steps / (ms * 1e-3), "sample_batches": batches, "timesteps_per_batch": fragment * E,
           "gpu_launches": int(env.ukf.launch_count - l0), "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
           "dones_in_last_fragment": n_done, "finite": ok, "wall_s": t_wall,
           "note": "our kernels: one CUDA graph per vector step (gpu_launches counts its kernel nodes); the policy is ~12 small torch "
                   "kernels per step, launched from Python: the loop is host-launch bound"}
    env.close()
    return out


def c2_measure(local_rank, steps, warmup):
    """BASELINE.json config 2 on THIS rank's GPU: the 20 000-orbit catalog, every object predicted and updated once per
    step; per-step CUDA events, L2 flushed between steps.  Returns a small dict."""
    import torch
    from ssa_gym_b200 import _lib as F
    from ssa_gym_b200.ukf import BatchedUKF
    n = 20000
    cat, x, P0, zn = workload_inputs(n, 0, 4)
    cfg = make_cfg(n)
    ukf = BatchedUKF(n_envs=1, m=n, dt=20.0, Q=np.array(cfg.Q).reshape(6, 6), R=np.array(cfg.R).reshape(3, 3),
                     obs_lla=[np.radians(38.828198), np.radians(-77.305352), 20.0], obs_limit_rad=np.radians(-90.0),
                     device=local_rank)
    stream = torch.cuda.current_stream()
    sp = ctypes.c_void_p(stream.cuda_stream)
    ukf.reset(cat, x, P0, stream=sp)
    M = np.array(CEL2TER06AXY)
    flags = F.STEP_TRUTH | F.STEP_PREDICT | F.STEP_UPDATE_ALL | F.STEP_EPILOGUE
    zn_dev = torch.from_numpy(zn).cuda()
    zview = ukf.torch_view(F.F_Z_NOISE)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    for w in range(max(warmup, 3)):
        zview.copy_(zn_dev[w % 4], non_blocking=True)
        ukf.step(M, flags, stream=sp)
    torch.cuda.synchronize()
    l0 = ukf.launch_count
    evs = []
    for s in range(steps):
        zview.copy_(zn_dev[s % 4], non_blocking=True)
        flush.fill_(s & 0xFF)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        ukf.step(M, flags, stream=sp)
        e1.record(stream)
        evs.append((e0, e1))
    torch.cuda.synchronize()
    ms = float(np.mean([e0.elapsed_time(e1) for e0, e1 in evs]))
    out = {"workload": "C2: 20000-orbit catalog on one GPU, UKF predict+update of every object per step",
           "value": n / (ms * 1e-3), "unit": "object-updates/s", "ms_per_step": ms, "steps": steps,
           "gpu_launches": int(ukf.launch_count - l0), "failed_filters": int((ukf.download(F.F_STATUS) & 1).sum()),
           "l2": "flushed between timed steps (256 MiB write)"}
    ukf.close()
    del flush
    return out


def python_reference_style_baseline(seconds):
    """BASELINE.md §3 items 1-2: the reference's own execution style — one filterpy-shaped UKF object per RSO driven by
    Python loops (numpy restatement of filterpy, oracle/filterpy_restated.py; fx / hx evaluated per call through the C
    oracle, as the reference calls its numba functions), first in ONE process (how the reference runs an env), then one
    worker process per host core (its only parallelism: one env per Ray worker, rl_agents/RLLib_PPO_training.py:17)."""
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    one = _python_style_worker((0, seconds / 2))
    with mp.get_context("fork").Pool(cores) as pool:
        res = pool.map(_python_style_worker, [(i + 1, seconds / 2) for i in range(cores)])
    return {"single_process": {"value": one[0] / one[1], "unit": "object-updates/s", "cores": 1, "object_updates": one[0], "seconds": one[1]},
            "one_env_per_core": {"value": float(sum(r[0] / r[1] for r in res)), "unit": "object-updates/s", "cores": cores,
                                 "object_updates": int(sum(r[0] for r in res))},
            "kind": "port", "what": "numpy restatement of filterpy's UnscentedKalmanFilter (predict + update per object in a "
                                    "Python loop, m = 10 objects per env, default env_config), fx / hx per call through oracle/liboracle.so"}


def _python_style_worker(arg):
    seed, seconds = arg
    os.environ["OMP_NUM_THREADS"] = "1"
    from oracle import dynamics_restated as D
    from oracle.env_oracle import OracleEnv
    from ssa_gym_b200 import env_config
    from ssa_gym_b200.catalog import synthetic_catalog
    from ssa_gym_b200.transformations import gcrs2irts_matrix_approx, time_table
    oracle_lib()
    cfg = dict(env_config)
    cfg["orbits"] = synthetic_catalog(2000, 0)
    cfg["reward_type"] = "trinary"   # 'jones' ends an episode within a handful of steps; the filter work per step is the same
    tm = gcrs2irts_matrix_approx(time_table(cfg["t_0"], cfg["time_step"], cfg["steps"]))
    env = OracleEnv(cfg, D.oracle_fx_callable(), tm)
    env.seed(seed)
    env.reset()
    t0 = time.perf_counter()
    n = 0
    k = 0
    while time.perf_counter() - t0 < seconds:
        _, _, done, _ = env.step(k % env.m)
        k += 1
        n += env.m   # m predicts (+ one update) per env step, counted as m object-updates: generous to this baseline
        if done:
            env.reset()
    return n, time.perf_counter() - t0


def main():
    a = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if a.gpus != world:
        if world == 1 and a.gpus > 1:
            raise SystemExit(f"bench.py --gpus {a.gpus}: launch one rank per GPU, e.g. python -m torch.distributed.run --nnodes=1 "
                             f"--nproc-per-node {a.gpus} --master-addr 127.0.0.1 bench.py --gpus {a.gpus} ...")
        raise SystemExit(f"bench.py: --gpus {a.gpus} does not match WORLD_SIZE {world}")

    if a.impl == "reference":
        return run_reference_arm(a, rank, world)

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the UKF hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        if a.workload == "c3":
            line = c3_measure(a, rank, local_rank, world, a.steps, a.warmup, a.gather, a.dump_outputs)
            if rank == 0:
                if a.collector == "mlp":
                    line["extra"]["ppo_collector_on_device"] = c3_collector_measure(a, local_rank, a.steps, a.warmup)
                print(json.dumps(line))
        else:
            run_catalog(a, rank, local_rank, world)
    finally:
        if world > 1:
            dist.destroy_process_group()
    return 0


def catalog_layout(a, world, rank):
    """(total objects of the job, this rank's [lo, hi), workload name, scaling)"""
    from ssa_gym_b200.dist import shard_bounds
    if a.workload == "c2":
        n = a.objects or 20000
        return n * world, 0, n, f"C2: {n}-orbit catalog per GPU, UKF predict+update of every object per step", "weak"
    total = a.objects or N_CATALOG
    lo, hi = shard_bounds(total, world, rank)
    name = (f"C4: {total}-object synthetic catalog sharded over {world} GPU(s) in contiguous blocks, per-step UKF predict+update of "
            f"every object + shard reward terms (ssa_ukf_catalog_stats) + NCCL all_gather of them, all inside the timed events")
    return total, lo, hi, name, "strong"


def run_reference_arm(a, rank, world):
    """The reference's CPU implementation of the path on the box's host cores: the oracle port (the reference is pure
    Python around filterpy and cannot be installed offline), all host threads, a bounded sample of the arm's workload."""
    if rank != 0:
        return 0
    total, _, _, name, scaling = catalog_layout(a, world, 0)
    n_s = min(total, 200_000)   # bounded sample: the first 200 000 objects of the catalog (a step of the whole 1M takes ~0.5 s)
    cat, x, P0, zn = workload_inputs(total, 0, 4, 0, n_s)
    cfg = make_cfg(n_s)
    for w in range(max(a.warmup, 1)):   # warm-up passes: page-in, OpenMP thread pool, clocks
        run_oracle_steps(cfg, cat, x, P0, zn, 1)
    val, done, threads, dt = run_oracle_steps(cfg, cat, x, P0, zn, a.steps, budget_s=120.0)
    line = {"impl": "reference", "metric": "RSO UKF predict+update per second", "value": val, "unit": "object-updates/s",
            "n_gpus": a.gpus, "steps": done, "warmup": max(a.warmup, 1), "ms_per_step": dt / done * 1e3 * (total / n_s),
            "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": name, "objects_total": total, "dt_s": 20.0, "obs_type": "aer",
                       "sigma_points": "merwe alpha=1e-4 beta=2 kappa=-3", "trans_matrix": "SOFA Cel2Ter06aXY (tests.py:107-109)"},
            "cpu_baseline": {"value": val, "unit": "object-updates/s", "cores": threads, "kind": "port",
                             "sample": f"{done} steps x the first {n_s} objects of the {total}-object catalog, oracle/ukf_oracle.c "
                                       f"(reference operation order, libm), OpenMP over {threads} host threads; ms_per_step is scaled to the whole catalog"},
            "e2e": {"value": val, "unit": "object-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


def run_catalog(a, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    from ssa_gym_b200 import _lib
    from ssa_gym_b200.ukf import BatchedUKF, fp64_peak_tflops
    F = _lib
    total, lo, hi, wl_name, scaling = catalog_layout(a, world, rank)
    n_obj = hi - lo
    c4 = a.workload == "c4"
    config = {"workload": wl_name, "objects_total": total, "objects_per_gpu": n_obj, "dt_s": 20.0, "obs_type": "aer",
              "sigma_points": "merwe alpha=1e-4 beta=2 kappa=-3", "trans_matrix": "SOFA Cel2Ter06aXY (tests.py:107-109)",
              "l2": "flushed between timed steps (256 MiB write)"}
    if c4:
        cat, x, P0, zn = workload_inputs(total, rank, 8, lo, hi)
    else:
        cat, x, P0, zn = workload_inputs(n_obj, rank, 8)
    cfg = make_cfg(n_obj)
    ukf = BatchedUKF(n_envs=1, m=n_obj, dt=20.0, Q=np.array(cfg.Q).reshape(6, 6), R=np.array(cfg.R).reshape(3, 3),
                     obs_lla=[np.radians(38.828198), np.radians(-77.305352), 20.0], obs_limit_rad=np.radians(-90.0),
                     device=local_rank)
    stream = torch.cuda.current_stream()
    sp = ctypes.c_void_p(stream.cuda_stream)
    ukf.reset(cat, x, P0, stream=sp)
    M = np.array(CEL2TER06AXY)
    flags = F.STEP_TRUTH | F.STEP_PREDICT | F.STEP_UPDATE_ALL | F.STEP_EPILOGUE
    # device-resident measurement noise for `value` (inputs already in HBM): 8 pre-drawn slices, rotated
    zn_dev = torch.from_numpy(zn).cuda()
    zview = ukf.torch_view(F.F_Z_NOISE)  # zero-copy torch view of the handle's z_noise buffer [N,3]
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")

    def load_noise(s):
        # device-to-device copy of slice s into the handle's z_noise buffer (outside the timed events)
        zview.copy_(zn_dev[s % 8], non_blocking=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # C4 (BASELINE.json config 4: "per-step UKF + reward, NCCL gather of rewards"): every step reduces the shard's reward
    # terms on the device (ssa_ukf_catalog_stats: 2 small kernels) and all-gathers the 5 doubles per rank over NCCL.
    # The collective is enqueued stream-ordered (async_op=False makes the launching stream wait for it), so the step's
    # closing event is recorded after the gather has completed: the gather is inside every step's timed interval.
    gathered = torch.zeros(world * 5, dtype=torch.float64, device="cuda") if c4 else None
    stats_view = None
    if c4:
        ukf.catalog_stats(index_offset=lo, stream=sp)
        stats_view = ukf.torch_view(F.F_CATALOG_STATS)

    step_flags = flags | (F.STEP_CATALOG_STATS if c4 else 0)   # C4: the reward reduction rides in the step's own graph

    def reward_gather():
        if world > 1:
            dist.all_gather_into_tensor(gathered, stats_view)
        else:
            gathered.copy_(stats_view, non_blocking=True)

    # ---- warm-up -----------------------------------------------------------------------------------
    for w in range(max(a.warmup, 3)):
        load_noise(w)
        ukf.step(M, step_flags, stream=sp)
        if c4:
            reward_gather()
    torch.cuda.synchronize()
    peak_tf = fp64_peak_tflops(local_rank, sp)

    # ---- timed: exactly K steps, per-step CUDA events on the launching stream, L2 flushed between steps ---
    sampler = ClockSampler(local_rank)
    launches0 = ukf.launch_count
    barrier()
    sampler.start()
    evs = []
    t_wall0 = time.perf_counter()
    for s in range(a.steps):
        load_noise(s)
        flush.fill_(s & 0xFF)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        ukf.step(M, step_flags, stream=sp)
        if c4:
            reward_gather()
        e1.record(stream)
        evs.append((e0, e1))
    barrier()
    t_wall = time.perf_counter() - t_wall0
    if a.dump_outputs and rank == 0:   # before the profiling and e2e passes below advance the state further
        dump_catalog_outputs(a.dump_outputs, ukf, gathered)
    step_ms = [e0.elapsed_time(e1) for e0, e1 in evs]
    total_ms = float(np.sum(step_ms))
    launches = ukf.launch_count - launches0
    status = ukf.download(F.F_STATUS)
    n_failed = int((status & 1).sum())
    c4_check = None
    if c4:  # the gathered shard terms of the LAST timed step against a host recomputation of this rank's shard
        g = gathered.cpu().numpy().reshape(world, 5)
        dpos_h, tr_h = ukf.download(F.F_DELTA_POS), ukf.download(F.F_TRACE)
        mine = g[rank]
        assert mine[0] == dpos_h.max() and mine[2] == n_obj and mine[3] == tr_h.max() and mine[4] == lo + int(np.argmax(tr_h))
        assert mine[1] == float(((dpos_h < 1e4).astype(int) + (dpos_h < 1e7).astype(int)).sum())
        assert g[:, 2].sum() == total
        best = int(np.argmax(g[:, 3]))
        c4_check = {"max_delta_pos_m": float(g[:, 0].max()), "trinary_reward": float(g[:, 1].sum() / g[:, 2].sum() / 2),
                    "argmax_trace_object": int(g[best, 4]), "gathered_ranks": int(world), "objects_gathered": int(g[:, 2].sum()),
                    "bytes_per_rank_per_step": 40, "in_timed_events": True,
                    "checked": "every rank's gathered row of the last step == host recomputation from its downloaded shard"}

    # per-kernel durations of the step (CUDA events between the launches, L2 flushed before each step)
    kms = []
    for s in range(min(a.steps, 20)):
        load_noise(s)
        flush.fill_(s & 0xFF)
        torch.cuda.synchronize()
        kms.append(ukf.step_profile(M, flags, stream=sp))
    kms = np.mean(np.array(kms), axis=0)

    # back-to-back (no flush) for reference
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for s in range(a.steps):
        ukf.step(M, step_flags, stream=sp)
        if c4:
            reward_gather()
    e1.record(stream)
    barrier()
    b2b_ms = e0.elapsed_time(e1) / a.steps

    # ---- e2e: the user-facing call with HOST buffers (ssa_ukf_step_pinned: double-buffered pinned blocks, the copies
    # overlap the neighbouring steps' kernels).  Every step: ONE H2D copy of that step's inputs (z_noise + trans_matrix)
    # from the handle's pinned input block, the kernel chain (one captured graph launch) and a D2H read of the step's
    # result.  C4's result is what BASELINE.json config 4 names — the per-step reward terms, reduced per shard on the
    # device, all-gathered over NCCL and read back to pinned host memory (40 B per rank); the filter state and the
    # observations stay device-resident for a device-side consumer.  `e2e.full_outputs` is the same loop with the whole
    # per-object output block (obs 96 B + delta_pos 8 B + status 4 B per object) copied to the host every step as well
    # (C2's e2e, and round 1's definition): that one is bound by PCIe / host memory, not by the GPUs.
    io = ukf.host_io()
    for b_ in range(2):
        io[b_]["z_noise"][:] = zn[b_]
        io[b_]["M"][:] = M.reshape(9)
    # The step's result is read back OFF the compute stream: with SSA_STEP_CATALOG_STATS a pinned step reduces the shard's
    # reward terms into the device slot of its parity and the library's download stream copies them to pinned host memory
    # (N = 1: that is the read-back).  N > 1: a side stream all-gathers the slot over NCCL and copies the gathered rows
    # to pinned host memory; the compute stream only waits — two steps later, before the slot is rewritten — for that
    # gather to have finished.  (Measured, tools/e2e_probe.py: the same copies issued on the compute stream cost 40 us
    # per step of serialisation between consecutive graph launches — 0.244 vs 0.204 ms per step at 125 000 objects.)
    side = torch.cuda.Stream()
    stats_host = [ukf.host_stats(b_)[0] for b_ in range(2)] if c4 else None
    stats_dev = [ukf.host_stats_torch(b_) for b_ in range(2)] if c4 else None
    gathered2 = [torch.zeros(world * 5, dtype=torch.float64, device="cuda") for _ in range(2)] if c4 else None
    gathered_host2 = [torch.zeros(world * 5, dtype=torch.float64).pin_memory() for _ in range(2)] if c4 else None

    host_issue = {}
    last_parity = {}

    def e2e_loop(extra_flags, read_reward, tag):
        for w in range(4):
            ukf.step_pinned(step_flags | extra_flags, stream=sp)
        ukf.host_join(stream=sp)
        barrier()
        side_done = [None, None]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = ukf.launch_count
        e0.record(stream)
        th0 = time.perf_counter()
        for s in range(a.steps):
            b_ = ukf.next_parity
            io[b_]["M"][:] = M.reshape(9)  # this step's trans_matrix[i] (72 B) travels with the noise
            if side_done[b_] is not None:
                stream.wait_event(side_done[b_])   # the gather of two steps ago has read this parity's slot
            ukf.step_pinned(step_flags | extra_flags, stream=sp)
            if c4 and read_reward and world > 1:
                ev = torch.cuda.Event()
                ev.record(stream)
                with torch.cuda.stream(side):
                    side.wait_event(ev)
                    dist.all_gather_into_tensor(gathered2[b_], stats_dev[b_])
                    gathered_host2[b_].copy_(gathered2[b_], non_blocking=True)
                    side_done[b_] = torch.cuda.Event()
                    side_done[b_].record(side)
            last_parity[tag] = b_
        host_issue[tag] = (time.perf_counter() - th0) / a.steps * 1e3   # host time to ISSUE one step (Python + driver + NCCL enqueue)
        ukf.host_join(stream=sp)
        stream.wait_stream(side)
        e1.record(stream)
        barrier()
        return e0.elapsed_time(e1) / a.steps, ukf.launch_count - l0

    full_ms, full_launches = e2e_loop(0, False, "full")   # (the reward terms follow from the downloaded outputs)
    h2d = io[0]["z_noise"].nbytes + 80 + 8  # z_noise, trans_matrix (+1 pad double), the env's action word
    d2h_full = io[0]["obs"].nbytes + (ukf.ld + ukf.ld // 2) * 8
    if c4:
        e2e_ms, e2e_launches = e2e_loop(F.STEP_NO_D2H, True, "reward")
        d2h = 40 * world
        lp = last_parity["reward"]
        g2 = (gathered_host2[lp].numpy() if world > 1 else np.array(stats_host[lp])).reshape(world, 5)
        assert g2[:, 2].sum() == total and np.isfinite(g2).all()
        assert g2[rank if world > 1 else 0, 2] == n_obj
    else:
        e2e_ms, e2e_launches, d2h = full_ms, full_launches, d2h_full
    obs_np = io[0]["obs"]
    clocks = sampler.stop()  # sampled over the timed regions (value and e2e)
    assert np.isfinite(obs_np).all()

    # ---- reduce over ranks (max time) --------------------------------------------------------------
    t = torch.tensor([total_ms, b2b_ms, e2e_ms, full_ms] + [float(v) for v in kms], dtype=torch.float64, device="cuda")
    per_rank = [total_ms / a.steps]
    if world > 1:
        allr = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allr, t)
        per_rank = [float(r_[0]) / a.steps for r_ in allr]
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    tl = [float(v) for v in t.tolist()]
    total_ms, b2b_ms, e2e_ms, full_ms = tl[:4]
    kms = np.array(tl[4:])
    ms_per_step = total_ms / a.steps
    units = total
    value = units / (ms_per_step * 1e-3)
    e2e_val = units / (e2e_ms * 1e-3)

    # ---- short C2 / C3 sub-measurements on rank 0 (the other ranks wait) ---------------------------------------
    extra_c2 = extra_c3 = None
    tile = os.environ.get("SSA_UKF_KERNEL", "tile") not in ("split", "team")
    if rank == 0 and not a.no_extra and world == 1:   # (N > 1: the other ranks would idle; the N = 1 line carries them)
        try:
            if a.workload != "c2":
                extra_c2 = c2_measure(local_rank, 50, 5)
            import copy
            a3 = copy.copy(a)
            l3 = c3_measure(a3, 0, local_rank, 1, 30, 5, None)
            extra_c3 = {k: l3[k] for k in ("value", "unit", "ms_per_step", "steps", "gpu_launches", "object_predicts_per_s")}
            extra_c3["workload"] = l3["config"]["workload"]
            extra_c3["e2e_bytes_per_step"] = {"h2d": l3["e2e"]["h2d_bytes_per_step"], "d2h": l3["e2e"]["d2h_bytes_per_step"]}
            if a3.rng == "device":  # the same loop with float32 observations (what an RLlib preprocessor makes of them anyway)
                a32 = copy.copy(a3)
                a32.obs_dtype = "float32"
                l32 = c3_measure(a32, 0, local_rank, 1, 30, 5, None)
                extra_c3["obs_float32"] = {"value": l32["value"], "unit": l32["unit"], "ms_per_step": l32["ms_per_step"],
                                           "d2h_bytes_per_step": l32["e2e"]["d2h_bytes_per_step"]}
            extra_c3["ppo_collector_on_device"] = c3_collector_measure(a3, local_rank, 128, 10)
        except Exception as ex:  # the headline must not be lost to a failure of an extra
            extra_c3 = {"error": repr(ex)}
    barrier()

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        kern_ms = float(np.mean(step_ms))
        team = os.environ.get("SSA_UKF_KERNEL") == "team"
        # dominant kernel: k_predict_tile (14 two-body propagations + unscented transform per object); split pipeline: k_fx
        dom_ms = float(kms[0] if team else kms[1])
        dom_name = "ssa_step_kernel" if team else ("k_predict_tile" if tile else "k_fx")
        dom_flop_ref = (FLOP_PER_UNIT_REF if team else (FLOP_PREDICT_TILE_REF if tile else 14 * FLOP_FX_REF)) * n_obj
        dom_flop_impl = (FLOP_PER_UNIT if team else (14 * FLOP_FX + (0.9e3 if tile else 0.0))) * n_obj
        dom_tf = dom_flop_ref / (dom_ms * 1e-3) / 1e12
        # DRAM bytes per launch from the committed `ncu --set full` capture of this kernel at this shard size
        traffic = traffic_step = hw = None
        try:
            cap = json.load(open(os.path.join(ROOT, "profiles", "r04_ncu_kernels.json")))
            ent = cap.get(str(n_obj))
            if ent and tile and not team:
                traffic = ent["k_predict_tile"]["dram_bytes_per_launch"]
                traffic_step = sum(v["dram_bytes_per_launch"] for v in ent.values() if isinstance(v, dict) and "dram_bytes_per_launch" in v)
                # FP64 arithmetic counted by the hardware in that capture (DADD + DMUL + 2 DFMA thread instructions per launch),
                # over THIS run's CUDA-event durations
                kf = ent["k_predict_tile"].get("fp64_flop_per_launch_hw")
                sf = sum(v.get("fp64_flop_per_launch_hw", 0.0) for v in ent.values() if isinstance(v, dict))
                if kf:
                    hw = {"flop_per_launch": kf, "achieved": kf / (dom_ms * 1e-3) / 1e12, "unit": "TFLOP/s",
                          "frac": kf / (dom_ms * 1e-3) / 1e12 / peak_tf,
                          "fp64_pipe_pct_ncu": ent["k_predict_tile"].get("fp64_pipe_pct"),
                          "whole_step": {"flop_per_object": sf / n_obj, "achieved": sf / (kern_ms * 1e-3) / 1e12,
                                         "frac": sf / (kern_ms * 1e-3) / 1e12 / peak_tf},
                          "what": "sm__sass_thread_inst_executed_op_{dadd,dmul,dfma}_pred_on of the committed ncu capture "
                                  "(profiles/r04_ncu_kernels.json): flops the threads actually executed, divisions / square roots / "
                                  "transcendentals expanded into their FMA sequences; the FP64 pipe is busier than this fraction "
                                  "because DADD / DMUL / DSETP occupy it like an FMA"}
        except Exception:
            pass
        # SURVEY 8(d)'s counts are estimates; the measured ones (tools/opcount.py: the reference's literal sequence run through
        # an operation-counting build of the oracle, priced with the same convention) are reported beside the fractions they give
        ref_counted = None
        try:
            oc = json.load(open(os.path.join(ROOT, "profiles", "opcount_reference_sequence.json")))
            fu = oc["unit (truth + predict + update + epilogue)"]["flop_survey_convention"]
            fp = oc["truth + predict"]["flop_survey_convention"]
            ref_counted = {"flop_per_object": fu, "flop_per_object_predict_and_truth": fp,
                           "flop_per_propagation": oc["fx (one propagation, dt = 20 s)"]["flop_survey_convention"],
                           "flop_per_object_every_operation_1": oc["unit (truth + predict + update + epilogue)"]["flop_every_op_1"],
                           "whole_step_frac": fu * n_obj / (kern_ms * 1e-3) / 1e12 / peak_tf,
                           "what": "operation count of the reference's literal sequence, MEASURED (profiles/opcount_reference_sequence.json) "
                                   "instead of SURVEY 8(d)'s estimate of 39 kflop / 27.5 kflop / 1.85 kflop, same pricing convention; the "
                                   "fraction it gives exceeds the executed-arithmetic fractions (hw_counted, frac_as_implemented) because "
                                   "the implementation does not execute most of the reference's divisions and transcendentals"}
        except Exception:
            pass
        impl_counted = None
        try:
            oi = json.load(open(os.path.join(ROOT, "profiles", "opcount_implemented.json")))
            fi = oi["unit (truth + predict + update + epilogue)"]["flop_survey_convention"]
            impl_counted = {"flop_per_object": fi, "flop_per_object_add_mul_2fma": oi["unit (truth + predict + update + epilogue)"]["flop_add_mul_2fma_only"],
                            "flop_per_propagation": oi["fx (one propagation, dt = 20 s)"]["flop_survey_convention"],
                            "whole_step_frac": fi * n_obj / (kern_ms * 1e-3) / 1e12 / peak_tf,
                            "what": "primitive operations the IMPLEMENTED algorithm executes per object, MEASURED with an operation-counting "
                                    "build of the host twin (profiles/opcount_implemented.json; add = mul = compare = 1, fma = 2, div = sqrt = "
                                    "10; the elementary functions are FMA polynomials and are counted through their primitives) - agrees with "
                                    "the hardware count hw_counted.whole_step.flop_per_object"}
        except Exception:
            pass
        step_tf = FLOP_PER_UNIT_REF * n_obj / (kern_ms * 1e-3) / 1e12
        step_gb = BYTES_PER_UNIT_REF * n_obj / (kern_ms * 1e-3) / 1e9
        line = {
            "metric": "RSO UKF predict+update per second", "value": value, "unit": "object-updates/s",
            "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config,
            "roofline": {"bound": "fp64", "kernel": dom_name, "achieved": dom_tf, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": dom_tf / peak_tf, "traffic": traffic,
                         "algorithmic_flop_per_launch": dom_flop_ref, "algorithmic_bytes_per_launch": BYTES_PREDICT_TILE * n_obj if tile else None,
                         "kernel_ms": dom_ms, "kernel_share_of_step": dom_ms / float(np.sum(kms)),
                         "frac_as_implemented": dom_flop_impl / (dom_ms * 1e-3) / 1e12 / peak_tf,
                         "hw_counted": hw,
                         "reference_sequence_measured": ref_counted,
                         "implemented_measured": impl_counted,
                         "step_kernels_ms": ({"k_factor": float(kms[0]), "k_predict_tile": float(kms[1]), "k_refactor": float(kms[2]),
                                              "k_update_tile": float(kms[4])} if tile and not team else
                                             {"factor": float(kms[0]), "fx": float(kms[1]), "ut": float(kms[2]), "hx": float(kms[3]),
                                              "update": float(kms[4])}),
                         "whole_step": {"achieved": step_tf, "frac": step_tf / peak_tf, "flop_per_object": FLOP_PER_UNIT_REF,
                                        "frac_as_implemented": step_tf * FLOP_PER_UNIT / FLOP_PER_UNIT_REF / peak_tf,
                                        "algorithmic_bytes": BYTES_PER_UNIT_REF * n_obj, "traffic": traffic_step,
                                        "hbm": {"achieved": step_gb, "peak": hbm_peak, "unit": "GB/s", "frac": step_gb / hbm_peak,
                                                "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback 6650"}},
                         "note": "SURVEY 8(d) counting (div = sqrt = 10, sin = cos = 40, atan2 = 80 flop ...): dominant kernel "
                                 "k_predict_tile = 14 fx x 1.85 kflop + sigma draw + unscented transform = 26.8 kflop per object per launch, "
                                 "divided by the mean CUDA-event duration of that kernel in this run (per rank: its shard); whole_step = "
                                 "39 kflop and 920 B per object over the mean step; frac_as_implemented prices the streamlined arithmetic "
                                 "actually executed (20.6 kflop per object); peak = DFMA microbenchmark measured live in this run "
                                 "(ssa_ukf_fp64_peak; FP64 is not in MEASURED_PEAKS.json); traffic = DRAM bytes of the kernel / of the "
                                 "step's kernels from the committed ncu capture (profiles/r04_ncu_kernels.json) when one exists for this shard size"},
            "e2e": {"value": e2e_val, "unit": "object-updates/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms, "gpu_launches": int(e2e_launches), "bytes_are": "per rank",
                    "api": "BatchedUKF.step_pinned (ssa_ukf_step_pinned): pinned host input block, 1 H2D + 1 graph launch per step"
                           + (" (shard reward terms reduced in the same graph) + their D2H read on the download stream"
                              + (" after an NCCL all_gather on a side stream" if world > 1 else "") if c4 else
                              " + 1 D2H of obs / delta_pos / status"),
                    "result_read_back": ("the step's reward terms (max delta_pos, trinary reward, arg-max trace: 5 doubles per shard) of "
                                         "every rank, after the NCCL all_gather; state and observations stay device-resident" if c4
                                         else "obs [N,12], delta_pos [N], status [N]"),
                    "full_outputs": {"value": units / (full_ms * 1e-3), "ms_per_step": full_ms, "d2h_bytes_per_step": d2h_full,
                                     "gpu_launches": int(full_launches),
                                     "what": "same loop, the whole per-object output block (obs, delta_pos, status: 108 B per object) "
                                             "also copied to pinned host memory every step",
                                     "limiter": f"PCIe / host memory: {(h2d + d2h_full) * world / 1e6:.1f} MB per step between the GPUs and one "
                                                f"host ({(h2d + d2h_full) * world / (full_ms * 1e-3) / 1e9:.1f} GB/s aggregate); the kernels "
                                                f"alone need {ms_per_step:.3f} ms"},
                    "host_issue_ms_per_step": host_issue.get("reward", host_issue.get("full")),
                    "limiter": (f"the kernels need {ms_per_step:.3f} ms per step, the host needs {host_issue.get('reward', host_issue.get('full')):.3f} ms to "
                                f"issue one (Python + 1 H2D + 1 graph launch" + (" + NCCL all_gather and D2H enqueued on a side stream" if world > 1 else "") + "; the reward read-back is off the compute stream); H2D of the measurements "
                                f"({h2d * world / 1e6:.1f} MB per step, {h2d * world / (e2e_ms * 1e-3) / 1e9:.1f} GB/s aggregate) overlaps the kernels"),
                    "l2": "not flushed: the filter state is device-resident between steps by design; every step's inputs arrive "
                          "from pinned host memory and its result leaves to pinned host memory inside the timed region"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "extra": {"ms_per_step_back_to_back_no_flush": b2b_ms, "wall_s_timed_region": t_wall, "failed_filters": n_failed,
                      "ms_per_step_of_each_rank": per_rank, "c4_reward_gather": c4_check,
                      "step_ms_min": float(np.min(step_ms)), "step_ms_max": float(np.max(step_ms)),
                      "c2": extra_c2, "c3": extra_c3},
        }
        if not a.no_cpu_baseline and world == 1:   # the CPU baseline is timed on rank 0 at N = 1 only
            n_s = min(n_obj, 200_000)
            if c4:
                catc, xc, P0c, znc = workload_inputs(total, 0, 4, 0, n_s)
            else:
                catc, xc, P0c, znc = workload_inputs(n_s, 0, 4)
            val, done, threads, dtc = run_oracle_steps(make_cfg(n_s), catc, xc, P0c, znc, 10 ** 6, budget_s=a.cpu_seconds)
            line["cpu_baseline"] = {"value": val, "unit": "object-updates/s", "cores": threads, "kind": "port",
                                    "sample": f"{done} steps x the first {n_s} objects of the catalog in {dtc:.1f} s, oracle/ukf_oracle.c "
                                              f"(reference operation order, libm), OpenMP over host threads"}
            try:
                line["cpu_baseline"]["reference_style_python"] = python_reference_style_baseline(a.cpu_seconds)
            except Exception as ex:
                line["cpu_baseline"]["reference_style_python"] = {"error": repr(ex)}
        print(json.dumps(line))
    ukf.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
