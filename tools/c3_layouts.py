#!/usr/bin/env python
"""C3 (VecSSATaskerEnv, rng='device') step time per observation layout and reward type.

Variants, each one VecSSATaskerEnv in one process, measured in alternation and repeated (--reps):
  flatten/jones      today's default layout (regression guard)
  aer/jones (new)    'aer' rows computed in the step graph (SSA_ROLLOUT_OBS_AER), 32 B per object cross PCIe
  aer/trinary (new)
  aer/jones (old)    a flatten env plus the host formatting the device path replaces: one hx_aer_erfa call
                     (ssa_unit_hx_aer: 2 cudaMalloc, H2D, kernel, D2H, 2 cudaFree) per distinct step index
  flatten/shaped     the 'shaped' reward with its history on the device
Actions come from the device visible-greedy tasker (as bench.py's C3 workload).  Reported per variant: ms per step
(CUDA events around a run of --steps vector_step calls, each ending in a synchronise; every repetition), D2H bytes
per step computed from the shapes, graph kernels per step (launch_count), and distinct step indices per step.
  python tools/c3_layouts.py [--envs 4096] [--steps 200] [--warmup 300] [--reps 3] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

VARIANTS = [("flatten", "jones", "new"), ("aer", "jones", "new"), ("aer", "trinary", "new"), ("aer", "jones", "old"),
            ("flatten", "shaped", "new")]


def old_aer(vec, obs12):
    """vec_env._format_obs of 'aer' as the device mode ran it before the layout moved into the step graph."""
    from ssa_gym_b200 import dynamics
    o = np.asarray(obs12).reshape(-1, vec.m, 12)
    steps = np.minimum(vec.i, len(vec.trans_matrix) - 1)
    out = np.empty((len(o), vec.m, 4))
    for i in np.unique(steps):
        sel = np.where(steps == i)[0]
        out[sel, :, :3] = dynamics.hx_aer_erfa(o[sel, :, :6], vec.trans_matrix[i], vec.obs_lla, vec.obs_itrs, device=vec._device)
    d = o[:, :, 6:]
    out[:, :, 3] = ((((d[:, :, 0] + d[:, :, 1]) + d[:, :, 2]) + d[:, :, 3]) + d[:, :, 4]) + d[:, :, 5]
    return np.nan_to_num(out.reshape(len(o), vec.m * 4), copy=False, nan=0.001, posinf=0.001, neginf=0.001)


def gpu_info():
    import torch
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": "not available"}
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30)
        if r.returncode == 0 and r.stdout.strip():
            info["power_limit_w"] = float(r.stdout.strip().splitlines()[0])
    except (OSError, ValueError, subprocess.TimeoutExpired):
        pass
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=300)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from ssa_gym_b200 import env_config, _lib as F
    from ssa_gym_b200.catalog import synthetic_catalog
    from ssa_gym_b200.transformations import gcrs2irts_matrix_approx, time_table
    from ssa_gym_b200.vec_env import VecSSATaskerEnv
    if not torch.cuda.is_available():
        raise SystemExit("c3_layouts measures on the GPU: no CUDA device visible")
    E = a.envs
    base = dict(env_config)
    base["orbits"] = synthetic_catalog(20000, 0)
    base["trans_matrix"] = gcrs2irts_matrix_approx(time_table(base["t_0"], base["time_step"], base["steps"]))
    m = base["rso_count"]
    N = E * m
    tail = 8 * E + 4 * F.N_TASKERS * E + ((E + 7) // 8) * 8  # reward, greedy, done of the output block
    envs, res = {}, {}
    for layout, reward, path in VARIANTS:
        key = f"{layout}/{reward} ({path})"
        cfg = dict(base, reward_type=reward, obs_returned=("flatten" if path == "old" else layout))
        env = VecSSATaskerEnv(cfg, E, seeds=list(range(E)), rng="device")
        envs[key] = (env, path == "old")
        obs_bytes = (32 if layout == "aer" and path == "new" else 96) * N
        res[key] = {"obs_returned": layout, "reward_type": reward, "path": path, "ms_per_step": [], "wall_ms_per_step": [],
                    "d2h_obs_bytes_per_step": obs_bytes, "d2h_bytes_per_step": obs_bytes + tail,
                    "graph_kernels_per_step": None, "distinct_step_indices_per_step": []}
        if path == "old":
            res[key]["per_distinct_index"] = ("one ssa_unit_hx_aer call: 2 cudaMalloc, pageable H2D of 48 B and D2H of 24 B "
                                              "per object at that index, 1 kernel, 2 cudaFree")

    def step(env, old):
        obs, r, d, _ = env.vector_step(env.greedy_actions())
        if old:
            obs = old_aer(env, obs)
        return obs

    for key, (env, old) in envs.items():  # episodes spread over many step indices before the first timed run
        for _ in range(a.warmup):
            step(env, old)
    torch.cuda.synchronize()
    for rep in range(a.reps):
        for key, (env, old) in envs.items():
            distinct = 0
            l0 = env.ukf.launch_count
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record()
            for _ in range(a.steps):
                step(env, old)
                distinct += len(np.unique(env.i))
            e1.record()
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            r = res[key]
            r["ms_per_step"].append(e0.elapsed_time(e1) / a.steps)
            r["wall_ms_per_step"].append(wall * 1e3 / a.steps)
            r["graph_kernels_per_step"] = (env.ukf.launch_count - l0) / a.steps
            r["distinct_step_indices_per_step"].append(distinct / a.steps)
    for r in res.values():
        r["ms_per_step_median"] = float(np.median(r["ms_per_step"]))
    out = {"tool": "tools/c3_layouts.py", "gpu": gpu_info(), "envs": E, "rso_count": m, "episode_steps": base["steps"],
           "steps_per_rep": a.steps, "reps": a.reps, "warmup_steps": a.warmup, "actions": "device visible-greedy tasker",
           "timing": "CUDA events around --steps vector_step calls, each of which ends in a synchronise",
           "variants": res}
    txt = json.dumps(out, indent=1)
    print(txt)
    if a.out:
        with open(a.out, "w") as f:
            f.write(txt + "\n")
    for env, _ in envs.values():
        env.close()


if __name__ == "__main__":
    main()
