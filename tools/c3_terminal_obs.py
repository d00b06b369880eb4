#!/usr/bin/env python
"""C3 (VecSSATaskerEnv, rng='device', flatten layout) step time with and without the episode-boundary infos
(config['terminal_observation']: infos[e]['TimeLimit.truncated'] and infos[e]['terminal_observation'] of every finished
environment, one ssa_ukf_rollout_terminal_obs_download per step on which environments finished).

Variants, each one VecSSATaskerEnv in one process, measured in alternation and repeated (--reps): jones / trinary
reward, switch off / on. Actions are the device's visible-greedy picks (greedy_actions, as bench.py's C3 workload).
Reported per variant: ms per step (CUDA events around a run of --steps vector_step calls, each ending in a synchronise;
every repetition), the same for vector_step_device (actions already on the device, outputs left there, no host copies
and no info dicts: the step graph alone, which records the final observations whatever the switch), graph kernels per
step (launch_count), and for the switch-on variants the steps on which final rows were downloaded, the environments
finished per such step and the host time of each download call (a host clock around rollout_terminal_obs, which ends in
a stream synchronise).
  python tools/c3_terminal_obs.py [--envs 4096] [--steps 500] [--warmup 300] [--reps 3] [--out FILE]"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

VARIANTS = [("jones", False), ("jones", True), ("trinary", False), ("trinary", True)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--warmup", type=int, default=300)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from c3_layouts import gpu_info
    from ssa_gym_b200 import env_config
    from ssa_gym_b200.catalog import synthetic_catalog
    from ssa_gym_b200.transformations import gcrs2irts_matrix_approx, time_table
    from ssa_gym_b200.vec_env import VecSSATaskerEnv
    if not torch.cuda.is_available():
        raise SystemExit("c3_terminal_obs measures on the GPU: no CUDA device visible")
    E = a.envs
    base = dict(env_config)
    base["orbits"] = synthetic_catalog(20000, 0)
    base["trans_matrix"] = gcrs2irts_matrix_approx(time_table(base["t_0"], base["time_step"], base["steps"]))
    m = base["rso_count"]
    envs, res, dl = {}, {}, {}
    for reward, on in VARIANTS:
        key = f"flatten/{reward} terminal_observation {'on' if on else 'off'}"
        env = VecSSATaskerEnv(dict(base, reward_type=reward, obs_returned="flatten", terminal_observation=on), E,
                              seeds=list(range(E)), rng="device")
        envs[key] = env
        res[key] = {"reward_type": reward, "terminal_observation": on, "ms_per_step": [], "device_io_ms_per_step": [],
                    "graph_kernels_per_step": None}
        if on:  # time every download call of the env's vector_step
            calls = dl[key] = []
            inner = env.ukf.rollout_terminal_obs

            def timed(envs_, _inner=inner, _calls=calls):
                t0 = time.perf_counter()
                out = _inner(envs_)
                _calls.append(((time.perf_counter() - t0) * 1e3, len(envs_)))
                return out
            env.ukf.rollout_terminal_obs = timed
            res[key].update({"download_steps": [], "download_ms": [], "finished_per_download_step": []})

    for env in envs.values():  # episodes spread over many step indices before the first timed run
        for _ in range(a.warmup):
            env.vector_step(env.greedy_actions())
    torch.cuda.synchronize()
    for rep in range(a.reps):
        for key, env in envs.items():
            if key in dl:
                dl[key].clear()
            l0 = env.ukf.launch_count
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.steps):
                env.vector_step(env.greedy_actions())
            e1.record()
            torch.cuda.synchronize()
            r = res[key]
            r["ms_per_step"].append(e0.elapsed_time(e1) / a.steps)
            if key in dl:
                r["download_steps"].append(len(dl[key]))
                r["download_ms"] += [c[0] for c in dl[key]]
                r["finished_per_download_step"] += [c[1] for c in dl[key]]
                # (launch_count includes the gather kernel of each download)
                r["graph_kernels_per_step"] = (env.ukf.launch_count - l0 - len(dl[key])) / a.steps
            else:
                r["graph_kernels_per_step"] = (env.ukf.launch_count - l0) / a.steps
            e0.record()
            for _ in range(a.steps):
                env.vector_step_device()
            e1.record()
            torch.cuda.synchronize()
            r["device_io_ms_per_step"].append(e0.elapsed_time(e1) / a.steps)
    for key, r in res.items():
        r["ms_per_step_median"] = float(np.median(r["ms_per_step"]))
        r["device_io_ms_per_step_median"] = float(np.median(r["device_io_ms_per_step"]))
        if key in dl:
            r["download_ms_median"] = float(np.median(r["download_ms"])) if r["download_ms"] else None
            r["finished_per_download_step_median"] = (float(np.median(r["finished_per_download_step"]))
                                                      if r["finished_per_download_step"] else None)
            r["download_ms"] = [round(v, 4) for v in r["download_ms"]]
    for reward in ("jones", "trinary"):
        on, off = res[f"flatten/{reward} terminal_observation on"], res[f"flatten/{reward} terminal_observation off"]
        on["overhead_ms_per_step_median"] = on["ms_per_step_median"] - off["ms_per_step_median"]
    out = {"tool": "tools/c3_terminal_obs.py", "gpu": gpu_info(), "envs": E, "rso_count": m, "episode_steps": base["steps"],
           "steps_per_rep": a.steps, "reps": a.reps, "warmup_steps": a.warmup, "actions": "device visible-greedy picks",
           "timing": "CUDA events around --steps vector_step calls, each of which ends in a synchronise; the switch-on "
                     "steps include their final-row downloads and info dicts",
           "variants": res}
    txt = json.dumps(out, indent=1)
    print(txt)
    if a.out:
        with open(a.out, "w") as f:
            f.write(txt + "\n")
    for env in envs.values():
        env.close()


if __name__ == "__main__":
    main()
