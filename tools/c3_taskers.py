#!/usr/bin/env python
"""The nine agents of agents.py as device taskers (VecSSATaskerEnv.set_tasker, ssa_ukf_rollout_tasker) at C3:
E = 4 096 environments, the default configuration (m = 10, 'jones'), flatten layout, config['episode_stats'] on.

1. Agent comparison (the loop of the reference's rl_agents/compare_agents.py): each agent from a fresh reset until every
   environment has finished --episodes episodes; per agent the mean return, length, ANEES and NIS (means of the finite
   values) over those first episodes of every environment, from the device's episode records (infos[e]['episode']).
2. Step time, one env per agent, measured in alternation and repeated (--reps) after --warmup steps: ms per
   vector_step() with the tasker picking the actions (one graph launch, one D2H of the outputs and the taken actions),
   ms per vector_step_device() (the graph alone, no host copies), graph kernels per step (launch_count); and, for
   visible_greedy, the same env stepped by vector_step(env.greedy_actions()) with external actions (D2H of the greedy
   block, host fill-in of the -1 columns, H2D of the actions).  CUDA events around --steps calls, each vector_step
   ending in a synchronise.
  python tools/c3_taskers.py [--envs 4096] [--steps 300] [--warmup 200] [--reps 3] [--episodes 1] [--out FILE]"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

AGENTS = ["naive_greedy", "visible_greedy", "pos_error_greedy", "vel_error_greedy", "visible_greedy_aer", "shannon",
          "naive_random", "visible_random", "visible_greedy_spoiled"]


def compare(env, k):
    """Records of the first k finished episodes of every environment (from the current fresh reset)."""
    E = env.E
    seen = np.zeros(E, np.int64)
    recs = []
    steps = 0
    while seen.min() < k:
        _, _, dones, infos = env.vector_step()
        steps += 1
        for e in np.flatnonzero(dones):
            if seen[e] < k:
                recs.append(infos[e]["episode"])
            seen[e] += 1
    mean = lambda key: float(np.nanmean([r[key] for r in recs]))  # noqa: E731
    return {"episodes": len(recs), "vector_steps": steps, "mean_return": mean("r"), "mean_length": mean("l"),
            "mean_anees": mean("anees"), "mean_nis": mean("nis")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--episodes", type=int, default=1)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from c3_layouts import gpu_info
    from ssa_gym_b200 import env_config
    from ssa_gym_b200.catalog import synthetic_catalog
    from ssa_gym_b200.transformations import gcrs2irts_matrix_approx, time_table
    from ssa_gym_b200.vec_env import VecSSATaskerEnv
    if not torch.cuda.is_available():
        raise SystemExit("c3_taskers measures on the GPU: no CUDA device visible")
    E = a.envs
    cfg = dict(env_config)
    cfg["orbits"] = synthetic_catalog(20000, 0)
    cfg["trans_matrix"] = gcrs2irts_matrix_approx(time_table(cfg["t_0"], cfg["time_step"], cfg["steps"]))
    cfg.update(obs_returned="flatten", episode_stats=True)

    def make(agent):
        env = VecSSATaskerEnv(cfg, E, seeds=list(range(E)), rng="device")
        if agent is not None:
            env.set_tasker(agent)
        return env

    envs = {name: make(name) for name in AGENTS}
    envs["visible_greedy external"] = make(None)
    steppers = {name: env.vector_step for name, env in envs.items()}
    ext = envs["visible_greedy external"]
    steppers["visible_greedy external"] = lambda: ext.vector_step(ext.greedy_actions())

    table = {name: compare(envs[name], a.episodes) for name in AGENTS}

    res = {name: {"ms_per_step": [], "device_io_ms_per_step": [], "graph_kernels_per_step": None} for name in envs}
    for name in envs:
        for _ in range(a.warmup):
            steppers[name]()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(a.reps):
        for name, env in envs.items():
            r = res[name]
            e0.record()
            for _ in range(a.steps):
                steppers[name]()
            e1.record()
            torch.cuda.synchronize()
            r["ms_per_step"].append(e0.elapsed_time(e1) / a.steps)
            if name.endswith("external"):
                continue  # (its device loop is the same graph as the visible_greedy tasker's, with no pick)
            l0 = env.ukf.launch_count
            e0.record()
            for _ in range(a.steps):
                env.vector_step_device()
            e1.record()
            torch.cuda.synchronize()
            r["device_io_ms_per_step"].append(e0.elapsed_time(e1) / a.steps)
            r["graph_kernels_per_step"] = (env.ukf.launch_count - l0) / a.steps
    for r in res.values():
        r["ms_per_step_median"] = float(np.median(r["ms_per_step"]))
        r["device_io_ms_per_step_median"] = float(np.median(r["device_io_ms_per_step"])) if r["device_io_ms_per_step"] else None
    out = {"tool": "tools/c3_taskers.py", "gpu": gpu_info(), "envs": E, "rso_count": cfg["rso_count"],
           "episode_steps": cfg["steps"], "reward_type": cfg["reward_type"], "update_interval": cfg["update_interval"],
           "steps_per_rep": a.steps, "reps": a.reps, "warmup_steps": a.warmup,
           "timing": "CUDA events around --steps calls; every vector_step ends in a synchronise and includes the "
                     "episode-record downloads of the steps on which episodes finished",
           "comparison": {"episodes_per_env": a.episodes, "seeds": f"0 .. {E - 1}", "agents": table},
           "step_time": res}
    txt = json.dumps(out, indent=1)
    print(txt)
    if a.out:
        with open(a.out, "w") as f:
            f.write(txt + "\n")
    for env in envs.values():
        env.close()


if __name__ == "__main__":
    main()
