#!/usr/bin/env python
"""C3 (VecSSATaskerEnv, rng='device', 'flatten' layout) with running normalization of observations and returns
(config['normalize'] = True, k_normalize inside the step graph) against the raw environment, and against the same
normalization written as torch ops over device_views() by the caller.

Environments, each measured in alternation and repeated (--reps), all with the device's visible-greedy tasker (so the
same step serves vector_step and vector_step_device):
  raw_f64   obs float64 (the default)       raw_f32   obs_dtype float32       norm   normalize=True (float32 normalized obs)
Reported per environment: ms per step of vector_step (CUDA events around --steps calls, each ending in a synchronise) and
of vector_step_device (the step graph alone, no host copies), graph kernels per step.  For norm, k_normalize's own time
(torch.profiler, a separate pass).  Collector-shaped loops on the device (every step copies the observations and rewards
into a 32-step fragment): 'kernel' = norm's vector_step_device reading obs_norm / reward_norm; 'torch_ops' = raw_f64's
vector_step_device followed by VecNormalize's arithmetic as torch ops (batch mean / var, merge, normalize, clip, returns).
  python tools/c3_normalize.py [--envs 4096] [--steps 500] [--warmup 300] [--reps 3] [--out FILE]"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))


class TorchNormalize:
    """VecNormalize's step arithmetic as torch ops on the device views of a raw environment."""

    def __init__(self, E, F, dev, gamma=0.99, eps=1e-8, clip=10.0):
        import torch
        t = lambda *s: torch.zeros(*s, dtype=torch.float64, device=dev)
        self.mean, self.var, self.count = t(F), t(F) + 1, 1e-4
        self.rmean, self.rvar, self.rcount = t(()), t(()) + 1, 1e-4
        self.returns = t(E)
        self.gamma, self.eps, self.clip = gamma, eps, clip

    @staticmethod
    def _merge(mean, var, count, x):
        bm, bv, bc = x.mean(0), x.var(0, unbiased=False), x.shape[0]
        delta = bm - mean
        tot = count + bc
        new_mean = mean + delta * bc / tot
        m2 = var * count + bv * bc + delta * delta * count * bc / tot
        return new_mean, m2 / tot, tot

    def step(self, obs, reward, done):
        self.mean, self.var, self.count = self._merge(self.mean, self.var, self.count, obs)
        o = ((obs - self.mean) / (self.var + self.eps).sqrt()).clamp(-self.clip, self.clip).float()
        self.returns = self.returns * self.gamma + reward
        self.rmean, self.rvar, self.rcount = self._merge(self.rmean, self.rvar, self.rcount, self.returns)
        r = (reward / (self.rvar + self.eps).sqrt()).clamp(-self.clip, self.clip)
        self.returns.masked_fill_(done.bool(), 0.0)
        return o, r


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
        raise SystemExit("c3_normalize measures on the GPU: no CUDA device visible")
    E = a.envs
    base = dict(env_config)
    base["orbits"] = synthetic_catalog(20000, 0)
    base["trans_matrix"] = gcrs2irts_matrix_approx(time_table(base["t_0"], base["time_step"], base["steps"]))
    m = base["rso_count"]
    F = 12 * m
    variants = {"raw_f64": {}, "raw_f32": {"obs_dtype": "float32"}, "norm": {"normalize": True}}
    envs, res = {}, {}
    for key, over in variants.items():
        env = VecSSATaskerEnv(dict(base, obs_returned="flatten", **over), E, seeds=list(range(E)), rng="device")
        env.set_tasker("visible_greedy")
        envs[key] = env
        res[key] = {"config": over, "ms_per_step": [], "device_io_ms_per_step": [], "graph_kernels_per_step": None}
    dev = torch.device("cuda", 0)
    frag_o = torch.empty((32, E, F), dtype=torch.float32, device=dev)
    frag_r = torch.empty((32, E), dtype=torch.float64, device=dev)
    tn = TorchNormalize(E, F, dev)
    vraw, vnorm = envs["raw_f64"].device_views(), envs["norm"].device_views()

    def loop_kernel(t):
        envs["norm"].vector_step_device()
        frag_o[t % 32].copy_(vnorm["obs_norm"])
        frag_r[t % 32].copy_(vnorm["reward_norm"])

    def loop_torch(t):
        envs["raw_f64"].vector_step_device()
        o, r = tn.step(vraw["obs"], vraw["reward"], vraw["done"])
        frag_o[t % 32].copy_(o)
        frag_r[t % 32].copy_(r)
    loops = {"kernel": loop_kernel, "torch_ops": loop_torch}
    coll = {k: [] for k in loops}

    for env in envs.values():  # episodes spread over many step indices before the first timed run
        for _ in range(a.warmup):
            env.vector_step()
    for k, f in loops.items():
        for t in range(50):
            f(t)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for rep in range(a.reps):
        for key, env in envs.items():
            l0 = env.ukf.launch_count
            e0.record()
            for _ in range(a.steps):
                env.vector_step()
            e1.record()
            torch.cuda.synchronize()
            r = res[key]
            r["ms_per_step"].append(e0.elapsed_time(e1) / a.steps)
            r["graph_kernels_per_step"] = (env.ukf.launch_count - l0) / a.steps
            e0.record()
            for _ in range(a.steps):
                env.vector_step_device()
            e1.record()
            torch.cuda.synchronize()
            r["device_io_ms_per_step"].append(e0.elapsed_time(e1) / a.steps)
        for k, f in loops.items():
            e0.record()
            for t in range(a.steps):
                f(t)
            e1.record()
            torch.cuda.synchronize()
            coll[k].append(e0.elapsed_time(e1) / a.steps)
    for r in res.values():
        r["ms_per_step_median"] = float(np.median(r["ms_per_step"]))
        r["device_io_ms_per_step_median"] = float(np.median(r["device_io_ms_per_step"]))
    res["norm"]["graph_overhead_ms_per_step_median"] = (res["norm"]["device_io_ms_per_step_median"] -
                                                        res["raw_f64"]["device_io_ms_per_step_median"])
    # k_normalize's own time: torch.profiler over device steps of the normalized environment (its own pass)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(200):
            envs["norm"].vector_step_device()
        torch.cuda.synchronize()
    kern = {}
    for ev in prof.key_averages():
        if ev.device_type is not None and "k_normalize" in ev.key:
            t_us = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
            kern = {"name": ev.key, "calls": ev.count, "mean_us": t_us / max(ev.count, 1)}
    out = {"tool": "tools/c3_normalize.py", "gpu": gpu_info(), "envs": E, "rso_count": m, "features": F,
           "episode_steps": base["steps"], "steps_per_rep": a.steps, "reps": a.reps, "warmup_steps": a.warmup,
           "actions": "device visible-greedy tasker (set_tasker)",
           "timing": "CUDA events around --steps calls; vector_step ends each step in a synchronise, the device loops do not",
           "variants": res, "k_normalize": kern,
           "collector_ms_per_step": {k: {"runs": v, "median": float(np.median(v))} for k, v in coll.items()}}
    txt = json.dumps(out, indent=1)
    print(txt)
    if a.out:
        with open(a.out, "w") as f:
            f.write(txt + "\n")
    for env in envs.values():
        env.close()


if __name__ == "__main__":
    main()
