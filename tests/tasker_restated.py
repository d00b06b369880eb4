"""numpy restatement of the device taskers (ssa_tasker_pick, csrc/ssa_rng.h; ssa_ukf_rollout_tasker) and an EpisodicTwin
that runs them: shared by tests/test_tasker_pick_host.py (CPU) and tests/test_gpu_taskers.py."""
import numpy as np

import helpers as H
from ssa_gym_b200 import _lib as F

STREAM_ACT = 3


def philox(ctr, key):
    """Philox4x32-10 through the host twin: four uint32 words."""
    c = np.array(ctr, dtype=np.uint32); k = np.array(key, dtype=np.uint32); o = np.zeros(4, np.uint32)
    H.twin().twin_philox(H.p(c), H.p(k), H.p(o))
    return [int(v) for v in o]


def mulhi32(a, b):
    return (int(a) * int(b)) >> 32


def u52(hi, lo):
    """ssa_u52: (k + 0.5) / 2^52 of the top 52 bits of hi:lo."""
    return (float(((int(hi) << 32) | int(lo)) >> 12) + 0.5) * 2.220446049250313e-16


def candidates(vis):
    """agents._candidates on the visibility flags: the visible indices, None where `not np.any(idx)`."""
    idx = np.flatnonzero(vis)
    return idx if np.any(idx) else None


def pick(key, ep, step, m, tasker, greedy, vis, p):
    """(action, how) of tasker 0 .. 8 for environment key (uint64 seed) at episode ep, step `step`; how is 'column',
    'fallback' (the uniform action of an empty greedy column or of no candidates), 'random' (naive_random),
    'visible' (visible_random among the candidates), 'greedy' or 'spoiled' (visible_greedy_spoiled)."""
    key = int(key)
    v = philox([ep, STREAM_ACT, 0, step], [key & 0xFFFFFFFF, key >> 32])
    fallback = mulhi32(v[0], m)
    if tasker < F.N_TASKERS:
        return (int(greedy[tasker]), "column") if greedy[tasker] >= 0 else (fallback, "fallback")
    if tasker == F.TASKER_NAIVE_RANDOM:
        return fallback, "random"
    idx = candidates(vis)
    if idx is None:
        return fallback, "fallback"
    if tasker == F.TASKER_VISIBLE_RANDOM:
        return int(idx[mulhi32(v[1], len(idx))]), "visible"
    assert tasker == F.TASKER_VISIBLE_GREEDY_SPOILED
    # np.random.choice([greedy, fallback], p=[1 - p, p]): searchsorted(cdf, u, side='right')
    if u52(v[2], v[3]) < 1.0 - p:
        return int(greedy[F.TASKER_VISIBLE_GREEDY]), "greedy"
    return fallback, "spoiled"


class TaskerTwin(H.EpisodicTwin):
    """EpisodicTwin whose step picks the actions as the device tasker does, from the greedy block and visibility the
    previous step left; counts what the picks went through in `seen`."""

    def __init__(self, vec, cfg, tasker, p=0.25):
        super().__init__(vec, cfg)
        self.tasker, self.p = tasker, p
        self.seen = {"resets": 0, "fallback": 0, "only_object_0": 0, "none_visible": 0, "spoiled": 0, "skipped": 0}

    def step(self, actions=None, auto_reset=True):
        assert actions is None
        E, m = self.E, self.m
        vis = self.st.visible.reshape(E, m).astype(bool)
        step = self.step_idx + 1
        a = np.empty(E, np.int32)
        for e in range(E):
            a[e], how = pick(self.keys[e], int(self.episode[e]) - 1, int(step[e]), m, self.tasker, self.greedy[e],
                             vis[e], self.p)
            self.seen["fallback"] += how in ("fallback", "random", "spoiled")
            self.seen["spoiled"] += how == "spoiled"
        self.seen["skipped"] += int((step % self.update_interval != 0).sum())
        self.seen["none_visible"] += int((~vis.any(1)).sum())
        self.seen["only_object_0"] += int((vis[:, 0] & ~vis[:, 1:].any(1)).sum())
        self.last_actions = a.astype(np.int64)
        out = super().step(a, auto_reset)
        self.seen["resets"] += int(out[2].sum())
        return out
