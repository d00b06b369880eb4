"""CPU: ssa_tasker_pick (csrc/ssa_rng.h), the action a device tasker takes, equals its numpy restatement
(tests/tasker_restated.py, built on the twin's Philox) exactly, over random inputs and the corner cases of agents.py:
nothing visible, only object 0 visible (`not np.any(idx)`), one visible object other than 0, m = 1, p = 0 and 1,
greedy columns of -1.  The header is compiled for the host with the host twin's flags into a temporary directory."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import helpers as H
import tasker_restated as R
from ssa_gym_b200 import _lib as F
from ssa_gym_b200 import agents

_SRC = ('#include "ssa_rng.h"\n'
        'extern "C" int tasker_pick(uint32_t k0, uint32_t k1, uint32_t ep, uint32_t step, int m, int tasker,\n'
        '                           const int32_t* greedy, const uint8_t* vis, double p) {\n'
        '  return ssa_tasker_pick(k0, k1, ep, step, m, tasker, greedy, vis, p);\n'
        '}\n')
TASKERS = list(range(F.TASKER_VISIBLE_GREEDY_SPOILED + 1))


@pytest.fixture(scope="module")
def tasker_pick(tmp_path_factory):
    gxx = "/usr/bin/g++" if os.path.isfile("/usr/bin/g++") else "g++"  # (as helpers.build_twin)
    d = tmp_path_factory.mktemp("tasker_pick")
    (d / "tasker_pick.cpp").write_text(_SRC)
    lib = d / "libtasker_pick.so"
    subprocess.run([gxx, "-O2", "-std=c++17", "-ffp-contract=off", "-mfma", "-mavx2", "-shared", "-fPIC",
                    "-Wno-unknown-pragmas", "-I", os.path.join(H.ROOT, "ssa_gym_b200", "csrc"), "-o", str(lib),
                    str(d / "tasker_pick.cpp")], check=True)
    fn = ctypes.CDLL(str(lib)).tasker_pick
    u32 = ctypes.c_uint32
    fn.argtypes = [u32, u32, u32, u32, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_double]
    fn.restype = ctypes.c_int

    def call(key, ep, step, m, tasker, greedy, vis, p):
        g = np.ascontiguousarray(greedy, dtype=np.int32)
        v = np.ascontiguousarray(vis, dtype=np.uint8)
        key = int(key)
        return fn(key & 0xFFFFFFFF, key >> 32, ep, step, m, tasker, g.ctypes.data, v.ctypes.data, p)
    return call


def _greedy(rng, m, vis):
    """A greedy row as the reduction leaves it: column 0 any object, the visible-* columns a visible object or -1."""
    g = np.full(F.N_TASKERS, -1, np.int32)
    g[0] = rng.randint(m)
    idx = R.candidates(vis)
    if idx is not None:
        g[1:] = rng.choice(idx, size=F.N_TASKERS - 1)
    return g


def _cases():
    rng = np.random.RandomState(5)
    for _ in range(400):  # random inputs
        m = int(rng.choice([1, 2, 4, 10, 40, 70, 130]))
        vis = rng.rand(m) < rng.uniform(0.0, 1.0)
        yield m, vis, _greedy(rng, m, vis), float(rng.choice([0.0, 0.25, rng.rand(), 1.0]))
    for m in (1, 2, 10, 70):
        none = np.zeros(m, bool)
        only0 = none.copy(); only0[0] = True
        yield m, none, _greedy(rng, m, none), 0.25
        yield m, only0, _greedy(rng, m, only0), 0.25
        if m > 1:
            one = none.copy(); one[m - 1] = True
            both = only0.copy(); both[m // 2] = True
            for v in (one, both):
                for p in (0.0, 1.0, 0.5):
                    yield m, v, _greedy(rng, m, v), p
            yield m, np.ones(m, bool), np.full(F.N_TASKERS, -1, np.int32), 0.25  # greedy columns of -1


def test_pick_equals_restatement(tasker_pick):
    rng = np.random.RandomState(9)
    n, hows = 0, set()
    for m, vis, g, p in _cases():
        key = int(rng.randint(0, 2 ** 63, dtype=np.int64)) * 2 + int(rng.randint(2))
        ep, step = int(rng.randint(0, 2 ** 31)), int(rng.randint(0, 2 ** 31))
        for t in TASKERS:
            want, how = R.pick(key, ep, step, m, t, g, vis, p)
            got = tasker_pick(key, ep, step, m, t, g, vis, p)
            assert got == want, (m, t, p, vis.astype(int), g, got, want)
            assert 0 <= got < m
            hows.add((t, how))
            n += 1
    # every branch of every tasker was taken
    assert {h for t, h in hows if t < F.N_TASKERS} == {"column", "fallback"}
    assert {h for t, h in hows if t == F.TASKER_VISIBLE_RANDOM} == {"visible", "fallback"}
    assert {h for t, h in hows if t == F.TASKER_VISIBLE_GREEDY_SPOILED} == {"greedy", "spoiled", "fallback"}
    assert n > 3000


@pytest.mark.parametrize("p,how", [(0.0, "greedy"), (1.0, "spoiled")])
def test_spoiled_extremes(tasker_pick, p, how):
    """p = 0 always takes the visible-greedy column, p = 1 always the uniform action (u52 lies in (0, 1))."""
    m = 10
    vis = np.zeros(m, bool); vis[[0, 3, 7]] = True
    g = np.array([2, 7, 3, 3, 7, 3], np.int32)
    for step in range(200):
        want, h = R.pick(77, 1, step, m, F.TASKER_VISIBLE_GREEDY_SPOILED, g, vis, p)
        assert h == how and tasker_pick(77, 1, step, m, F.TASKER_VISIBLE_GREEDY_SPOILED, g, vis, p) == want


def test_candidate_rule_is_agents_candidates():
    """The restatement's candidates are agents._candidates of an env whose visible_objects() are the flagged indices."""
    class Stub:
        def __init__(self, vis):
            self.vis = vis

        def visible_objects(self):
            return np.where(self.vis)[0]

    rng = np.random.RandomState(3)
    cases = [np.zeros(5, bool), np.eye(5, dtype=bool)[0], np.eye(5, dtype=bool)[4], np.ones(1, bool), np.zeros(1, bool)]
    cases += [rng.rand(int(rng.randint(1, 40))) < rng.rand() for _ in range(300)]
    for vis in cases:
        want = agents._candidates(Stub(vis))
        got = R.candidates(vis)
        assert (got is None) == (want is None), vis
        if got is not None:
            assert np.array_equal(got, want)
