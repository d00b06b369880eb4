"""CPU: ssa_pairwise_sum (csrc/ssa_ukf_core.h), the history sum of the episodic mode's 'shaped' reward
(1 - np.sum(rewards[:i]), SS2:345), equals np.sum bit for bit - sign of zero included - on every prefix length
0 .. 4096.  The header is compiled for the host here, with the host twin's flags (contraction off, as on the device),
into a temporary directory."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import helpers as H

_SRC = ('#include "ssa_ukf_core.h"\n'
        'extern "C" void pairwise_sum(const double* a, long n, double* out) { *out = ssa_pairwise_sum(a, n); }\n')


@pytest.fixture(scope="module")
def pairwise_sum(tmp_path_factory):
    gxx = "/usr/bin/g++" if os.path.isfile("/usr/bin/g++") else "g++"  # (as helpers.build_twin)
    d = tmp_path_factory.mktemp("pairwise")
    (d / "pairwise.cpp").write_text(_SRC)
    lib = d / "libpairwise.so"
    subprocess.run([gxx, "-O2", "-std=c++17", "-ffp-contract=off", "-mfma", "-mavx2", "-shared", "-fPIC",
                    "-Wno-unknown-pragmas", "-I", os.path.join(H.ROOT, "ssa_gym_b200", "csrc"), "-o", str(lib),
                    str(d / "pairwise.cpp")], check=True)
    fn = ctypes.CDLL(str(lib)).pairwise_sum
    fn.argtypes = [ctypes.c_void_p, ctypes.c_long, ctypes.c_void_p]
    fn.restype = None
    return fn


N = 4096


def _sequences():
    rng = np.random.RandomState(7)
    yield "reward_steps", rng.choice([1.0 / 480, -1.0 / 480, 0.0], size=N)
    yield "normal_scaled", rng.normal(size=N) * 10.0 ** rng.uniform(-5, 5, size=N)
    b = rng.normal(size=N // 2) * 10.0 ** rng.uniform(-5, 5, size=N // 2)
    c = np.empty(N)
    c[0::2], c[1::2] = b, -b  # every pair cancels exactly: the sums are zeros of either sign and small remainders
    c[::7] *= 1 + 2.0 ** -40
    yield "cancelling", c
    yield "negative_zeros", np.full(N, -0.0)


@pytest.mark.parametrize("name,a", list(_sequences()))
def test_pairwise_sum_equals_np_sum_on_every_prefix(pairwise_sum, name, a):
    fn = pairwise_sum
    a = np.ascontiguousarray(a, dtype=np.float64)
    out = np.zeros(1)
    got, want = np.empty(N + 1), np.empty(N + 1)
    for k in range(N + 1):
        fn(a.ctypes.data, k, out.ctypes.data)
        got[k], want[k] = out[0], np.sum(a[:k])
    bad = np.where(got.view(np.uint64) != want.view(np.uint64))[0]
    assert bad.size == 0, (name, bad[:10], got[bad[:3]], want[bad[:3]])
    seq = np.empty(N + 1)  # the order matters: a sequential sum differs from np.sum on most prefixes of these inputs
    seq[0] = 0.0
    seq[1:] = np.cumsum(a)
    if name in ("reward_steps", "normal_scaled"):
        assert np.count_nonzero(seq != want) > N // 4
