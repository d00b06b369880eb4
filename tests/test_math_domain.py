"""The fp64 library (ssa_gym_b200/csrc/ssa_math.h) over every argument each function accepts, and at its special values.

tests/test_math_accuracy.py bounds the host build on the ranges the propagation uses; tests/test_gpu_bitexact.py shows
GPU == host twin there.  Neither sees NaN, inf, subnormals, overflow and underflow edges, the sign of zero or the
argument reduction of sin / cos far from zero.  Here, on the host twin (CPU) and through ssa_unit_math (-m gpu):
  * a special-value table per function, against numpy's results (Python's % for pymod): NaN where numpy gives NaN,
    the same infinities, the same sign of zero, finite results inside the function's ulp bound (mpmath, 200 bits);
  * log-uniform sweeps over each whole domain against mpmath, in ulps of the correctly rounded result (for a subnormal
    result: of its binade, 2^-1074);
  * sin / cos / tan at the doubles nearest k pi/2, 10^4 values of k per decade up to the end of the Cody-Waite range
    (2^30) and the Payne-Hanek range beyond it;
  * fx states that reach the true-anomaly conversion with a NaN hyperbolic anomaly: NaN and a failed filter, as the
    oracle (libm tanh) returns.
The bounds are those of test_math_accuracy.py wherever they hold; the few ranges that cannot meet them say why."""
import functools

import numpy as np
import pytest

import helpers as H

mp = pytest.importorskip("mpmath")
mp.mp.prec = 200

DMAX = np.finfo(np.float64).max
DMIN = np.finfo(np.float64).tiny
DEN = 5e-324
NAN_P = np.array([0x7FF8000000000000], np.uint64).view(np.float64)[0]
NAN_N = np.array([0xFFF8000000000000], np.uint64).view(np.float64)[0]
INF = np.inf
COMMON = [NAN_P, NAN_N, INF, -INF, 0.0, -0.0, DEN, -DEN, DMIN, -DMIN, DMAX, -DMAX, 1.0, -1.0, 0.5, -0.5]
EXP_O, EXP_U1, EXP_U0 = 709.782712893384, -708.3964185322641, -745.1332191019411   # overflow, DBL_MIN, 2^-1075
SINH_O = 710.4758600739439


def nb(v):
    """v and its two nextafter neighbours."""
    return [np.nextafter(v, -INF), v, np.nextafter(v, INF)]


def pm(vals):
    return list(vals) + [-v for v in vals]


# the same bounds as test_math_accuracy.py; pow23 has none there (see test_pow23_whole_domain)
BOUND = {"sin": 1.6, "cos": 1.6, "tan": 3.0, "atan": 1.1, "asin": 1.3, "acos": 1.3, "exp": 1.1, "log": 1.1,
         "sinh": 3.0, "cosh": 2.0, "tanh": 3.5, "atanh": 3.5, "asinh": 3.5, "acosh": 3.5, "atan2": 1.5}
MPF = {"sin": mp.sin, "cos": mp.cos, "tan": mp.tan, "atan": mp.atan, "asin": mp.asin, "acos": mp.acos, "exp": mp.exp,
       "log": mp.log, "sinh": mp.sinh, "cosh": mp.cosh, "tanh": mp.tanh, "atanh": mp.atanh, "asinh": mp.asinh,
       "acosh": mp.acosh, "pow23": lambda v: mp.power(v, mp.mpf(2) / 3)}
NPF = {"sin": np.sin, "cos": np.cos, "tan": np.tan, "atan": np.arctan, "asin": np.arcsin, "acos": np.arccos,
       "exp": np.exp, "log": np.log, "sinh": np.sinh, "cosh": np.cosh, "tanh": np.tanh, "atanh": np.arctanh,
       "asinh": np.arcsinh, "acosh": np.arccosh, "pow23": lambda v: np.power(v, 2.0 / 3.0)}
UNARY = [op for op in H.MATH_OPS if op not in ("atan2", "pymod")]

PIO2_NEAR = [float(mp.pi / 2), np.nextafter(float(mp.pi / 2), 0.0), np.nextafter(float(mp.pi / 2), 4.0)]
SPECIAL = {
    "sin": COMMON + pm([1e-300, 2.0 ** -27, np.nextafter(2.0 ** -27, 0), 2.0 ** 30, np.nextafter(2.0 ** 30, 0),
                        1e16, 2.0 ** 60, 1e22, 1e300]),
    "tan": COMMON + pm(PIO2_NEAR + [1e-300, 2.0 ** 30, 1e16, 1e22]),
    "atan": COMMON + pm([1e300, 2.0 ** 1020, 1e-300]),
    "asin": COMMON + pm(nb(1.0)), "acos": COMMON + pm(nb(1.0)),
    "exp": COMMON + nb(EXP_O) + nb(EXP_U1) + nb(EXP_U0) + [709.0, 709.5, -708.2, -740.0, -708.0, 1e300, -1e300],
    "log": COMMON + nb(0.0) + nb(1.0) + [1e-310, 1e300],
    "sinh": COMMON + pm(nb(EXP_O) + nb(SINH_O) + [709.0, 709.5, 22.0, 1e300]),
    "cosh": COMMON + pm(nb(EXP_O) + nb(SINH_O) + [709.0, 709.5, 22.0, 1e300]),
    "tanh": COMMON + pm([22.0, np.nextafter(22.0, 0), 1e-300, 1e300]),
    "atanh": COMMON + pm(nb(1.0) + [1e-300]),
    "asinh": COMMON + pm([1e8, np.nextafter(1e8, INF), 1e300, 1e-300]),
    "acosh": COMMON + nb(1.0) + [2.0 ** 28, np.nextafter(2.0 ** 28, INF), 1e154, 1e200, 1e300],
    # x^(2/3) = exp(2/3 log x) is NaN for every x < 0; numpy's pow(-inf, 2/3) = +inf (C99 Annex F) is the one exception
    "pow23": [v for v in COMMON if v != -INF] + nb(0.0) + [1e-310, 1e300],
}
SPECIAL["cos"] = SPECIAL["sin"]
assert set(SPECIAL) == set(UNARY)
SP2 = COMMON + [1e300, -1e300, 3.0, -3.0, 1e-300]


def ulp_err(y, x, fn):
    """|y - fn(x)| in ulps of the correctly rounded fn(x) (np.spacing: 2^-1074 for a subnormal one); a result that
    rounds to 0 must be 0."""
    out = np.empty(len(y))
    for i, (yi, xi) in enumerate(zip(y, x)):
        ref = fn(*[mp.mpf(float(v)) for v in np.atleast_1d(xi)])
        rf = float(ref)
        if rf == 0:
            out[i] = 0.0 if yi == 0 else np.inf
        elif not np.isfinite(yi):
            out[i] = np.inf
        else:
            out[i] = float(abs(mp.mpf(float(yi)) - ref) / mp.mpf(float(np.spacing(abs(rf)))))
    return out


def numpy_semantics(y, ref):
    """Positions of NaN equal, infinities equal, zeros of the same sign; returns the mask of finite non-zero ones."""
    y, ref = np.asarray(y), np.asarray(ref)
    assert np.array_equal(np.isnan(y), np.isnan(ref)), np.where(np.isnan(y) != np.isnan(ref))[0]
    inf = np.isinf(ref)
    assert np.array_equal(np.isinf(y), inf) and np.array_equal(y[inf], ref[inf]), np.where(np.isinf(y) != inf)[0]
    z = ref == 0
    assert np.array_equal(y[z], ref[z]) and np.array_equal(np.signbit(y[z]), np.signbit(ref[z])), \
        (np.where(z)[0], y[z], ref[z])
    return np.isfinite(ref) & ~z


def pow23_bound(x):
    """x^(2/3) = exp(2/3 log x): the rounding errors of log x and of 2/3 log x (an ulp each, relative) are multiplied
    by |2/3 log x| in the result, so the bound grows with it: 1.5 + 1.5 |2/3 log x| ulp, 1.5 around x = 1 and ~750 at
    the ends of the domain.  Barker's equation calls it on B + sqrt(B^2 + 1) >= 1 of moderate size."""
    return 1.5 + 1.5 * np.abs(2.0 / 3.0 * np.log(x))


def check_special(op, x, y):
    with np.errstate(all="ignore"):
        ref = NPF[op](x)
    fin = numpy_semantics(y, ref)
    e = ulp_err(y[fin], x[fin], MPF[op])
    bound = pow23_bound(x[fin]) if op == "pow23" else BOUND[op]
    assert np.all(e <= bound), (op, x[fin][np.argmax(e - bound)], y[fin][np.argmax(e - bound)], e.max())


def special_binary():
    a, b = np.meshgrid(SP2, SP2)
    return a.ravel(), b.ravel()


def check_atan2(a, b, y):
    ref = np.arctan2(a, b)
    fin = numpy_semantics(y, ref)
    # +-0 / +-pi for y = +-0 (mpmath has no signed zero), +-pi/4 / +-3pi/4 at two infinities: numpy's correctly
    # rounded values
    both = fin & ((np.isinf(a) & np.isinf(b)) | (a == 0))
    assert np.array_equal(y[both], ref[both]), (a[both], b[both], y[both])
    fin &= ~both
    big = mp.mpf(10) ** 1000  # one infinite argument: the limit, atan2 at +-10^1000
    e = ulp_err(y[fin], np.stack([a[fin], b[fin]], 1),
                lambda u, v: mp.atan2(*[mp.sign(t) * big if mp.isinf(t) else t for t in (u, v)]))
    assert e.max(initial=0.0) <= BOUND["atan2"], (a[fin][np.argmax(e)], b[fin][np.argmax(e)], e.max())


PYMOD_B = 2 * np.pi


def pymod_args():
    a = np.array(COMMON + [1e300, -1e300, 7.0, -7.0, PYMOD_B, -PYMOD_B, np.nextafter(PYMOD_B, 0), -1e-300])
    return a, np.full(a.size, PYMOD_B)


def python_mod(a, b):
    out = np.empty(a.size)
    for i, (u, v) in enumerate(zip(a, b)):
        out[i] = float(u) % float(v) if np.isfinite(u) else np.nan
    return out


# ---- special values -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("op", UNARY)
def test_special_values(op):
    x = np.array(SPECIAL[op])
    check_special(op, x, H.lib_math("twin", op, x))


def test_special_values_atan2():
    a, b = special_binary()
    check_atan2(a, b, H.lib_math("twin", "atan2", a, b))


def test_special_values_pymod():
    a, b = pymod_args()
    y = H.lib_math("twin", "pymod", a, b)
    ref = python_mod(a, b)
    assert H.bits_equal(y, ref) and np.array_equal(np.signbit(y[~np.isnan(y)]), np.signbit(ref[~np.isnan(ref)]))


# ---- whole-domain sweeps --------------------------------------------------------------------------------------------
RNG = np.random.default_rng(20)
N = 3000


def logu(lo, hi, n, signed=True):
    """n doubles log-uniform in [lo, hi], random signs when `signed`."""
    x = np.exp(RNG.uniform(np.log(lo), np.log(hi), n))
    x = np.clip(x, lo, hi)
    return x * RNG.choice([-1.0, 1.0], n) if signed else x


def sweep_args():
    acosh_near1 = 1.0 + logu(1e-16, 1.0, N // 2, False)
    atanh_top = 1.0 - logu(2.0 ** -53, 1.0, N // 2, False)
    d = {
        "exp": np.concatenate([RNG.uniform(EXP_U0, EXP_O, N), logu(1e-300, 745.0, N) * 0.999,
                               RNG.uniform(EXP_U0, EXP_U1, N // 2)]),
        "log": logu(DEN, DMAX, 2 * N, False),
        "sinh": logu(1e-300, SINH_O, N),
        "cosh": logu(1e-300, SINH_O, N),
        "tanh": logu(1e-300, DMAX, N),
        "asinh": logu(1e-300, DMAX, N),
        "acosh": np.concatenate([acosh_near1, logu(1.0, DMAX, N, False)]),
        "atanh": np.concatenate([logu(1e-300, 1.0 - 2.0 ** -53, N), atanh_top * RNG.choice([-1.0, 1.0], N // 2)]),
        "asin": logu(1e-300, 1.0, N), "acos": logu(1e-300, 1.0, N),
        "atan": logu(DEN, DMAX, N),
        "sin": logu(1e-300, DMAX, N), "cos": logu(1e-300, DMAX, N), "tan": logu(1e-300, DMAX, N),
        "pow23": logu(DEN, DMAX, N, False),
    }
    d["acosh"] = np.clip(d["acosh"], 1.0, DMAX)
    d["atanh"] = np.clip(d["atanh"], -(1.0 - 2.0 ** -53), 1.0 - 2.0 ** -53)
    return d


SWEEP = sweep_args()
A2 = (logu(1e-300, 1e300, 2 * N), logu(1e-300, 1e300, 2 * N))


@functools.lru_cache(maxsize=None)
def sweep_err(op):
    x = SWEEP[op]
    return x, ulp_err(H.lib_math("twin", op, x), x, MPF[op])


@pytest.mark.parametrize("op", [op for op in UNARY if op not in ("cosh", "pow23")])
def test_whole_domain_ulp(op):
    x, e = sweep_err(op)
    assert e.max() <= BOUND[op], (op, x[np.argmax(e)], e.max())


def test_cosh_sinh_beyond_exp_overflow():
    """sinh / cosh for |x| in (709.78, 710.48]: exp(|x|) overflows, so they are (t/2) t with t = exp(|x|/2).  The
    relative error of t counts twice: 2.5 ulp for both (cosh's bound of 2.0 holds up to exp's overflow)."""
    for op in ("sinh", "cosh"):
        x, e = sweep_err(op)
        beyond = np.abs(x) > EXP_O
        assert e[~beyond].max() <= BOUND[op], (op, e[~beyond].max())
        assert beyond.sum() == 0 or e[beyond].max() <= 2.5
    x = np.concatenate([RNG.uniform(EXP_O, SINH_O, 2000), -RNG.uniform(EXP_O, SINH_O, 2000)])
    for op in ("sinh", "cosh"):
        assert ulp_err(H.lib_math("twin", op, x), x, MPF[op]).max() <= 2.5, op


def test_pow23_whole_domain():
    x, e = sweep_err("pow23")
    allowed = pow23_bound(x)
    assert np.all(e <= allowed), (x[np.argmax(e - allowed)], e.max())


def test_atan2_whole_domain():
    a, b = A2
    e = ulp_err(H.lib_math("twin", "atan2", a, b), np.stack([a, b], 1), mp.atan2)
    assert e.max() <= BOUND["atan2"], e.max()


def test_exp_subnormal_results():
    """exp on [-745.13, -708.40): y 2^k rounded once to the subnormal grid, inside exp's bound in ulps of 2^-1074."""
    x = RNG.uniform(EXP_U0, EXP_U1, 3000)
    y = H.lib_math("twin", "exp", x)
    assert np.all(y < DMIN) and np.all(y[x > EXP_U0 + 0.7] > 0)
    assert ulp_err(y, x, mp.exp).max() <= BOUND["exp"]


# ---- argument reduction of sin / cos / tan --------------------------------------------------------------------------
def near_kpio2(k):
    """The doubles nearest k pi/2 (mpmath, 200 bits)."""
    h = mp.pi / 2
    return np.array([float(mp.mpf(int(v)) * h) for v in k])


def reduction_args():
    ks = [np.unique(np.floor(10.0 ** RNG.uniform(d, d + 1, 10000)).astype(np.int64)) for d in range(9)]
    fast = near_kpio2(np.concatenate(ks))
    fast = fast[np.abs(fast) < 2.0 ** 30]
    # Payne-Hanek range: 2^30 ... DBL_MAX, 50 per decade, and the double closest to a multiple of pi/2
    # (6381956970095103 2^797, Muller, "Elementary Functions", table 11.1)
    big = np.array([float(mp.mpf(2) ** 30 * mp.mpf(10) ** e) for e in RNG.uniform(0, 298.9, 15000)])
    big = near_kpio2([int(mp.nint(mp.mpf(float(v)) / (mp.pi / 2))) for v in big])
    worst = float(mp.mpf(6381956970095103) * mp.mpf(2) ** 797)
    return fast, np.concatenate([big, [worst, -worst], -big[:50]])


RED_FAST, RED_BIG = reduction_args()


@pytest.mark.parametrize("op", ["sin", "cos", "tan"])
def test_reduction_near_multiples_of_pio2(op):
    for x, where in ((RED_FAST, "Cody-Waite"), (RED_BIG, "Payne-Hanek")):
        e = ulp_err(H.lib_math("twin", op, x), x, MPF[op])
        assert e.max() <= BOUND[op], (op, where, x[np.argmax(e)], e.max())


# ---- fx: a NaN hyperbolic anomaly reaches the true-anomaly conversion ------------------------------------------------
# States just beyond escape speed (e = 1 + 5.3e-7, 1 + 2.6e-5) for which Newton's method on the hyperbolic Kepler
# equation does not converge in 100 iterations (ssa_newton_hyperbolic returns NaN), so ssa_F_to_nu gets tanh(NaN).
# They come from a search over perturbed near-parabolic states; the C5 stress batch reaches the same branch through
# the sigma points of near-parabolic objects with inflated covariances.
NAN_F_STATES = np.array([
    [-7.3552943989516020e+08, -2.6022586970649910e+08, 2.6712503290555486e+08, -8.8993699365131897e+02,
     -3.1711710100447817e+02, 3.2535387321917523e+02],
    [3.4208936270095474e+08, -3.0543586598201948e+08, 4.0355776813500971e+07, -9.8862650695297668e+02,
     8.8410792779125006e+02, -8.3207380359782675e+01]])
NAN_F_DTS = (20.0, -20.0, 600.0, 6000.0, -86400.0)


def test_fx_nan_anomaly_matches_oracle():
    for dt in NAN_F_DTS:
        o, eo = H.lib_fx("oracle", NAN_F_STATES, dt)
        t, et = H.lib_fx("twin", NAN_F_STATES, dt)
        assert np.isnan(o).all() and np.isnan(t).all(), dt
        assert np.array_equal(eo, et), dt


def c5_statuses(which, dt):
    from test_stress_c5 import _stress_batch
    n = 600
    cat, x, P = _stress_batch(n)
    zn = np.random.RandomState(4).normal(size=(3, n, 3)) * np.array([H.arcsec2rad, H.arcsec2rad, 1e3])
    cfg = H.make_cfg(n, dt=dt)
    st = H.HostState(cat, x, P)
    for s in range(3):
        H.cpu_step(which, cfg, st, H.CEL2TER06AXY, 0x1 | 0x2 | 0x4 | 0x10 | 0x20, z_noise=zn[s])
    return st.status


def test_c5_nan_anomaly_status_matches_oracle():
    """The near-parabolic objects 171, 180 and 188 of the C5 stress batch fail with a NaN predicted mean (and a
    covariance that needs more than 16 inflations): the status is FAILED | LINALG | NAN in the oracle and the twin."""
    for dt in (20.0, 6000.0):
        so, st = c5_statuses("oracle", dt), c5_statuses("twin", dt)
        rows = [171, 188] if dt == 6000.0 else [171, 180, 188]
        assert np.all(so[rows] == 7) and np.array_equal(st[rows], so[rows]), (dt, so[rows], st[rows])


# ---- the device ---------------------------------------------------------------------------------------------------
def gpu_and_twin(op, a, b=None):
    g, t = H.lib_math("gpu", op, a, b), H.lib_math("twin", op, a, b)
    assert H.bits_equal(g, t), (op, np.where(g.view(np.uint64) != t.view(np.uint64))[0])
    return g


@pytest.mark.gpu
@pytest.mark.parametrize("op", UNARY)
def test_gpu_special_values(op):
    """bits_equal ignores the sign of a NaN; numpy_semantics then checks the device's NaN positions and zero signs,
    and the finite results are compared exactly by bits_equal."""
    x = np.array(SPECIAL[op])
    check_special(op, x, gpu_and_twin(op, x))


@pytest.mark.gpu
def test_gpu_special_values_binary():
    a, b = special_binary()
    check_atan2(a, b, gpu_and_twin("atan2", a, b))
    a, b = pymod_args()
    y = gpu_and_twin("pymod", a, b)
    assert H.bits_equal(y, python_mod(a, b))


@pytest.mark.gpu
@pytest.mark.parametrize("op", UNARY)
def test_gpu_whole_domain(op):
    x = np.concatenate([SWEEP[op], RED_FAST, RED_BIG]) if op in ("sin", "cos", "tan") else SWEEP[op]
    gpu_and_twin(op, x)
    if op in ("sinh", "cosh"):
        gpu_and_twin(op, np.linspace(EXP_O, SINH_O, 5000))
    if op == "exp":
        gpu_and_twin(op, np.linspace(EXP_U0, EXP_U1, 5000))


@pytest.mark.gpu
def test_gpu_whole_domain_atan2():
    gpu_and_twin("atan2", *A2)


@pytest.mark.gpu
def test_gpu_fx_nan_anomaly():
    for dt in NAN_F_DTS:
        g, ge = H.lib_fx("gpu", NAN_F_STATES, dt)
        t, te = H.lib_fx("twin", NAN_F_STATES, dt)
        assert H.bits_equal(g, t) and np.array_equal(ge, te) and np.isnan(g).all(), dt
