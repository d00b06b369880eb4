// ssa_math.h — fp64 elementary functions with ONE definition for device and host.
//
// Why this exists: the UKF of the reference runs with alpha=1e-4 (envs/__init__.py:27), so the
// unscented-transform weights are +-2e8 and every ulp of the propagated sigma points is amplified
// ~1e8 times in the predicted mean.  To be able to state "GPU == CPU bit for bit" the kernels must
// not depend on libdevice vs glibc differences.  Every function below is built only from IEEE-754
// correctly rounded primitives (+ - * / sqrt fma, exact fmod/floor/rint, integer bit tricks), with
// every fused multiply-add written explicitly.  Translation units that include this header are
// compiled with contraction OFF (nvcc -fmad=false, gcc -ffp-contract=off), so the sequence of
// rounded operations is identical on sm_100a and on the host "twin" build used by the tests.
//
// Accuracy target: <= ~2 ulp on the argument ranges the path uses (measured against mpmath in
// tests/test_math_accuracy.py).  Polynomial coefficients are the classic fdlibm minimax sets.
//
// Domain and special values (tests/test_math_domain.py, against numpy and mpmath): every function accepts every double
// and keeps its ulp bound over its whole finite domain, with three stated exceptions: sinh / cosh on
// (709.78, 710.48] (2.5 ulp: exp(|x|/2) squared), pow23 (1.5 + 1.5 |2/3 log x| ulp) and the subnormal results of exp
// (counted in ulps of 2^-1074).  NaN in gives NaN out; results overflow and underflow where the true values do; odd
// functions keep the sign of zero; atan2 follows C99 Annex F for signed zeros and infinities.  pow23 is NaN for every
// x < 0, -inf included.  The inlined variants ssa_sincos_i and ssa_atan2_i are restricted to the ranges their hot
// callers use (see there).
//
// No CUDA libdevice transcendental is called anywhere on the hot path.
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define SSA_HD __host__ __device__ __forceinline__
#define SSA_HD_NOINLINE __host__ __device__ __noinline__
#else
#define SSA_HD static inline __attribute__((always_inline))
#define SSA_HD_NOINLINE static inline
#endif

#define SSA_PI      3.14159265358979311600e+00  /* RN(pi), == numpy.pi */
#define SSA_TWOPI   6.28318530717958623200e+00  /* 2*RN(pi), == 2*numpy.pi */
#define SSA_PIO2    1.57079632679489655800e+00


// ---------------------------------------------------------------------------------------------
// constant table
// ---------------------------------------------------------------------------------------------
// sm_100a has no 64-bit immediates: a double literal costs two UMOV/IMAD.MOV instructions every time it
// is used (measured: ~30 % of the instructions of the first propagation kernel).  Constants of the hot
// functions therefore live in one __constant__ table and are fetched two at a time by LDCU.128; the host
// build reads the same values from a static array, so both sides see identical bits.
#define SSA_KLIST(X)                                                                                   \
  X(INVPIO2, 6.36619772367581382433e-01) X(RMAGIC, 6755399441055744.0)                                 \
  X(PIO2_A, 1.57079632679489655800e+00) X(PIO2_B, 6.12323399573676603587e-17)                          \
  X(PIO2_C, -1.49738490485916983800e-33) X(HALF, 0.5)                                                  \
  X(S6, 1.58969099521155010221e-10) X(S5, -2.50507602534068634195e-08)                                 \
  X(S4, 2.75573137070700676789e-06) X(S3, -1.98412698298579493134e-04)                                 \
  X(S2, 8.33333333332248946124e-03) X(S1, -1.66666666666666324348e-01)                                 \
  X(C6, -1.13596475577881948265e-11) X(C5, 2.08757232129817482790e-09)                                 \
  X(C4, -2.75573143513906633035e-07) X(C3, 2.48015872894767294178e-05)                                 \
  X(C2, -1.38888888888741095749e-03) X(C1, 4.16666666666666019037e-02)                                 \
  X(AT10, 1.62858201153657823623e-02) X(AT8, 4.97687799461593236017e-02)                               \
  X(AT6, 6.66107313738753120669e-02) X(AT4, 9.09088713343650656196e-02)                                \
  X(AT2, 1.42857142725034663711e-01) X(AT0, 3.33333333333329318027e-01)                                \
  X(AT9, -3.65315727442169155270e-02) X(AT7, -5.83357013379057348645e-02)                              \
  X(AT5, -7.69187620504482999495e-02) X(AT3, -1.11111104054623557880e-01)                              \
  X(AT1, -1.99999999998764832476e-01) X(PI_LO, 1.2246467991473531772e-16)                              \
  X(ATHI0, 4.63647609000806093515e-01) X(ATLO0, 2.26987774529616870924e-17)                            \
  X(ATHI1, 7.85398163397448278999e-01) X(ATLO1, 3.06161699786838301793e-17)                            \
  X(ATHI2, 9.82793723247329054082e-01) X(ATLO2, 1.39033110312309984516e-17)                            \
  X(PI, 3.14159265358979311600e+00) X(TWOPI, 6.28318530717958623200e+00)                               \
  X(PS5, 3.47933107596021167570e-05) X(PS4, 7.91534994289814532176e-04)                                \
  X(PS3, -4.00555345006794114027e-02) X(PS2, 2.01212532134862925881e-01)                               \
  X(PS1, -3.25565818622400915405e-01) X(PS0, 1.66666666666666657415e-01)                               \
  X(QS4, 7.70381505559019352791e-02) X(QS3, -6.88283971605453293030e-01)                               \
  X(QS2, 2.02094576023350569471e+00) X(QS1, -2.40339491173441421878e+00)                               \
  X(PIO4_HI, 7.85398163397448278999e-01) X(ONE, 1.0)                                                   \
  X(MU, 398600441800000.0) X(MU_INV, 1.0 / 398600441800000.0)                                          \
  X(TOL8, 1e-8) X(TOL12, 1e-12) X(HYP101, 1.0 + 1e-2) X(NEWTON_TOL, 1.48e-08) X(P2_52, 4503599627370496.0) X(DELTA99, 1.0 - 1e-2)                        \
  X(INV_TWOPI, 1.0 / 6.28318530717958623200e+00)

enum {
#define SSA_X(n, v) SSA_K_##n,
  SSA_KLIST(SSA_X)
#undef SSA_X
  SSA_K_COUNT
};
#if defined(__CUDACC__)
static __constant__ double ssa_kdev[SSA_K_COUNT] = {
#define SSA_X(n, v) v,
    SSA_KLIST(SSA_X)
#undef SSA_X
};
#endif
static const double ssa_khost[SSA_K_COUNT] = {
#define SSA_X(n, v) v,
    SSA_KLIST(SSA_X)
#undef SSA_X
};
#if defined(__CUDA_ARCH__)
#define SSA_C(n) ssa_kdev[SSA_K_##n]
#else
#define SSA_C(n) ssa_khost[SSA_K_##n]
#endif

// ---------------------------------------------------------------------------------------------
// primitives
// ---------------------------------------------------------------------------------------------
SSA_HD double ssa_fma(double a, double b, double c) {
#if defined(__CUDA_ARCH__)
  return __fma_rn(a, b, c);
#else
  return __builtin_fma(a, b, c);
#endif
}
SSA_HD double ssa_mul(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __dmul_rn(a, b);
#else
  return a * b;
#endif
}
SSA_HD double ssa_add(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __dadd_rn(a, b);
#else
  return a + b;
#endif
}
// Division and square root are real function calls on the device: nvcc expands each `/` and sqrt into
// ~30 inline instructions plus an out-of-line slow path, and the propagation kernel has dozens of them
// on its hot path — inlined, the kernel's hot footprint (measured 1.7-6.7 k instructions) overflows the
// instruction cache and `no_instruction` becomes the top stall reason.  One shared copy keeps the hot
// code resident.  Both are IEEE-754 correctly rounded, so the host's `/` and sqrt return the same bits.
#if defined(__CUDA_ARCH__)
__device__ __noinline__ double ssa_div_dev(double a, double b) { return __ddiv_rn(a, b); }
__device__ __noinline__ double ssa_sqrt_dev(double a) { return __dsqrt_rn(a); }
#endif
// *_i: inlined variants for the (small) fast path of the propagation kernel, where the call overhead
// (argument/result moves, CALL/RET) measured ~25 % of the issued instructions.
SSA_HD double ssa_sqrt_i(double a) {
#if defined(__CUDA_ARCH__)
  return __dsqrt_rn(a);
#else
  return __builtin_sqrt(a);
#endif
}
SSA_HD double ssa_div_i(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __ddiv_rn(a, b);
#else
  return a / b;
#endif
}
SSA_HD double ssa_sqrt(double a) {
#if defined(__CUDA_ARCH__)
  return ssa_sqrt_dev(a);
#else
  return __builtin_sqrt(a);
#endif
}
SSA_HD double ssa_div(double a, double b) {
#if defined(__CUDA_ARCH__)
  return ssa_div_dev(a, b);
#else
  return a / b;
#endif
}
SSA_HD int32_t ssa_hi32(double x) {
#if defined(__CUDA_ARCH__)
  return __double2hiint(x);
#else
  uint64_t u; memcpy(&u, &x, 8); return (int32_t)(u >> 32);
#endif
}
SSA_HD int32_t ssa_lo32(double x) {
#if defined(__CUDA_ARCH__)
  return __double2loint(x);
#else
  uint64_t u; memcpy(&u, &x, 8); return (int32_t)(u & 0xffffffffu);
#endif
}
SSA_HD double ssa_from_hilo(int32_t hi, int32_t lo) {
#if defined(__CUDA_ARCH__)
  return __hiloint2double(hi, lo);
#else
  uint64_t u = ((uint64_t)(uint32_t)hi << 32) | (uint32_t)lo; double x; memcpy(&x, &u, 8); return x;
#endif
}
SSA_HD double ssa_fabs(double x) { return fabs(x); }
SSA_HD int ssa_isnan(double x) { return x != x; }
SSA_HD int ssa_signbit(double x) { return ssa_hi32(x) < 0; }
SSA_HD double ssa_nan() { return ssa_from_hilo(0x7ff80000, 0); }
SSA_HD double ssa_copysign(double mag, double sgn) {
  int32_t h = (ssa_hi32(mag) & 0x7fffffff) | (ssa_hi32(sgn) & (int32_t)0x80000000);
  return ssa_from_hilo(h, ssa_lo32(mag));
}

// Exact fmod(a, b) for b > 0 without the library's bit-serial loop: q = trunc(a/b) is right or off by
// one (a/b is rounded once), r = fma(-q, b, a) is exact because the true remainder is representable,
// and one conditional add repairs the off-by-one.  Falls back to the (exact) library fmod when
// |a/b| >= 2^52 or anything is non-finite.  Checked against numpy.fmod in tests/test_math_accuracy.py.
// Same with a pre-computed reciprocal of the divisor (binv ~ 1/b): q may now be off by one in either direction
// more often, which the repair step handles identically, so the result is still the exact fmod.
SSA_HD double ssa_fmod_pos_inv(double a, double b, double binv) {
  const double q0 = ssa_mul(a, binv);
  if (!(ssa_fabs(q0) < SSA_C(P2_52))) return fmod(a, b);
  const double q = trunc(q0);
  double r = ssa_fma(-q, b, a);
  if (a >= 0.0) {
    if (r < 0.0) r = ssa_add(r, b);
    else if (r >= b) r = r - b;
  } else {
    if (r > 0.0) r = r - b;
    else if (r <= -b) r = ssa_add(r, b);
  }
  return r;
}
SSA_HD double ssa_fmod_pos(double a, double b) {
  const double q0 = ssa_div(a, b);
  if (!(ssa_fabs(q0) < SSA_C(P2_52))) return fmod(a, b);
  const double q = trunc(q0);
  double r = ssa_fma(-q, b, a);
  if (a >= 0.0) {
    if (r < 0.0) r = ssa_add(r, b);
    else if (r >= b) r = r - b;
  } else {
    if (r > 0.0) r = r - b;
    else if (r <= -b) r = ssa_add(r, b);
  }
  return r;
}
// Python float modulo for a positive divisor (result in [0, b)), as numba lowers `a % b`
// (farnocchia.py:283,286,293,306,309,311,954,967): fmod, then + b when the remainder is negative.
SSA_HD double ssa_pymod(double a, double b) {
  double m = ssa_fmod_pos(a, b);
  if (m != 0.0 && m < 0.0) m = ssa_add(m, b);
  return m;
}

// ---------------------------------------------------------------------------------------------
// sin / cos
// ---------------------------------------------------------------------------------------------
// 3-term Cody-Waite reduction with FMA: the first step is exact for |x| < ~1e9, the next two add
// the next 106 bits of pi/2.
#define SSA_INVPIO2 6.36619772367581382433e-01
#define SSA_PIO2_A  1.57079632679489655800e+00
#define SSA_PIO2_B  6.12323399573676603587e-17
#define SSA_PIO2_C  -1.49738490485916983800e-33  /* pi/2 - A - B */
#define SSA_RMAGIC  6755399441055744.0            /* 1.5 * 2^52 */

typedef struct { double s, c; } ssa_sc;
// sin and cos of x = r + q pi/2, |r| <= ~pi/4: the fdlibm kernels, then the quadrant.
SSA_HD ssa_sc ssa_sincos_kern(double r, int32_t q) {
  double z = ssa_mul(r, r);
  // sin kernel: r + r^3 (S1 + z S2 + ... )
  double ps = ssa_fma(z, SSA_C(S6), SSA_C(S5));
  ps = ssa_fma(z, ps, SSA_C(S4));
  ps = ssa_fma(z, ps, SSA_C(S3));
  ps = ssa_fma(z, ps, SSA_C(S2));
  ps = ssa_fma(z, ps, SSA_C(S1));
  double sr = ssa_fma(ssa_mul(r, z), ps, r);
  // cos kernel: 1 - z/2 + z^2 (C1 + z C2 + ...)
  double pc = ssa_fma(z, SSA_C(C6), SSA_C(C5));
  pc = ssa_fma(z, pc, SSA_C(C4));
  pc = ssa_fma(z, pc, SSA_C(C3));
  pc = ssa_fma(z, pc, SSA_C(C2));
  pc = ssa_fma(z, pc, SSA_C(C1));
  double hz = ssa_mul(SSA_C(HALF), z);
  double w = SSA_C(ONE) - hz;
  double cr = w + (((SSA_C(ONE) - w) - hz) + ssa_mul(ssa_mul(z, z), pc));
  // quadrant
  double s_ = (q & 1) ? cr : sr;
  double c_ = (q & 1) ? sr : cr;
  if (q & 2) s_ = -s_;
  if ((q + 1) & 2) c_ = -c_;
  ssa_sc out;
  out.s = s_;
  out.c = c_;
  return out;
}

// 2/pi in binary, 32 bits a word, most significant first, after one word of zeros: table bit j is the bit of weight
// 2^(31 - j), so that the reduction below can read windows that start before the binary point.
#define SSA_TWO_OVER_PI_BITS(X)                                                                                      \
  X(0x00000000) X(0xa2f9836e) X(0x4e441529) X(0xfc2757d1) X(0xf534ddc0) X(0xdb629599) X(0x3c439041) X(0xfe5163ab)    \
  X(0xdebbc561) X(0xb7246e3a) X(0x424dd2e0) X(0x06492eea) X(0x09d1921c) X(0xfe1deb1c) X(0xb129a73e) X(0xe88235f5)    \
  X(0x2ebb4484) X(0xe99c7026) X(0xb45f7e41) X(0x3991d639) X(0x835339f4) X(0x9c845f8b) X(0xbdf9283b) X(0x1ff897ff)    \
  X(0xde05980f) X(0xef2f118b) X(0x5a0a6d1f) X(0x6d367ecf) X(0x27cb09b7) X(0x4f463f66) X(0x9e5fea2d) X(0x7527bac7)    \
  X(0xebe5f17b) X(0x3d0739f7) X(0x8a5292ea) X(0x6bfb5fb1) X(0x1f8d5d08) X(0x56033046) X(0xfc7b6bab) X(0xf0cfbc20)    \
  X(0x9af4361d)
#define SSA_W32(v) v##u,
#if defined(__CUDACC__)
static __constant__ uint32_t ssa_2opi_dev[] = {SSA_TWO_OVER_PI_BITS(SSA_W32)};
#endif
static const uint32_t ssa_2opi_host[] = {SSA_TWO_OVER_PI_BITS(SSA_W32)};
#undef SSA_W32
SSA_HD uint64_t ssa_2opi_bits64(int j) {  // table bits j .. j+63
#if defined(__CUDA_ARCH__)
  const uint32_t* T = ssa_2opi_dev;
#else
  const uint32_t* T = ssa_2opi_host;
#endif
  const int w = j >> 5, s = j & 31;
  const uint64_t a = ((uint64_t)T[w] << 32) | T[w + 1];
  const uint64_t b = ((uint64_t)T[w + 2] << 32) | T[w + 3];
  return s ? ((a << s) | (b >> (64 - s))) : a;
}
SSA_HD uint64_t ssa_umulhi64(uint64_t a, uint64_t b) {
#if defined(__CUDA_ARCH__)
  return __umul64hi(a, b);
#else
  return (uint64_t)(((unsigned __int128)a * b) >> 64);
#endif
}
SSA_HD int ssa_clz64(uint64_t v) {  // v != 0
#if defined(__CUDA_ARCH__)
  return __clzll((long long)v);
#else
  return __builtin_clzll(v);
#endif
}

// Arguments outside [2^-27, 2^30) in magnitude.  Tiny ones: sin x = x (this keeps the sign of -0), cos x = 1; the
// polynomial path returns the same bits except for -0.  Non-finite ones: NaN.  Large ones: Payne-Hanek reduction in
// integer arithmetic.  With x = M 2^E (M a 53-bit integer), the bits of 2/pi of weight 2^(1-E) and above multiply M
// into multiples of 4 and drop out; a 192-bit window from there gives M 2/pi 2^E mod 4 = q + f to 2^-137, and the
// closest double to a multiple of pi/2 keeps |f| above 2^-62.  f becomes a 106-bit double pair, r = f pi/2 one double.
SSA_HD_NOINLINE ssa_sc ssa_sincos_edge(double x) {
  const int32_t hx = ssa_hi32(x) & 0x7fffffff;
  ssa_sc out;
  if (hx < 0x3e400000) {
    out.s = x;
    out.c = 1.0;
    return out;
  }
  if (hx >= 0x7ff00000) {
    out.s = x - x;
    out.c = out.s;
    return out;
  }
  const int E = (hx >> 20) - 1075;  // >= -22
  const uint64_t M = ((uint64_t)(hx & 0x000fffff) << 32 | (uint32_t)ssa_lo32(x)) | ((uint64_t)1 << 52);
  const int j = E - 1 + 31;
  const uint64_t w0 = ssa_2opi_bits64(j), w1 = ssa_2opi_bits64(j + 64), w2 = ssa_2opi_bits64(j + 128);
  // P = M W mod 2^192, W = w0 w1 w2
  const uint64_t p2 = M * w2;
  const uint64_t h2 = ssa_umulhi64(M, w2);
  const uint64_t l1 = M * w1;
  const uint64_t p1 = l1 + h2;
  const uint64_t p0 = M * w0 + ssa_umulhi64(M, w1) + (uint64_t)(p1 < l1);
  int32_t q = (int32_t)(p0 >> 62);
  uint64_t fh = (p0 << 2) | (p1 >> 62), fl = (p1 << 2) | (p2 >> 62);  // f in [0, 1), 128 bits
  const bool neg = (fh >> 63) != 0;  // f >= 1/2: take f - 1 and the next quadrant
  if (neg) {
    q += 1;
    fl = ~fl + 1;
    fh = ~fh + (uint64_t)(fl == 0);
  }
  int sh = 0;
  if (fh == 0) {
    fh = fl;
    fl = 0;
    sh = 64;
  }
  const int lz = ssa_clz64(fh);
  if (lz) {
    fh = (fh << lz) | (fl >> (64 - lz));
    fl <<= lz;
  }
  sh += lz;
  // |f| = fh 2^-(64 + sh) + fl 2^-(128 + sh): a = the top 53 bits, b = the next 53
  const double a = ssa_mul((double)(int64_t)(fh >> 11), ssa_from_hilo((int32_t)((1023 - 53 - sh) << 20), 0));
  const double b = ssa_mul((double)(int64_t)(((fh & 0x7ff) << 42) | (fl >> 22)),
                           ssa_from_hilo((int32_t)((1023 - 106 - sh) << 20), 0));
  const double rh = ssa_mul(a, SSA_C(PIO2_A));
  const double rl = ssa_fma(a, SSA_C(PIO2_B), ssa_fma(b, SSA_C(PIO2_A), ssa_fma(a, SSA_C(PIO2_A), -rh)));
  double r = ssa_add(rh, rl);
  if (neg) r = -r;
  if (ssa_signbit(x)) {
    r = -r;
    q = -q;
  }
  return ssa_sincos_kern(r, q);
}

// Cody-Waite reduction, inlined into the propagation kernels.  Valid for 2^-27 <= |x| < 2^30: there the first step is
// exact, and the pi/2 tail A + B + C keeps sin / cos within their bounds at the doubles nearest every multiple of pi/2
// (tests/test_math_domain.py).  Its two callers stay inside that range without a test: ssa_fx's Newton iterates of
// Kepler's equation (e < 0.99, started in [-pi, pi]) and the azimuth / elevation of ssa_aer2uvw_t.  Outside it
// (beyond 2^51 pi/2 the quotient n is not even an integer) use ssa_sincos_v.
SSA_HD ssa_sc ssa_sincos_i(double x) {
  double t = ssa_fma(x, SSA_C(INVPIO2), SSA_C(RMAGIC));
  int32_t q = ssa_lo32(t);
  double n = t - SSA_C(RMAGIC);
  double r = ssa_fma(-n, SSA_C(PIO2_A), x);
  r = ssa_fma(-n, SSA_C(PIO2_B), r);
  r = ssa_fma(-n, SSA_C(PIO2_C), r);
  return ssa_sincos_kern(r, q);
}
// Every double: one unsigned compare of the high word sends |x| outside [2^-27, 2^30) to ssa_sincos_edge.  A real
// (non-inlined) device function for the big kernels: the fused step kernel calls it from ~60 sites and would
// otherwise exceed the instruction cache several times over.  Results are returned by value so they travel in
// registers.
SSA_HD_NOINLINE ssa_sc ssa_sincos_v(double x) {
  if ((uint32_t)(ssa_hi32(x) & 0x7fffffff) - 0x3e400000u >= 0x41d00000u - 0x3e400000u) return ssa_sincos_edge(x);
  return ssa_sincos_i(x);
}
SSA_HD void ssa_sincos(double x, double* sn, double* cs) {
  const ssa_sc r = ssa_sincos_v(x);
  *sn = r.s;
  *cs = r.c;
}
SSA_HD double ssa_sin(double x) { return ssa_sincos_v(x).s; }
SSA_HD double ssa_cos(double x) { return ssa_sincos_v(x).c; }
// tan(x) = sin/cos (one division; ~2 ulp).  Used only as tan(angle/2) in the anomaly conversions
// (farnocchia.py:432,467,503,539).
SSA_HD double ssa_tan(double x) { double s, c; ssa_sincos(x, &s, &c); return ssa_div(s, c); }

// ---------------------------------------------------------------------------------------------
// atan2 / atan  — one division: the fdlibm interval reduction (2t-1)/(2+t) etc. is applied to the
// pair (|y|,|x|) directly, so t = |y|/|x| is never formed.
// ---------------------------------------------------------------------------------------------
SSA_HD_NOINLINE double ssa_atan2_big(double y, double x);
// FULL: every argument pair.  |y| >= 2^1020 (where the interval tests below overflow) and inf go to ssa_atan2_big, and
// atan2(+-0, NaN) is NaN.
template <bool FULL>
SSA_HD double ssa_atan2_t(double y, double x) {
  const double ax = ssa_fabs(x), ay = ssa_fabs(y);
  const double ay16 = ssa_mul(16.0, ay);
  double num, den, hi, lo;
  if (ay16 < ssa_mul(7.0, ax)) {
    num = ay; den = ax; hi = 0.0; lo = 0.0;
  } else if (ay16 < ssa_mul(11.0, ax)) {
    num = ssa_fma(2.0, ay, -ax); den = ssa_fma(2.0, ax, ay);
    hi = SSA_C(ATHI0); lo = SSA_C(ATLO0);
  } else if (ay16 < ssa_mul(19.0, ax)) {
    num = ay - ax; den = ax + ay;
    hi = SSA_C(ATHI1); lo = SSA_C(ATLO1);
  } else if (ay16 < ssa_mul(39.0, ax)) {
    num = ssa_fma(-1.5, ax, ay); den = ssa_fma(1.5, ay, ax);
    hi = SSA_C(ATHI2); lo = SSA_C(ATLO2);
  } else {
    if (FULL && ssa_hi32(ay16) >= 0x7ff00000) return ssa_atan2_big(y, x);
    num = -ax; den = ay;
    hi = SSA_C(PIO2_A); lo = SSA_C(PIO2_B);
  }
  double z;
  if (den == 0.0) {
    z = FULL ? num - num : 0.0;  // atan2(+-0, +-0): fdlibm returns +-0 / +-pi through the quadrant logic below
  } else {
    const double t = ssa_div_i(num, den);
    const double t2 = ssa_mul(t, t);
    const double t4 = ssa_mul(t2, t2);
    double s1 = ssa_fma(t4, SSA_C(AT10), SSA_C(AT8));
    s1 = ssa_fma(t4, s1, SSA_C(AT6));
    s1 = ssa_fma(t4, s1, SSA_C(AT4));
    s1 = ssa_fma(t4, s1, SSA_C(AT2));
    s1 = ssa_fma(t4, s1, SSA_C(AT0));
    s1 = ssa_mul(t2, s1);
    double s2 = ssa_fma(t4, SSA_C(AT9), SSA_C(AT7));
    s2 = ssa_fma(t4, s2, SSA_C(AT5));
    s2 = ssa_fma(t4, s2, SSA_C(AT3));
    s2 = ssa_fma(t4, s2, SSA_C(AT1));
    s2 = ssa_mul(t4, s2);
    // hi - ((t*(s1+s2) - lo) - t)
    z = hi - ((ssa_mul(t, s1 + s2) - lo) - t);
  }
  if (ssa_signbit(x)) z = SSA_C(PI) - (z - SSA_C(PI_LO));
  return ssa_signbit(y) ? -z : z;
}
// Both arguments scaled by 2^-6 keep the interval tests finite.  The scaling is exact for y (|y| >= 2^1020) and for
// every x that does not make the result pi/2 to the last bit anyway.  Equal magnitudes, inf included, give the
// octant bisectors: atan2(+-inf, +-inf) = +-pi/4, +-3pi/4.
SSA_HD_NOINLINE double ssa_atan2_big(double y, double x) {
  if (ssa_fabs(x) == ssa_fabs(y)) return ssa_atan2_t<false>(ssa_copysign(1.0, y), ssa_copysign(1.0, x));
  return ssa_atan2_t<false>(ssa_mul(y, 0.015625), ssa_mul(x, 0.015625));
}
// Inlined variant for the hot kernels, without the two FULL cases: their arguments stay far below 2^1020 (ssa_fx:
// e sin E0 and e cos E0 with e < 0.99; the azimuths of ssa_meas.h: coordinates in metres, 1e20 for a failed filter).
SSA_HD double ssa_atan2_i(double y, double x) { return ssa_atan2_t<false>(y, x); }
SSA_HD_NOINLINE double ssa_atan2(double y, double x) { return ssa_atan2_t<true>(y, x); }
SSA_HD double ssa_atan(double x) { return ssa_atan2(x, 1.0); }

// ---------------------------------------------------------------------------------------------
// asin / acos — fdlibm rational kernel R(t) = t*P(t)/Q(t)
// ---------------------------------------------------------------------------------------------
// INL selects the inlined division / square root (ssa_div_i / ssa_sqrt_i) for the kernels that are bound by issue
// slots rather than code size (k_hx); both variants are IEEE operations and return the same bits.
template <bool INL> SSA_HD double ssa_div_t(double a, double b) { return INL ? ssa_div_i(a, b) : ssa_div(a, b); }
template <bool INL> SSA_HD double ssa_sqrt_t(double a) { return INL ? ssa_sqrt_i(a) : ssa_sqrt(a); }
template <bool INL>
SSA_HD double ssa_asin_R_t(double t) {
  double p = ssa_fma(t, SSA_C(PS5), SSA_C(PS4));
  p = ssa_fma(t, p, SSA_C(PS3));
  p = ssa_fma(t, p, SSA_C(PS2));
  p = ssa_fma(t, p, SSA_C(PS1));
  p = ssa_fma(t, p, SSA_C(PS0));
  p = ssa_mul(t, p);
  double q = ssa_fma(t, SSA_C(QS4), SSA_C(QS3));
  q = ssa_fma(t, q, SSA_C(QS2));
  q = ssa_fma(t, q, SSA_C(QS1));
  q = ssa_fma(t, q, SSA_C(ONE));
  return ssa_div_t<INL>(p, q);
}
template <bool INL>
SSA_HD double ssa_asin_t(double x) {
  const double ax = ssa_fabs(x);
  double res;
  if (ax < SSA_C(HALF)) {
    res = ssa_fma(ax, ssa_asin_R_t<INL>(ssa_mul(ax, ax)), ax);
  } else if (ax <= SSA_C(ONE)) {
    // asin(x) = pi/2 - 2 asin(sqrt((1-x)/2)); c = (t - s*s)/(2s) is the FMA residual of the square root,
    // folded in so that pi/2 - 2(s + c)(1 + r) does not lose the low part of s.
    const double t = ssa_mul(SSA_C(HALF), SSA_C(ONE) - ax);
    const double s = ssa_sqrt_t<INL>(t);
    const double r = ssa_asin_R_t<INL>(t);
    const double c = (s == 0.0) ? 0.0 : ssa_div_t<INL>(ssa_fma(-s, s, t), ssa_add(s, s));
    const double p = ssa_fma(2.0, ssa_mul(s, r), -(SSA_C(PIO2_B) - ssa_mul(2.0, c)));
    const double q = SSA_C(PIO4_HI) - ssa_mul(2.0, s);
    res = SSA_C(PIO4_HI) - (p - q);
  } else {
    res = ssa_nan();
  }
  return ssa_signbit(x) ? -res : res;
}
SSA_HD double ssa_asin_R(double t) {
  double p = ssa_fma(t, SSA_C(PS5), SSA_C(PS4));
  p = ssa_fma(t, p, SSA_C(PS3));
  p = ssa_fma(t, p, SSA_C(PS2));
  p = ssa_fma(t, p, SSA_C(PS1));
  p = ssa_fma(t, p, SSA_C(PS0));
  p = ssa_mul(t, p);
  double q = ssa_fma(t, SSA_C(QS4), SSA_C(QS3));
  q = ssa_fma(t, q, SSA_C(QS2));
  q = ssa_fma(t, q, SSA_C(QS1));
  q = ssa_fma(t, q, SSA_C(ONE));
  return ssa_div(p, q);
}
SSA_HD_NOINLINE double ssa_asin(double x) { return ssa_asin_t<false>(x); }
SSA_HD_NOINLINE double ssa_acos(double x) {
  const double ax = ssa_fabs(x);
  if (ax < SSA_C(HALF)) {
    const double r = ssa_asin_R(ssa_mul(x, x));
    return SSA_C(PIO2_A) - (x - (SSA_C(PIO2_B) - ssa_mul(x, r)));
  } else if (ax <= SSA_C(ONE)) {
    const double t = ssa_mul(SSA_C(HALF), SSA_C(ONE) - ax);
    const double s = ssa_sqrt(t);
    const double r = ssa_asin_R(t);
    const double c = (s == 0.0) ? 0.0 : ssa_div(ssa_fma(-s, s, t), ssa_add(s, s));
    if (x > 0.0) {
      return ssa_mul(2.0, s + ssa_fma(s, r, c));  // 2*(s + (s*r + c))
    }
    const double w = ssa_fma(s, r, c) - SSA_C(PIO2_B);
    return SSA_C(PI) - ssa_mul(2.0, s + w);
  }
  return ssa_nan();
}

// ---------------------------------------------------------------------------------------------
// exp / log and the hyperbolic family (only reached in the e >= 1 regimes of farnocchia.py)
// ---------------------------------------------------------------------------------------------
SSA_HD double ssa_scalbn_small(double x, int k) {  // x * 2^k for |k| < 1000, x normal result
  return ssa_mul(x, ssa_from_hilo((int32_t)((k + 1023) << 20), 0));
}
SSA_HD_NOINLINE double ssa_exp(double x) {
  if (ssa_isnan(x)) return x;
  // fdlibm's thresholds: exp(x) > DBL_MAX above o, < 2^-1075 (rounds to 0) below u
  if (x > 7.09782712893383973096e+02) return ssa_from_hilo(0x7ff00000, 0);
  if (x < -7.45133219101941108420e+02) return 0.0;
  const double t = ssa_fma(x, 1.44269504088896338700e+00, SSA_RMAGIC);
  const int32_t k = ssa_lo32(t);
  const double n = t - SSA_RMAGIC;
  const double hi = ssa_fma(-n, 6.93147180369123816490e-01, x);
  const double lo = ssa_mul(n, 1.90821492927058770002e-10);
  const double r = hi - lo;
  const double z = ssa_mul(r, r);
  double c = ssa_fma(z, 4.13813679705723846039e-08, -1.65339022054652515390e-06);
  c = ssa_fma(z, c, 6.61375632143793436117e-05);
  c = ssa_fma(z, c, -2.77777777770155933842e-03);
  c = ssa_fma(z, c, 1.66666666666666019037e-01);
  c = ssa_fma(-z, c, r);  // r - z*P(z)
  const double y = 1.0 - ((lo - ssa_div(ssa_mul(r, c), 2.0 - c)) - hi);
  // scale by 2^k, k in [-1075, 1024], in two steps: both factors are normal, so a subnormal result is y 2^k rounded once
  const int k1 = k / 2, k2 = k - k1;
  return ssa_mul(ssa_scalbn_small(y, k1), ssa_from_hilo((int32_t)((k2 + 1023) << 20), 0));
}
SSA_HD_NOINLINE double ssa_log(double x) {
  if (ssa_isnan(x) || x < 0.0) return ssa_nan();
  if (x == 0.0) return -ssa_from_hilo(0x7ff00000, 0);
  int32_t hx = ssa_hi32(x), lx = ssa_lo32(x);
  if (hx >= 0x7ff00000) return x;
  int k = 0;
  if (hx < 0x00100000) {  // subnormal
    x = ssa_mul(x, 18014398509481984.0);
    k -= 54; hx = ssa_hi32(x); lx = ssa_lo32(x);
  }
  k += (hx >> 20) - 1023;
  hx &= 0x000fffff;
  const int32_t i = (hx + 0x95f64) & 0x100000;
  x = ssa_from_hilo(hx | (i ^ 0x3ff00000), lx);  // normalise x or x/2
  k += (i >> 20);
  const double f = x - 1.0;
  const double dk = (double)k;
  const double s = ssa_div(f, 2.0 + f);
  const double z = ssa_mul(s, s);
  const double w = ssa_mul(z, z);
  double t1 = ssa_fma(w, 1.531383769920937332e-01, 2.222219843214978396e-01);
  t1 = ssa_fma(w, t1, 3.999999999940941908e-01);
  t1 = ssa_mul(w, t1);
  double t2 = ssa_fma(w, 1.479819860511658591e-01, 1.818357216161805012e-01);
  t2 = ssa_fma(w, t2, 2.857142874366239149e-01);
  t2 = ssa_fma(w, t2, 6.666666666666735130e-01);
  t2 = ssa_mul(z, t2);
  const double R = t2 + t1;
  const double hfsq = ssa_mul(0.5, ssa_mul(f, f));
  // k*ln2_hi - ((hfsq - (s*(hfsq+R) + k*ln2_lo)) - f)
  return ssa_fma(dk, 6.93147180369123816490e-01,
                 -((hfsq - ssa_fma(s, hfsq + R, ssa_mul(dk, 1.90821492927058770002e-10))) - f));
}
// log1p-quality log(1+y) for the small-argument inverse hyperbolics: uses the exact-error trick.
SSA_HD double ssa_log1p(double y) {
  const double u = 1.0 + y;
  if (u == 1.0) return y;
  if (u == ssa_from_hilo(0x7ff00000, 0)) return u;  // log1p(inf) = inf
  // log(u) * y/(u-1) corrects the rounding of 1+y (Kahan/HP-15C trick)
  return ssa_mul(ssa_log(u), ssa_div(y, u - 1.0));
}
SSA_HD double ssa_expm1(double x) {
  // Kahan's trick: expm1(x) = (e^x - 1) * x / log(e^x), accurate to a few ulp.
  const double u = ssa_exp(x);
  if (u == 1.0) return x;
  const double um1 = u - 1.0;
  if (um1 == -1.0) return -1.0;
  if (ssa_fabs(x) > 30.0) return um1;
  return ssa_mul(um1, ssa_div(x, ssa_log(u)));
}
SSA_HD double ssa_sinh(double x) {
  const double ax = ssa_fabs(x);
  double r;
  if (ax < 22.0) {
    const double t = ssa_expm1(ax);
    r = ssa_mul(0.5, t + ssa_div(t, t + 1.0));
  } else if (ax > 7.09782712893383973096e+02) {  // exp(ax) overflows, sinh(ax) up to 710.4758600739439
    const double t = ssa_exp(ssa_mul(0.5, ax));
    r = ssa_mul(ssa_mul(0.5, t), t);
  } else {
    r = ssa_mul(0.5, ssa_exp(ax));
  }
  return ssa_signbit(x) ? -r : r;
}
SSA_HD double ssa_cosh(double x) {
  const double ax = ssa_fabs(x);
  if (ax > 7.09782712893383973096e+02) {  // as ssa_sinh
    const double t = ssa_exp(ssa_mul(0.5, ax));
    return ssa_mul(ssa_mul(0.5, t), t);
  }
  const double t = ssa_exp(ax);
  return ssa_fma(0.5, t, ssa_div(0.5, t));
}
SSA_HD double ssa_tanh(double x) {
  const double ax = ssa_fabs(x);
  double r;
  if (ax < 22.0) {
    const double t = ssa_expm1(ssa_mul(2.0, ax));
    r = ssa_div(t, t + 2.0);
  } else if (ax >= 22.0) {
    r = 1.0;
  } else {
    return x;  // NaN
  }
  return ssa_signbit(x) ? -r : r;
}
SSA_HD double ssa_atanh(double x) {
  const double ax = ssa_fabs(x);
  // 0.5 * log1p(2a/(1-a))
  const double r = ssa_mul(0.5, ssa_log1p(ssa_div(ssa_add(ax, ax), 1.0 - ax)));
  return ssa_signbit(x) ? -r : r;
}
SSA_HD double ssa_asinh(double x) {
  const double ax = ssa_fabs(x);
  double r;
  if (ax > 1e8) {
    r = ssa_log(ax) + 6.93147180559945286227e-01;
  } else {
    const double x2 = ssa_mul(ax, ax);
    r = ssa_log1p(ax + ssa_div(x2, 1.0 + ssa_sqrt(1.0 + x2)));
  }
  return ssa_signbit(x) ? -r : r;
}
SSA_HD double ssa_acosh(double x) {
  if (!(x >= 1.0)) return ssa_nan();
  if (x > 268435456.0) return ssa_log(x) + 6.93147180559945286227e-01;  // 2^28: t*t would overflow for large x
  const double t = x - 1.0;
  return ssa_log1p(t + ssa_sqrt(ssa_fma(t, t, ssa_mul(2.0, t))));
}
// x^(2/3) for x > 0 (Barker's equation, farnocchia.py:650)
SSA_HD double ssa_pow23(double x) {
  return ssa_exp(ssa_mul(6.66666666666666629659e-01, ssa_log(x)));
}
