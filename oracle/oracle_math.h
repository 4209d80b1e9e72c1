/*
 * oracle/oracle_math.h -- TEST INFRASTRUCTURE (CPU oracle), not product code.
 *
 * "Platform" arithmetic of the reference shaders, frozen.
 *
 * The reference (apbodnar/FSPT) leaves sin/cos/atan/asin/pow/min/max/normalize
 * to whatever GLSL ES 3.00 implementation runs the shaders.  Nothing in the
 * reference pins them, so the oracle pins them itself, as spec "FSPT-DM2":
 *
 *   - every f32 operation is a single IEEE-754 binary32 round-to-nearest-even
 *     operation, no contraction (compile with -ffp-contract=off, no fast-math);
 *   - transcendental built-ins are evaluated in binary32 by the fixed operation
 *     sequences below (+ - * / sqrt rint and single-rounded fmaf), i.e. what a GPU
 *     does natively (DM1, the first version, used binary64: 46 % of the shading
 *     kernel's instructions, and FP64 is vestigial on some Blackwell parts);
 *   - min/max are IEEE-754-2019 minimumNumber/maximumNumber: a NaN operand
 *     loses, -0 < +0 (what GPU FMNMX does; GLSL leaves both cases undefined);
 *   - vector built-ins follow the formulas printed in the GLSL ES 3.00 spec
 *     section 8 (normalize = x/length(x), reflect, refract, mix, clamp, fract).
 *
 * The CUDA product implements the same spec independently in
 * fspt_b200/csrc/dm_math.cuh; tests/ compare the two bit for bit.
 */
#ifndef FSPT_ORACLE_MATH_H
#define FSPT_ORACLE_MATH_H

#include <math.h>
#include <stdint.h>
#include <string.h>

namespace om {

/* ---- scalar helpers --------------------------------------------------- */
/* min/max are IEEE 754-2019 minimumNumber/maximumNumber, what sm_100a's FMNMX computes (measured over every pair of
 * tests/test_gpu_dm_exhaustive.py's edge set): a NaN operand loses to a number, and -0 orders below +0 whichever
 * operand it is, so min(+0, -0) = -0, max(-0, +0) = +0 and clamp(-0, 0, hi) = +0. */
static inline float fminN(float a, float b) {
  if (a != a) return b;
  if (b != b) return a;
  if (a == b) return signbit(a) ? a : b; /* equal: the zero with the sign bit, if either has it */
  return b < a ? b : a;
}
static inline float fmaxN(float a, float b) {
  if (a != a) return b;
  if (b != b) return a;
  if (a == b) return signbit(a) ? b : a;
  return a < b ? b : a;
}
static inline float clampf(float x, float lo, float hi) { return fminN(fmaxN(x, lo), hi); }
static inline float fractf(float x) { return x - floorf(x); }
static inline float mixf(float x, float y, float a) { return x * (1.0f - a) + y * a; }

/* ---- FSPT-DM2 transcendental kernels ------------------------------------------------------------
 * All binary32.  fmaf() is a single-rounded fused multiply-add (x86 FMA3 / glibc fmaf; GPU FFMA.RN via
 * __fmaf_rn); every other operation is a separately rounded IEEE operation.  The operation sequences below ARE
 * the specification; the CUDA side (fspt_b200/csrc/dm_math.cuh) restates them with explicit intrinsics.
 * Accuracy against float64 libm, maxima over every f32 input of each range (tools/dm_accuracy.py, DESIGN.md section 2;
 * checked at the worst arguments by tests/test_oracle_cpu.py): sin/cos <= 1.554 ulp for |x| <= 64, absolute error
 * <= 1.085e-7 (sin) / 1.020e-7 (cos) up to |x| = 1e7 (the sin-hash RNG range); asin <= 3.671 ulp; exp2 <= 1.136 ulp on
 * [-126, 127]; log2 <= 3.010 ulp for finite x > 0; pow(x, 0.454545) within 2.321e-5 of an 8-bit step on [0, 1];
 * atan2 <= 2.901 ulp (sampled). */
static inline float dm_fma(float a, float b, float c) { return __builtin_fmaf(a, b, c); }

static const float DM_TWO_OVER_PI = 0x1.45f306p-1f;
static const float DM_PIO2_1 = 0x1.921fb6p+0f;   /* pi/2 rounded to f32            */
static const float DM_PIO2_2 = -0x1.777a5cp-25f; /* pi/2 - P1 rounded to f32       */
static const float DM_PIO2_3 = -0x1.ee59dap-50f; /* pi/2 - P1 - P2 rounded to f32  */
static const float DM_PI = 0x1.921fb6p+1f;
static const float DM_PIO2 = 0x1.921fb6p+0f;
static const float DM_PIO4 = 0x1.921fb6p-1f;
static const float DM_LN2 = 0x1.62e430p-1f;
static const float DM_LOG2E = 0x1.715476p+0f;

/* r = x - k*pi/2 with a three-term Cody-Waite reduction; the products k*P are exact inside the FMAs */
static inline float dm_reduce(float x, int* q) {
  if (!(fabsf(x) <= 1.0e9f)) { *q = 0; return 0.0f; } /* NaN / inf / huge: defined as angle 0 */
  float k = __builtin_rintf(x * DM_TWO_OVER_PI);
  float r = dm_fma(-k, DM_PIO2_1, x);
  r = dm_fma(-k, DM_PIO2_2, r);
  r = dm_fma(-k, DM_PIO2_3, r);
  /* for |x| > ~1e5 the f32 product x*2/pi can miss the nearest integer by one: fold the residue once more */
  float k2 = __builtin_rintf(r * DM_TWO_OVER_PI);
  r = dm_fma(-k2, DM_PIO2_1, r);
  r = dm_fma(-k2, DM_PIO2_2, r);
  *q = ((int)k + (int)k2) & 3;
  return r;
}
/* sin(r) = r + r z (S0 + S1 z + S2 z^2 + S3 z^3), z = r^2, |r| <= pi/4 (least-squares fit at Chebyshev nodes) */
static inline float dm_ksin(float r) {
  float z = r * r;
  float p = dm_fma(2.7234684694121825e-06f, z, -0.00019839966262225062f);
  p = dm_fma(p, z, 0.008333331905305386f);
  p = dm_fma(p, z, -0.1666666716337204f);
  return dm_fma(r * z, p, r);
}
/* cos(r) = 1 - z/2 + z^2 (C0 + C1 z + C2 z^2) */
static inline float dm_kcos(float r) {
  float z = r * r;
  float p = dm_fma(2.453538400004618e-05f, z, -0.001388824312016368f);
  p = dm_fma(p, z, 0.0416666641831398f);
  return dm_fma(z * z, p, dm_fma(-0.5f, z, 1.0f));
}
static inline float dm_sin(float x) {
  int q;
  float r = dm_reduce(x, &q);
  float a = dm_ksin(r), b = dm_kcos(r);
  float s = (q & 1) ? b : a;
  return (q & 2) ? -s : s;
}
static inline float dm_cos(float x) {
  int q;
  float r = dm_reduce(x, &q);
  float a = dm_ksin(r), b = dm_kcos(r);
  float s = (q & 1) ? a : b;
  return (q == 1 || q == 2) ? -s : s;
}
/* atan on [0,1]: one reduction about tan(pi/8), then a + a z (A0 + A1 z + ... + A4 z^4) */
static inline float dm_atan01(float a) {
  float base = 0.0f;
  if (a > 0.4142135679721832f) {
    a = (a - 1.0f) / (a + 1.0f);
    base = DM_PIO4;
  }
  float z = a * a;
  float p = dm_fma(-0.06418270617723465f, z, 0.10733865201473236f);
  p = dm_fma(p, z, -0.14263083040714264f);
  p = dm_fma(p, z, 0.19999517500400543f);
  p = dm_fma(p, z, -0.3333333134651184f);
  return base + dm_fma(a * z, p, a);
}
static inline float dm_atan2(float y, float x) {
  float ax = fabsf(x), ay = fabsf(y);
  float hi = ax > ay ? ax : ay;
  float lo = ax > ay ? ay : ax;
  if (!(hi > 0.0f)) return 0.0f; /* atan(0,0) and NaN inputs: defined as 0 */
  float r = dm_atan01(lo / hi);
  if (ay > ax) r = DM_PIO2 - r;
  if (x < 0.0f) r = DM_PI - r;
  if (y < 0.0f) r = -r;
  return r;
}
static inline float dm_asin(float x) {
  if (x > 1.0f) x = 1.0f; /* |x| may exceed 1 by an ulp after normalize() */
  if (x < -1.0f) x = -1.0f;
  return dm_atan2(x, sqrtf((1.0f - x) * (1.0f + x)));
}
/* 2^x: n = rint(x), f = x - n, 2^f = 1 + f ln2 + f^2 (E0 + E1 f + ... + E4 f^4), scaled by 2^n in two exact steps */
static inline float dm_exp2(float x) {
  if (x != x) return x;
  if (x > 130.0f) x = 130.0f;
  if (x < -160.0f) x = -160.0f;
  float n = __builtin_rintf(x);
  float f = x - n;
  float p = dm_fma(0.0001545316627016291f, f, 0.00133813067805022f);
  p = dm_fma(p, f, 0.009618083015084267f);
  p = dm_fma(p, f, 0.055503811687231064f);
  p = dm_fma(p, f, 0.24022650718688965f);
  float r = dm_fma(f * f, p, dm_fma(f, DM_LN2, 1.0f));
  int ni = (int)n;
  int n1 = ni / 2, n2 = ni - n1;
  uint32_t b1 = (uint32_t)(n1 + 127) << 23, b2 = (uint32_t)(n2 + 127) << 23;
  float s1, s2;
  memcpy(&s1, &b1, 4);
  memcpy(&s2, &b2, 4);
  return (r * s1) * s2;
}
/* log2(x), x > 0: x = m 2^e, m in (sqrt(.5), sqrt(2)], ln m = 2s + s z (L0 + L1 z + L2 z^2 + L3 z^3), s = (m-1)/(m+1) */
static inline float dm_log2(float x) {
  int e = 0;
  if (x < 1.17549435e-38f) { x = x * 16777216.0f; e = -24; } /* subnormal */
  uint32_t b;
  memcpy(&b, &x, 4);
  e += (int)((b >> 23) & 0xff) - 127;
  b = (b & 0x007fffffu) | 0x3f800000u;
  float m;
  memcpy(&m, &b, 4);
  if (m > 1.4142135381698608f) { m = m * 0.5f; e += 1; }
  float s = (m - 1.0f) / (m + 1.0f);
  float z = s * s;
  float p = dm_fma(0.233596533536911f, z, 0.2855019271373749f);
  p = dm_fma(p, z, 0.4000011682510376f);
  p = dm_fma(p, z, 0.6666666865348816f);
  float lnm = dm_fma(s * z, p, 2.0f * s);
  return dm_fma(lnm, DM_LOG2E, (float)e);
}
/* pow(x,y) = exp2(y*log2(x)) (GLSL ES 3.00 8.2); x <= 0 or NaN -> 0 (GLSL: undefined).  log2(2) is exactly 1. */
static inline float dm_pow(float x, float y) {
  if (!(x > 0.0f)) return 0.0f;
  if (x > 3.0e38f) return x;
  return dm_exp2(y * dm_log2(x));
}

/* ---- vec types ---------------------------------------------------------- */
struct v2 { float x, y; };
struct v3 { float x, y, z; };
struct v4 { float x, y, z, w; };

static inline v3 mk3(float x, float y, float z) { v3 r = {x, y, z}; return r; }
static inline v3 add(v3 a, v3 b) { return mk3(a.x + b.x, a.y + b.y, a.z + b.z); }
static inline v3 sub(v3 a, v3 b) { return mk3(a.x - b.x, a.y - b.y, a.z - b.z); }
static inline v3 mul(v3 a, v3 b) { return mk3(a.x * b.x, a.y * b.y, a.z * b.z); }
static inline v3 mul(v3 a, float s) { return mk3(a.x * s, a.y * s, a.z * s); }
static inline v3 mul(float s, v3 a) { return mk3(s * a.x, s * a.y, s * a.z); }
static inline v3 div(v3 a, float s) { return mk3(a.x / s, a.y / s, a.z / s); }
static inline v3 neg(v3 a) { return mk3(-a.x, -a.y, -a.z); }
static inline float dot(v3 a, v3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
static inline v3 cross(v3 x, v3 y) { /* GLSL ES 3.00 8.4 */
  return mk3(x.y * y.z - y.y * x.z, x.z * y.x - y.z * x.x, x.x * y.y - y.x * x.y);
}
static inline float length(v3 a) { return sqrtf(dot(a, a)); }
static inline v3 normalize(v3 a) { return div(a, length(a)); }
static inline v3 reflect(v3 I, v3 N) { return sub(I, mul(2.0f * dot(N, I), N)); }
static inline v3 refract(v3 I, v3 N, float eta) {
  float d = dot(N, I);
  float k = 1.0f - eta * eta * (1.0f - d * d);
  if (k < 0.0f) return mk3(0.0f, 0.0f, 0.0f);
  return sub(mul(eta, I), mul(eta * d + sqrtf(k), N));
}
static inline v3 mix3(v3 x, v3 y, float a) { return mk3(mixf(x.x, y.x, a), mixf(x.y, y.y, a), mixf(x.z, y.z, a)); }
static inline v3 clamp3(v3 a, float lo, float hi) { return mk3(clampf(a.x, lo, hi), clampf(a.y, lo, hi), clampf(a.z, lo, hi)); }

}  // namespace om
#endif
