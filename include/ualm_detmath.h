/*
 * ualm_detmath.h -- deterministic sin / cos / atan2 built ONLY from IEEE-754 double +,-,*,/ and
 * floor/fabs, so that a host build (gcc, -ffp-contract=off) and a device build (nvcc, -fmad=false)
 * return bit-identical results.  glibc's and CUDA's libm differ in the last bit, and the optimizer
 * this repo reproduces is chaotic with respect to last-bit differences (DESIGN.md, "Why bit-exact"),
 * so both the CUDA path and the CPU oracle call these instead of libm.
 *
 * Accuracy (pinned in tests/test_detmath.py against numpy/libm): <= 2 ulp for |x| <= 1e5 (sin/cos)
 * and everywhere for atan2.  The polynomial coefficients are the classical double-precision minimax
 * sets for sin/cos on [-pi/4,pi/4] and atan on [0,7/16] with the 4-breakpoint reduction.
 *
 * No FMA may be formed from these expressions: compile with contraction OFF on both sides.
 */
#ifndef UALM_DETMATH_H
#define UALM_DETMATH_H

#include <math.h>

#if defined(__CUDACC__)
#define UALM_HD __host__ __device__ __forceinline__
#else
#define UALM_HD static inline
#endif

/* ---- kernels on |r| <= pi/4 ---- */
UALM_HD double ualm_ksin(double r)
{
    const double S1 = -1.66666666666666324348e-01, S2 = 8.33333333332248946124e-03,
                 S3 = -1.98412698298579493134e-04, S4 = 2.75573137070700676789e-06,
                 S5 = -2.50507602534068634195e-08, S6 = 1.58969099521155010221e-10;
    const double z = r * r;
    const double v = z * r;
    const double p = S2 + z * (S3 + z * (S4 + z * (S5 + z * S6)));
    return r + v * (S1 + z * p);
}

UALM_HD double ualm_kcos(double r)
{
    const double C1 = 4.16666666666666019037e-02, C2 = -1.38888888888741095749e-03,
                 C3 = 2.48015872894767294178e-05, C4 = -2.75573143513906633035e-07,
                 C5 = 2.08757232129817482790e-09, C6 = -1.13596475577881948265e-11;
    const double z = r * r;
    const double p = z * (C1 + z * (C2 + z * (C3 + z * (C4 + z * (C5 + z * C6)))));
    const double hz = 0.5 * z;
    const double w = 1.0 - hz;
    return w + (((1.0 - w) - hz) + z * p);
}

/* sin and cos of x; Cody-Waite reduction by pi/2 in three parts (valid for |x| up to ~1e5 rad,
 * far beyond the |yaw| < ~50 this path produces). */
UALM_HD void ualm_sincos(double x, double *s, double *c)
{
    const double INV_PIO2 = 6.36619772367581382433e-01;
    const double P1 = 1.57079632673412561417e+00;  /* first 33 bits of pi/2 */
    const double P2 = 6.07710050630396597660e-11;  /* next 33 bits */
    const double P3 = 2.02226624871116645580e-21;  /* next 33 bits */
    const double P4 = 8.47842766036889956997e-32;  /* tail */
    const double fk = floor(x * INV_PIO2 + 0.5);
    double r = x - fk * P1;
    r = r - fk * P2;
    r = r - fk * P3;
    r = r - fk * P4;
    const double ks = ualm_ksin(r), kc = ualm_kcos(r);
    /* quadrant = fk mod 4, computed in floating point (exact for |fk| < 2^51) */
    const double q = fk - 4.0 * floor(fk * 0.25);
    if (q == 0.0) { *s = ks; *c = kc; }
    else if (q == 1.0) { *s = kc; *c = -ks; }
    else if (q == 2.0) { *s = -ks; *c = -kc; }
    else { *s = -kc; *c = ks; }
}

UALM_HD double ualm_sin(double x) { double s, c; ualm_sincos(x, &s, &c); return s; }
UALM_HD double ualm_cos(double x) { double s, c; ualm_sincos(x, &s, &c); return c; }

/* atan(x) for x >= 0 */
UALM_HD double ualm_atan_pos(double x)
{
    const double aT0 = 3.33333333333329318027e-01, aT1 = -1.99999999998764832476e-01,
                 aT2 = 1.42857142725034663711e-01, aT3 = -1.11111104054623557880e-01,
                 aT4 = 9.09088713343650656196e-02, aT5 = -7.69187620504482999495e-02,
                 aT6 = 6.66107313738753120669e-02, aT7 = -5.83357013379057348645e-02,
                 aT8 = 4.97687799461593236017e-02, aT9 = -3.65315727442169155270e-02,
                 aT10 = 1.62858201153657823623e-02;
    double hi, lo;
    int reduced = 1;
    if (x > 1.0e18) return 1.57079632679489655800e+00; /* pi/2 */
    if (x < 0.4375) { reduced = 0; hi = 0.0; lo = 0.0; }
    else if (x < 0.6875) { x = (2.0 * x - 1.0) / (2.0 + x); hi = 4.63647609000806093515e-01; lo = 2.26987774529616870924e-17; }
    else if (x < 1.1875) { x = (x - 1.0) / (x + 1.0); hi = 7.85398163397448278999e-01; lo = 3.06161699786838301793e-17; }
    else if (x < 2.4375) { x = (x - 1.5) / (1.0 + 1.5 * x); hi = 9.82793723247329054082e-01; lo = 1.39033110312309984516e-17; }
    else { x = -1.0 / x; hi = 1.57079632679489655800e+00; lo = 6.12323399573676603587e-17; }
    const double z = x * x;
    const double w = z * z;
    const double s1 = z * (aT0 + w * (aT2 + w * (aT4 + w * (aT6 + w * (aT8 + w * aT10)))));
    const double s2 = w * (aT1 + w * (aT3 + w * (aT5 + w * (aT7 + w * aT9))));
    if (!reduced) return x - x * (s1 + s2);
    return hi - ((x * (s1 + s2) - lo) - x);
}

UALM_HD double ualm_atan2(double y, double x)
{
    const double PI = 3.14159265358979311600e+00, PIO2 = 1.57079632679489655800e+00;
    if (x != x || y != y) return x + y;
    if (y == 0.0) {
        if (x > 0.0 || (x == 0.0 && !signbit(x))) return y;   /* +-0 */
        return signbit(y) ? -PI : PI;
    }
    if (x == 0.0) return y > 0.0 ? PIO2 : -PIO2;
    const double ay = fabs(y), ax = fabs(x);
    const double a = ualm_atan_pos(ay / ax);
    double r;
    if (x > 0.0) r = a;
    else r = PI - (a - 1.2246467991473531772e-16);
    return y > 0.0 ? r : -r;
}

/* tan and acos for the front-end (turning radius, motion primitives, the Dubins words RLR / LRL), from the kernels above with
 * one more IEEE operation: tan = sin / cos of one reduction, acos(x) = atan2(sqrt((1 - x)(1 + x)), x), which keeps its accuracy as
 * |x| -> 1 where 1 - x*x would cancel.  NaN outside [-1, 1] like libm. */
UALM_HD double ualm_tan(double x) { double s, c; ualm_sincos(x, &s, &c); return s / c; }
UALM_HD double ualm_acos(double x) { return ualm_atan2(sqrt((1.0 - x) * (1.0 + x)), x); }

#endif
