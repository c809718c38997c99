/*
 * asinh.h -- ccb_asinh: one asinh for the host library (hostio.c, plain C) and the kernels (CUDA), with the same bits on
 * both.  The arcsinh(x / cofactor) transform of cytometry intensities feeds epsilon and argmin tests, so where the
 * transform runs must not change a cell's value: numpy's arcsinh, glibc's asinh and CUDA's asinh are three different
 * implementations that disagree in the last bits, and numpy's choice depends on the CPU features it detects.
 *
 * The algorithms are fdlibm 5.3's (s_asinh.c, which calls e_log.c and s_log1p.c), restated for the arguments asinh passes
 * to them: log of a finite x >= 2, log1p of a finite x >= 2^-28.  One change: for 2^-28 <= |x| <= 2 the rounding error of
 * log1p's argument is carried as a first-order correction (see ccb_asinh); fdlibm as written is up to 2 ulp off there.  Only + - * / and sqrt (which IEEE 754 requires to be
 * correctly rounded) and bit operations on the representation are used, and no libm or CUDA math function besides
 * sqrt.  Both sides must be compiled without contraction of a * b + c: the device library is built with -fmad=false,
 * libccb_hostio.so with -ffp-contract=off.  Then every operation rounds once, in the same order, on both.
 *
 * Specials: +-0 -> +-0, +-inf -> +-inf, NaN -> the same NaN; asinh(-x) == -asinh(x) bit for bit (the magnitude is computed
 * from |x| and x * x only).  |x| < 2^-28, subnormals included, returns x (asinh(x) = x - x^3 / 6 + ..., the cubic term is
 * below half an ulp).  Accuracy: within 1 ulp of the correctly rounded value (tests/test_arcsinh.py checks it against
 * mpmath).
 *
 * The restatement keeps fdlibm's notice:
 *
 * ====================================================
 * Copyright (C) 1993 by Sun Microsystems, Inc. All rights reserved.
 *
 * Developed at SunPro, a Sun Microsystems, Inc. business.
 * Permission to use, copy, modify, and distribute this
 * software is freely granted, provided that this notice
 * is preserved.
 * ====================================================
 */
#ifndef CCB_ASINH_H
#define CCB_ASINH_H

#include <stdint.h>

#ifdef __CUDACC__
#define CCB_ASINH_FN static __host__ __device__ __forceinline__
#else
#include <math.h>
#include <string.h>
#define CCB_ASINH_FN static inline
#endif

CCB_ASINH_FN uint64_t ccb_dbits(double x) {
#ifdef __CUDA_ARCH__
    return (uint64_t)__double_as_longlong(x);
#else
    uint64_t u;
    memcpy(&u, &x, sizeof u);
    return u;
#endif
}

CCB_ASINH_FN double ccb_dfrom(uint64_t u) {
#ifdef __CUDA_ARCH__
    return __longlong_as_double((long long)u);
#else
    double x;
    memcpy(&x, &u, sizeof x);
    return x;
#endif
}

CCB_ASINH_FN int32_t ccb_dhi(double x) { return (int32_t)(ccb_dbits(x) >> 32); } /* fdlibm's __HI(x) */

CCB_ASINH_FN double ccb_dset_hi(double x, int32_t hi) { /* __HI(x) = hi */
    return ccb_dfrom(((uint64_t)(uint32_t)hi << 32) | (ccb_dbits(x) & 0xffffffffu));
}

CCB_ASINH_FN double ccb_dsqrt(double x) {
#ifdef __CUDA_ARCH__
    return __dsqrt_rn(x);
#else
    return sqrt(x);
#endif
}

/* e_log.c for a finite x >= 2: the zero, negative, subnormal and non-finite branches cannot be reached, and k >= 1 */
CCB_ASINH_FN double ccb_log_ge2(double x) {
    const double ln2_hi = 6.93147180369123816490e-01, /* 3fe62e42 fee00000 */
        ln2_lo = 1.90821492927058770002e-10,          /* 3dea39ef 35793c76 */
        Lg1 = 6.666666666666735130e-01,               /* 3FE55555 55555593 */
        Lg2 = 3.999999999940941908e-01,               /* 3FD99999 9997FA04 */
        Lg3 = 2.857142874366239149e-01,               /* 3FD24924 94229359 */
        Lg4 = 2.222219843214978396e-01,               /* 3FCC71C5 1D8E78AF */
        Lg5 = 1.818357216161805012e-01,               /* 3FC74664 96CB03DE */
        Lg6 = 1.531383769920937332e-01,               /* 3FC39A09 D078C69F */
        Lg7 = 1.479819860511658591e-01;               /* 3FC2F112 DF3E5244 */
    int32_t hx = ccb_dhi(x);
    int32_t k = (hx >> 20) - 1023;
    hx &= 0x000fffff;
    int32_t i = (hx + 0x95f64) & 0x100000;
    x = ccb_dset_hi(x, hx | (i ^ 0x3ff00000)); /* normalize x or x/2 */
    k += i >> 20;
    const double f = x - 1.0, dk = (double)k;
    if ((0x000fffff & (2 + hx)) < 3) { /* |f| < 2**-20 */
        if (f == 0.0) return dk * ln2_hi + dk * ln2_lo;
        const double R = f * f * (0.5 - 0.33333333333333333 * f);
        return dk * ln2_hi - ((R - dk * ln2_lo) - f);
    }
    const double s = f / (2.0 + f), z = s * s, w = z * z;
    i = hx - 0x6147a;
    const int32_t j = 0x6b851 - hx;
    const double t1 = w * (Lg2 + w * (Lg4 + w * Lg6));
    const double t2 = z * (Lg1 + w * (Lg3 + w * (Lg5 + w * Lg7)));
    i |= j;
    const double R = t2 + t1;
    if (i > 0) {
        const double hfsq = 0.5 * f * f;
        return dk * ln2_hi - ((hfsq - (s * (hfsq + R) + dk * ln2_lo)) - f);
    }
    return dk * ln2_hi - ((s * (f - R) - dk * ln2_lo) - f);
}

/* s_log1p.c for a finite x >= 2^-28: the x <= -1, |x| < 2^-29, negative and non-finite branches cannot be reached */
CCB_ASINH_FN double ccb_log1p_pos(double x) {
    const double ln2_hi = 6.93147180369123816490e-01, /* 3fe62e42 fee00000 */
        ln2_lo = 1.90821492927058770002e-10,          /* 3dea39ef 35793c76 */
        Lp1 = 6.666666666666735130e-01,               /* 3FE55555 55555593 */
        Lp2 = 3.999999999940941908e-01,               /* 3FD99999 9997FA04 */
        Lp3 = 2.857142874366239149e-01,               /* 3FD24924 94229359 */
        Lp4 = 2.222219843214978396e-01,               /* 3FCC71C5 1D8E78AF */
        Lp5 = 1.818357216161805012e-01,               /* 3FC74664 96CB03DE */
        Lp6 = 1.531383769920937332e-01,               /* 3FC39A09 D078C69F */
        Lp7 = 1.479819860511658591e-01;               /* 3FC2F112 DF3E5244 */
    const int32_t hx = ccb_dhi(x);
    int32_t k, hu;
    double c = 0.0, f;
    if (hx < 0x3FDA827A) { /* x < 0.41422 */
        k = 0, f = x, hu = 1;
    } else {
        double u = 1.0 + x;
        hu = ccb_dhi(u);
        k = (hu >> 20) - 1023;
        c = k > 0 ? 1.0 - (u - x) : x - (u - 1.0); /* correction term */
        c /= u;
        hu &= 0x000fffff;
        if (hu < 0x6a09e) {
            u = ccb_dset_hi(u, hu | 0x3ff00000); /* normalize u */
        } else {
            k += 1;
            u = ccb_dset_hi(u, hu | 0x3fe00000); /* normalize u/2 */
            hu = (0x00100000 - hu) >> 2;
        }
        f = u - 1.0;
    }
    const double hfsq = 0.5 * f * f;
    if (hu == 0) { /* |f| < 2**-20 (only after the normalisation above, so k >= 1) */
        if (f == 0.0) {
            c += k * ln2_lo;
            return k * ln2_hi + c;
        }
        const double R = hfsq * (1.0 - 0.66666666666666666 * f);
        return k * ln2_hi - ((R - (k * ln2_lo + c)) - f);
    }
    const double s = f / (2.0 + f), z = s * s;
    const double R = z * (Lp1 + z * (Lp2 + z * (Lp3 + z * (Lp4 + z * (Lp5 + z * (Lp6 + z * Lp7))))));
    if (k == 0) return f - (hfsq - s * (hfsq + R));
    return k * ln2_hi - ((hfsq - (s * (hfsq + R) + (k * ln2_lo + c))) - f);
}

/* s_asinh.c */
CCB_ASINH_FN double ccb_asinh(double x) {
    const double ln2 = 6.93147180559945286227e-01; /* 0x3FE62E42, 0xFEFA39EF */
    const uint64_t bits = ccb_dbits(x);
    const int32_t hx = (int32_t)(bits >> 32), ix = hx & 0x7fffffff;
    if (ix >= 0x7ff00000) return x; /* inf or NaN (fdlibm returns x + x; x keeps a NaN's bits on every platform) */
    if (ix < 0x3e300000) return x;  /* |x| < 2**-28 */
    const double t = ccb_dfrom(bits & 0x7fffffffffffffffull);
    double w;
    if (ix > 0x41b00000) { /* |x| > 2**28 */
        w = ccb_log_ge2(t) + ln2;
    } else if (ix > 0x40000000) { /* 2**28 > |x| > 2.0 */
        w = ccb_log_ge2(2.0 * t + 1.0 / (ccb_dsqrt(x * x + 1.0) + t));
    } else { /* 2.0 > |x| > 2**-28 */
        // fdlibm: log1p(t + q), whose argument's rounding alone costs up to 0.6 ulp of the result (2 ulp in all near
        // |x| = 0.52).  The rounding error of t + q is exact here (Fast2Sum: q < t) and enters to first order,
        // log1p(a + e) = log1p(a) + e / (1 + a), which keeps every result within 1 ulp of the correctly rounded one.
        const double t2 = x * x, q = t2 / (1.0 + ccb_dsqrt(1.0 + t2)), a = t + q;
        w = ccb_log1p_pos(a) + ((t - a) + q) / (1.0 + a);
    }
    return hx > 0 ? w : -w;
}

#endif
