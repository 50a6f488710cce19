/*
 * idk_cbrtf.h -- the single-precision cube root the BLAS builder's pre-splitting priority uses, on the host and on the device.
 *
 * The reference calls MathF.Cbrt, which on Linux is the C library's cbrtf. glibc's cbrtf is not correctly rounded (it
 * differs from the rounded long-double cube root on about 2.3e8 positive inputs), so neither CUDA's cbrtf (1 ulp) nor a
 * correctly rounded root reproduces it, and a split count that depends on the last bit would flip. This is a restatement
 * of glibc's generic sysdeps/ieee754/flt-32/s_cbrtf.c (Ulrich Drepper, LGPL-2.1-or-later): a quadratic first guess in the
 * mantissa, one Halley step in double, a scale by 2^(e mod 3 / 3) and ldexp by e / 3. It equals glibc 2.39's cbrtf on all
 * 2^32 inputs, so the host mirror and the kernels share it and neither depends on the platform's libm.
 *
 * Build with contraction off (-ffp-contract=off on the host, -fmad=false under nvcc): every operation below is one IEEE
 * operation in the written precision.
 */
#ifndef IDK_CBRTF_H
#define IDK_CBRTF_H

#include <math.h>

#if defined(__CUDACC__)
#define IDK_CBRT_HD __host__ __device__ __forceinline__
#else
#define IDK_CBRT_HD static inline
#endif

IDK_CBRT_HD float idk_cbrtf(float x) {
    /* 2^(k/3) for k = -2 .. 2 */
    const double F[5] = {1.0 / 1.5874010519681994748, 1.0 / 1.2599210498948731648, 1.0, 1.2599210498948731648, 1.5874010519681994748};
    int e;
    const float xm = frexpf(fabsf(x), &e);
    if (!(x != 0.0f && x - x == 0.0f)) return x + x;   /* zero, infinity, NaN */
    const float u = (float)(0.492659620528969547 + (0.697570460207922770 - 0.191502161678719066 * (double)xm) * (double)xm);
    const float t2 = u * u * u;
    const float ym = (float)((double)u * ((double)t2 + 2.0 * (double)xm) / (2.0 * (double)t2 + (double)xm) * F[2 + e % 3]);
    return ldexpf(x > 0.0f ? ym : -ym, e / 3);
}

#undef IDK_CBRT_HD
#endif /* IDK_CBRTF_H */
