// agc_math.h — logf / expf for the RMS AGC recurrence (liquid agc_crcf_execute: g *= expf(-0.5 alpha logf(y2')),
// reference src/agc.c:92-100), written for LATENCY: the recurrence is one serial chain per block of the stream, so what
// counts is the number of DEPENDENT operations per sample, not throughput.
//
// Both functions evaluate in double to a relative error of a few 1e-16 and round once to float, i.e. they return the
// correctly rounded float result except when the exact value lies within ~1e-15 (relative) of a float rounding boundary —
// which is what a good libm returns (checked against long double by tests/native/agc_math_check.cpp, run from
// tests/test_agc_rms_exact.py: plain C++, the same IEEE double operations the GPU executes).  The serial reference of the
// RMS AGC (tests/native/agc_rms_serial.cpp) evaluates the recurrence with these same functions on the CPU.
//
//   logf:  glibc-style table method, 128 intervals over [0.699, 1.398): z = x / 2^k, r = z * invc - 1 (|r| < 0.008, exact
//          for the two intervals around 1 where c = 1), log x = k ln2 + log c + log1p(r), log1p by a degree-7 polynomial
//          in Estrin form: 6 dependent double operations after the table lookup (the Horner evaluation of an atanh series
//          it replaces had 20).
//   expf:  |t| <= 0.125 (t = -alpha/2 * log y2', alpha <= 1e-2: always): degree-10 Taylor polynomial in Estrin form,
//          5 dependent operations instead of 14; agc_exp_small covers 0.125 < |t| <= 0.5 off the fast path.
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define AGC_HD __host__ __device__ __forceinline__
#else
#define AGC_HD static inline
#endif

struct AgcLogEntry { double invc, logc; };
constexpr int AGC_LOG_N = 128;
constexpr uint32_t AGC_LOG_OFF = 0x3f330000u;      // interval 77 starts exactly at 1.0

AGC_HD uint32_t agc_f2u(float f)
{
#if defined(__CUDA_ARCH__)
    return __float_as_uint(f);
#else
    uint32_t u; memcpy(&u, &f, 4); return u;
#endif
}
AGC_HD float agc_u2f(uint32_t u)
{
#if defined(__CUDA_ARCH__)
    return __uint_as_float(u);
#else
    float f; memcpy(&f, &u, 4); return f;
#endif
}
// float -> double for a positive normal float, by integer arithmetic (exact; off the conversion pipe)
AGC_HD double agc_pos_float_to_double(uint32_t bits)
{
    const uint32_t hi = (bits >> 3) + 0x38000000u, lo = bits << 29;
#if defined(__CUDA_ARCH__)
    return __hiloint2double((int)hi, (int)lo);
#else
    const uint64_t u = ((uint64_t)hi << 32) | lo;
    double d; memcpy(&d, &u, 8); return d;
#endif
}

// host: the table (c = interval midpoint; the two intervals adjacent to 1.0 use c = 1 so that log near 1 keeps full
// relative accuracy); logc = -log(invc) for the ROUNDED invc, so the identity log z = log1p(z invc - 1) + logc is exact
static inline void agc_log_table(AgcLogEntry (&tab)[AGC_LOG_N])
{
    for (int i = 0; i < AGC_LOG_N; i++) {
        const uint32_t lo = AGC_LOG_OFF + ((uint32_t)i << 16), hi = lo + (1u << 16);
        float zl, zh;
        memcpy(&zl, &lo, 4); memcpy(&zh, &hi, 4);
        if (i == 76 || i == 77) { tab[i].invc = 1.0; tab[i].logc = 0.0; continue; }
        const long double c = 0.5L * ((long double)zl + (long double)zh);
        tab[i].invc = (double)(1.0L / c);
        tab[i].logc = (double)(-logl((long double)tab[i].invc));
    }
}

// polynomial coefficients, in one table so that the device reads them as constant-bank operands of the DFMAs (64-bit
// immediates would cost two UMOVs each, in program order in front of every dependent step)
#define AGC_COEF_LIST                                                                                              \
    {0.6931471805599453, 1.0 / 3.0, -0.5, 0.2, -0.25, 1.0 / 7.0, -1.0 / 6.0,          /* 0..6   log */              \
     1.0 / 6.0, 0.5, 1.0 / 120.0, 1.0 / 24.0, 1.0 / 5040.0, 1.0 / 720.0,               /* 7..12  exp */              \
     1.0 / 362880.0, 1.0 / 40320.0, 1.0 / 3628800.0, 1.0, -1.0}                        /* 13..17     */
constexpr int AGC_NCOEF = 18;

// log(x) in double for a positive normal float x (caller guarantees x > 1e-6); K = AGC_COEF_LIST.
// Device form: TAB is the table's 32-bit shared-window address (a generic pointer makes the compiler rebuild the window
// base — S2UR + ULEA, in program order in front of the load — in every step of the serial chain).
template <typename TAB>
AGC_HD double agc_log_fast(float x, TAB tab, const double* __restrict__ K)
{
    const uint32_t ix = agc_f2u(x);
    const uint32_t tmp = ix - AGC_LOG_OFF;
    const int i = (int)((tmp >> 16) & (AGC_LOG_N - 1));
    const int k = (int)tmp >> 23;                              // arithmetic shift
    const uint32_t iz = ix - (tmp & 0xff800000u);
    const double z = agc_pos_float_to_double(iz);
    AgcLogEntry e;
#if defined(__CUDA_ARCH__)
    if constexpr (sizeof(TAB) == 4) {
        asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(e.invc), "=d"(e.logc) : "r"((uint32_t)tab + 16u * (uint32_t)i));
    } else
#endif
    {
        e = reinterpret_cast<const AgcLogEntry*>((uintptr_t)tab)[i];
    }
    const double r = fma(z, e.invc, K[17]);
    const double y0 = fma((double)k, K[0], e.logc);
    const double r2 = r * r;
    // log1p(r) = r + r2 (-1/2 + r/3 + r2 (-1/4 + r/5 + r2 (-1/6 + r/7)))
    const double u = fma(r, K[1], K[2]);
    const double v = fma(r, K[3], K[4]);
    const double w = fma(r, K[5], K[6]);
    const double q = fma(r2, w, v);
    const double p = fma(r2, q, u);
    return fma(r2, p, r) + y0;
}

// exp(t) in double, |t| <= 0.125
AGC_HD double agc_exp_tiny(double t, const double* __restrict__ K)
{
    const double t2 = t * t;
    const double a0 = K[16] + t;
    const double a1 = fma(t, K[7], K[8]);
    const double a2 = fma(t, K[9], K[10]);
    const double a3 = fma(t, K[11], K[12]);
    const double a4 = fma(t, K[13], K[14]);
    const double t4 = t2 * t2;
    const double b0 = fma(t2, a1, a0);
    const double b1 = fma(t2, a3, a2);
    const double b2 = fma(t2, K[15], a4);
    const double c1 = fma(t4, b2, b1);
    return fma(t4, c1, b0);
}

// exp(t) in double, |t| <= 0.5: degree-13 Taylor polynomial in Horner form.  Off the fast path: 0.125 < |t| needs
// y2' > e^25 at alpha = 1e-2 (a full-scale burst after a gain held at its 1e6 clamp), so latency does not matter here.
AGC_HD double agc_exp_small(double t)
{
    double p = 1.0 / 6227020800.0;
    p = fma(p, t, 1.0 / 479001600.0); p = fma(p, t, 1.0 / 39916800.0); p = fma(p, t, 1.0 / 3628800.0);
    p = fma(p, t, 1.0 / 362880.0);    p = fma(p, t, 1.0 / 40320.0);    p = fma(p, t, 1.0 / 5040.0);
    p = fma(p, t, 1.0 / 720.0);       p = fma(p, t, 1.0 / 120.0);      p = fma(p, t, 1.0 / 24.0);
    p = fma(p, t, 1.0 / 6.0);         p = fma(p, t, 0.5);              p = fma(p, t, 1.0);
    return fma(p, t, 1.0);
}
