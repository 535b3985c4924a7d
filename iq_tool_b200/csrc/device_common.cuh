// device_common.cuh — device helpers shared by kernels.cu and fused_front.cu
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

#include "../../include/iqgpu.h"
#include "kernels.hpp"

namespace iqgpu {

// =============================================================================================
// raw sample loaders: reference src/sample_convert.c:127-211 (convert_block_to_cf32)
//   (x * 2^-k) * gain  ==  x * (2^-k * gain) bit for bit: the power-of-two factor is exact, so
//   both forms round once.  32-bit formats go through double like the reference (:174-196).
// =============================================================================================
template <int FMT> struct Fmt;
template <> struct Fmt<IQGPU_FMT_CS16>    { static constexpr int bytes = 4; };
template <> struct Fmt<IQGPU_FMT_SC16Q11> { static constexpr int bytes = 4; };
template <> struct Fmt<IQGPU_FMT_CU16>    { static constexpr int bytes = 4; };
template <> struct Fmt<IQGPU_FMT_CS8>     { static constexpr int bytes = 2; };
template <> struct Fmt<IQGPU_FMT_CU8>     { static constexpr int bytes = 2; };
template <> struct Fmt<IQGPU_FMT_CS24>    { static constexpr int bytes = 6; };
template <> struct Fmt<IQGPU_FMT_CS32>    { static constexpr int bytes = 8; };
template <> struct Fmt<IQGPU_FMT_CU32>    { static constexpr int bytes = 8; };
template <> struct Fmt<IQGPU_FMT_CF32>    { static constexpr int bytes = 8; };

template <int FMT>
__device__ __forceinline__ float in_scale(float gain)
{
    if (FMT == IQGPU_FMT_CS16 || FMT == IQGPU_FMT_CU16) return gain * (1.0f / 32768.0f);
    if (FMT == IQGPU_FMT_SC16Q11) return gain * (1.0f / 2048.0f);
    if (FMT == IQGPU_FMT_CS8 || FMT == IQGPU_FMT_CU8) return gain * (1.0f / 128.0f);
    if (FMT == IQGPU_FMT_CS24) return gain * (1.0f / 8388608.0f);
    return gain;
}

// one frame -> cf32 (sc = in_scale<FMT>(gain))
template <int FMT>
__device__ __forceinline__ float2 load_frame(const void* __restrict__ raw, size_t i, float sc, float gain)
{
    float2 r;
    if (FMT == IQGPU_FMT_CS16 || FMT == IQGPU_FMT_SC16Q11) {
        const short2 v = __ldg(reinterpret_cast<const short2*>(raw) + i);
        r.x = __fmul_rn((float)v.x, sc); r.y = __fmul_rn((float)v.y, sc);
    } else if (FMT == IQGPU_FMT_CU16) {
        const ushort2 v = __ldg(reinterpret_cast<const ushort2*>(raw) + i);
        r.x = __fmul_rn((float)v.x - 32767.5f, sc); r.y = __fmul_rn((float)v.y - 32767.5f, sc);
    } else if (FMT == IQGPU_FMT_CS8) {
        const char2 v = __ldg(reinterpret_cast<const char2*>(raw) + i);
        r.x = __fmul_rn((float)v.x, sc); r.y = __fmul_rn((float)v.y, sc);
    } else if (FMT == IQGPU_FMT_CU8) {
        const uchar2 v = __ldg(reinterpret_cast<const uchar2*>(raw) + i);
        r.x = __fmul_rn((float)v.x - 127.5f, sc); r.y = __fmul_rn((float)v.y - 127.5f, sc);
    } else if (FMT == IQGPU_FMT_CS24) {
        const unsigned char* p = reinterpret_cast<const unsigned char*>(raw) + i * 6;
        int a = (int)(((unsigned)p[0] << 8) | ((unsigned)p[1] << 16) | ((unsigned)p[2] << 24)) >> 8;
        int b = (int)(((unsigned)p[3] << 8) | ((unsigned)p[4] << 16) | ((unsigned)p[5] << 24)) >> 8;
        r.x = __fmul_rn((float)a, sc); r.y = __fmul_rn((float)b, sc);
    } else if (FMT == IQGPU_FMT_CS32) {
        const int2 v = __ldg(reinterpret_cast<const int2*>(raw) + i);
        r.x = (float)(((double)v.x * (1.0 / 2147483648.0)) * (double)gain);
        r.y = (float)(((double)v.y * (1.0 / 2147483648.0)) * (double)gain);
    } else if (FMT == IQGPU_FMT_CU32) {
        const uint2 v = __ldg(reinterpret_cast<const uint2*>(raw) + i);
        r.x = (float)((((double)v.x - 2147483647.5) * (1.0 / 2147483648.0)) * (double)gain);
        r.y = (float)((((double)v.y - 2147483647.5) * (1.0 / 2147483648.0)) * (double)gain);
    } else {  // CF32
        const float2 v = __ldg(reinterpret_cast<const float2*>(raw) + i);
        r.x = __fmul_rn(v.x, gain); r.y = __fmul_rn(v.y, gain);
    }
    return r;
}

// four consecutive frames starting at i (i % 4 == 0 relative to a 16-byte aligned base); frames
// at or beyond n read as zero.
template <int FMT>
__device__ __forceinline__ void load_quad(const void* __restrict__ raw, size_t i, size_t n, float sc, float gain,
                                          bool aligned, float2 (&x)[4])
{
    if (aligned && i + 4 <= n) {
        if (FMT == IQGPU_FMT_CS16 || FMT == IQGPU_FMT_SC16Q11) {
            const uint4 v = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const char*>(raw) + i * 4));
            const unsigned w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int k = 0; k < 4; k++) {
                x[k].x = __fmul_rn((float)(short)(w[k] & 0xffffu), sc);
                x[k].y = __fmul_rn((float)(short)(w[k] >> 16), sc);
            }
            return;
        }
        if (FMT == IQGPU_FMT_CU8 || FMT == IQGPU_FMT_CS8) {
            const uint2 v = __ldg(reinterpret_cast<const uint2*>(reinterpret_cast<const char*>(raw) + i * 2));
            const unsigned w[2] = {v.x, v.y};
#pragma unroll
            for (int k = 0; k < 4; k++) {
                unsigned b0 = (w[k >> 1] >> ((k & 1) * 16)) & 0xffu, b1 = (w[k >> 1] >> ((k & 1) * 16 + 8)) & 0xffu;
                if (FMT == IQGPU_FMT_CU8) {
                    x[k].x = __fmul_rn((float)b0 - 127.5f, sc); x[k].y = __fmul_rn((float)b1 - 127.5f, sc);
                } else {
                    x[k].x = __fmul_rn((float)(signed char)b0, sc); x[k].y = __fmul_rn((float)(signed char)b1, sc);
                }
            }
            return;
        }
        if (FMT == IQGPU_FMT_CF32) {
            const float4 a = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const char*>(raw) + i * 8));
            const float4 b = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const char*>(raw) + i * 8) + 1);
            x[0] = make_float2(__fmul_rn(a.x, gain), __fmul_rn(a.y, gain));
            x[1] = make_float2(__fmul_rn(a.z, gain), __fmul_rn(a.w, gain));
            x[2] = make_float2(__fmul_rn(b.x, gain), __fmul_rn(b.y, gain));
            x[3] = make_float2(__fmul_rn(b.z, gain), __fmul_rn(b.w, gain));
            return;
        }
    }
#pragma unroll
    for (int k = 0; k < 4; k++)
        x[k] = (i + k < n) ? load_frame<FMT>(raw, i + k, sc, gain) : make_float2(0.f, 0.f);
}

// =============================================================================================
// DC blocker as a blocked linear scan.
//   reference src/dc_block.c:76 -> liquid iirfilt (direct form II):  v[n] = x[n] + c v[n-1],
//   y[n] = v[n] - v[n-1]  ==  x[n] - (1-c) v[n-1].
// A warp owns a contiguous "run"; each lane owns 4 consecutive samples of every 128-sample
// row.  Row-local weighted prefix sums use shuffles; the run carry is kept in double.
// =============================================================================================
struct DcDev {
    float c, a;        // pole, 1-pole
    float w[5];        // c^(4*2^d), d = 0..4
    float lanepow[32]; // c^(4*lane)
    double c128;       // c^128
};

__host__ static inline DcDev make_dc_dev(float c, float a)
{
    DcDev d;
    d.c = c; d.a = a;
    for (int k = 0; k < 5; k++) d.w[k] = (float)pow((double)c, 4.0 * (double)(1 << k));
    for (int l = 0; l < 32; l++) d.lanepow[l] = (float)pow((double)c, 4.0 * l);
    d.c128 = pow((double)c, 128.0);
    return d;
}

// the same for a lane that owns 16 consecutive frames of a 512-frame tick (fused front v2, tick pre-pass)
struct DcDev16 {
    float c, a;          // pole, 1-pole
    float w[5];          // c^(16*2^s)
    float lanepow[32];   // c^(16*lane)
    float nac[16];       // -a c^k
};
__host__ static inline DcDev16 make_dc_dev16(float c, float a)
{
    DcDev16 d;
    d.c = c; d.a = a;
    for (int k = 0; k < 16; k++) d.nac[k] = (float)(-(double)a * pow((double)c, (double)k));
    for (int k = 0; k < 5; k++) d.w[k] = (float)pow((double)c, 16.0 * (double)(1 << k));
    for (int l = 0; l < 32; l++) d.lanepow[l] = (float)pow((double)c, 16.0 * l);
    return d;
}

// returns the row's inclusive weighted total in lane 31 (all lanes get it via shfl) and, per lane,
// E = v contribution of the lanes below (relative to a zero state at the row start)
__device__ __forceinline__ void dc_row_scan(const float2 (&x)[4], const DcDev& d, int lane, float2& E, float2& T)
{
    // local weighted sum of the lane's 4 samples
    float pr = x[0].x, pi = x[0].y;
#pragma unroll
    for (int k = 1; k < 4; k++) { pr = fmaf(pr, d.c, x[k].x); pi = fmaf(pi, d.c, x[k].y); }
#pragma unroll
    for (int s = 0; s < 5; s++) {
        const int dist = 1 << s;
        float qr = __shfl_up_sync(0xffffffffu, pr, dist);
        float qi = __shfl_up_sync(0xffffffffu, pi, dist);
        if (lane >= dist) { pr = fmaf(d.w[s], qr, pr); pi = fmaf(d.w[s], qi, pi); }
    }
    float er = __shfl_up_sync(0xffffffffu, pr, 1), ei = __shfl_up_sync(0xffffffffu, pi, 1);
    E = (lane == 0) ? make_float2(0.f, 0.f) : make_float2(er, ei);
    T.x = __shfl_sync(0xffffffffu, pr, 31);
    T.y = __shfl_sync(0xffffffffu, pi, 31);
}

// liquid LIQUID_NCO mix: 32-bit phase, 1024-entry sine table, nearest entry (nco.proto.c)
__device__ __forceinline__ float2 nco_mix(float2 x, uint32_t theta, float sign, const float* __restrict__ lut)
{
    const unsigned idx = ((theta + (1u << 21)) >> 22) & 0x3ffu;
    const float s = lut[idx] * sign;
    const float c = lut[(idx + 256u) & 0x3ffu];
    float2 y;
    y.x = __fsub_rn(__fmul_rn(x.x, c), __fmul_rn(x.y, s));
    y.y = __fadd_rn(__fmul_rn(x.x, s), __fmul_rn(x.y, c));
    return y;
}


// =============================================================================================
// packed FP32 pairs (sm_100a FFMA2 / FMUL2 / FADD2: fma.rn.f32x2, mul.rn.f32x2, add.rn.f32x2).
// Each half is an ordinary IEEE-754 round-to-nearest operation, so results are bit-identical to
// fmaf / __fmul_rn / __fadd_rn on the two components; one issue slot does the work of two.  A
// complex sample {re, im} that is scaled by a real tap is exactly this shape.
// =============================================================================================
typedef unsigned long long f32x2_t;
__device__ __forceinline__ f32x2_t pk2(float lo, float hi)
{
    f32x2_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ f32x2_t pk2(float2 v) { return pk2(v.x, v.y); }
__device__ __forceinline__ float2 unpk2(f32x2_t v)
{
    float2 r;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(v));
    return r;
}
__device__ __forceinline__ f32x2_t fma2(f32x2_t a, f32x2_t b, f32x2_t c)
{
    f32x2_t r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ f32x2_t mul2(f32x2_t a, f32x2_t b)
{
    f32x2_t r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2_t add2(f32x2_t a, f32x2_t b)
{
    f32x2_t r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
// h * {x.re, x.im} + {acc.re, acc.im}
__device__ __forceinline__ f32x2_t fma2s(float h, f32x2_t x, f32x2_t acc) { return fma2(pk2(h, h), x, acc); }

// The closed-form DC term of the warp-streaming front for output sample `o` (absolute index, o >= g.O0), which belongs to
// stretch w = (nk - B0) / L_full (nk = the input frame its polyphase window ends at).  ONE definition, used by the in-memory
// pass (w2_dc_correct_kernel) and by consumers that add the term while they load the stream (fir_param_kernel): same bits.
// Dp = o * step - g.pos.p_base (mod 2^64, ArbBase): exact, where o * step itself wraps from input frame 2^(40+S) on.
__device__ __forceinline__ long long dc_fold_frame(unsigned long long Dp, const W2DcGeom& g, int S)
{
    return (g.pos.k_base + (long long)(Dp >> 24)) << S;
}
// Pp = o * step, or o * step - p_base (the caller may carry it from sample to sample; the row bits are the same),
// since = nk - (first frame of stretch w's warm-up): below 2^31 for any stretch a launch can make (fused_launch_v2 checks)
__device__ __forceinline__ float2 dc_fold_add_at(float2 v, unsigned long long Pp, int since, float lnc, const W2DcCorr& c,
                                                 const float* __restrict__ sG)
{
    // (ex2.approx: 2^-22 relative on a term that is itself a small correction; the full expf cost the FIR 15 instructions
    // per staged sample, profiles/r02m_fir_fold_cfg2.md)
    const float e = __expf(lnc * (float)since) * sG[(unsigned)(Pp >> 16) & 0xffu];
    v.x = fmaf(c.c_out.x, e, v.x);
    v.y = fmaf(c.c_out.y, e, v.y);
    return v;
}
__device__ __forceinline__ float2 dc_fold_add(float2 v, unsigned long long Dp, long long nk, long long w,
                                              const W2DcGeom& g, float lnc, const W2DcCorr& c, const float* __restrict__ sG)
{
    return dc_fold_add_at(v, Dp, (int)(nk - (g.B0 + w * g.L_full - g.warm_frames)), lnc, c, sG);
}

}  // namespace iqgpu
