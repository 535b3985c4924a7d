// kernels.cu — stage kernels of the chain (sm_100a).  One kernel family per reference
// primitive; each header comment names the reference function it replaces.
//
// Layout conventions: cf32 streams are interleaved float2 {re, im}; raw integer inputs are
// interleaved I,Q.  "Stream" pointers address the first NEW sample of a call; older samples
// (filter history) live at negative offsets in the same allocation (see chain.cu DevStream).
#include "kernels.hpp"

#include <cooperative_groups.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "../../include/iqgpu.h"
#include "device_common.cuh"
#include "agc_math.h"

namespace cg = cooperative_groups;

namespace iqgpu {

template <int FMT>
__global__ void __launch_bounds__(256) dc_run_sums_kernel(const void* __restrict__ raw, size_t n, size_t lo, float gain,
                                                          DcDev d, uint32_t run_len, size_t n_runs, bool aligned,
                                                          double2* __restrict__ run_sums)
{
    const int lane = threadIdx.x & 31;
    const size_t warp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const size_t nwarps = ((size_t)gridDim.x * blockDim.x) >> 5;
    const float sc = in_scale<FMT>(gain);
    for (size_t run = warp; run < n_runs; run += nwarps) {
        const size_t base = run * run_len;
        const size_t end = (base + run_len < n) ? base + run_len : n;
        double vr = 0.0, vi = 0.0;
        for (size_t i0 = base; i0 < end; i0 += 128) {
            float2 x[4], E, T;
            const size_t i = i0 + lane * 4;
            if (i >= lo) load_quad<FMT>(raw, i, n, sc, gain, aligned, x);
            else {
#pragma unroll
                for (int k = 0; k < 4; k++)
                    x[k] = (i + k >= lo && i + k < n) ? load_frame<FMT>(raw, i + k, sc, gain) : make_float2(0.f, 0.f);
            }
            dc_row_scan(x, d, lane, E, T);
            vr = fma(d.c128, vr, (double)T.x);
            vi = fma(d.c128, vi, (double)T.y);
        }
        if (lane == 0) run_sums[run] = make_double2(vr, vi);
    }
}

// DC pre-pass for the fused front v2: one weighted sum per 512-frame tick, S_t = sum_k c^(511-k) x[k].
// A lane owns 16 consecutive frames (4 x LDG.128 issued back to back for cs16), folds them serially and
// the warp combines the 32 partial sums with a weighted shuffle tree; frames below `lo` and at or beyond
// `n` read as zero.
__global__ void __launch_bounds__(256) dc_tick_sums_kernel(const void* __restrict__ raw, size_t n, size_t lo, int fmt, float gain,
                                                           DcDev16 d, size_t n_ticks, bool aligned, double2* __restrict__ sums)
{
    const int lane = threadIdx.x & 31;
    const size_t warp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const size_t nwarps = ((size_t)gridDim.x * blockDim.x) >> 5;
    const bool cs16 = (fmt == IQGPU_FMT_CS16 || fmt == IQGPU_FMT_SC16Q11);
    float sc;
    switch (fmt) {
        case IQGPU_FMT_CS16: case IQGPU_FMT_CU16: sc = gain * (1.0f / 32768.0f); break;
        case IQGPU_FMT_SC16Q11: sc = gain * (1.0f / 2048.0f); break;
        case IQGPU_FMT_CS8: case IQGPU_FMT_CU8: sc = gain * (1.0f / 128.0f); break;
        default: sc = gain;
    }
    for (size_t tick = warp; tick < n_ticks; tick += nwarps) {
        const size_t t0 = tick * 512, a0 = t0 + (size_t)lane * 16;
        float2 x[16];
        if (cs16 && aligned && t0 >= lo && t0 + 512 <= n) {
            const uint4* src = reinterpret_cast<const uint4*>(reinterpret_cast<const char*>(raw) + a0 * 4);
            uint4 q[4];
#pragma unroll
            for (int j = 0; j < 4; j++) q[j] = __ldg(src + j);
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const unsigned w[4] = {q[j].x, q[j].y, q[j].z, q[j].w};
#pragma unroll
                for (int kk = 0; kk < 4; kk++) {
                    x[4 * j + kk].x = __fmul_rn((float)(short)(w[kk] & 0xffffu), sc);
                    x[4 * j + kk].y = __fmul_rn((float)(short)(w[kk] >> 16), sc);
                }
            }
        } else {
#pragma unroll
            for (int kk = 0; kk < 16; kk++) {
                const size_t i = a0 + kk;
                float2 v = make_float2(0.f, 0.f);
                if (i >= lo && i < n) {
                    switch (fmt) {
                        case IQGPU_FMT_CS16: case IQGPU_FMT_SC16Q11: v = load_frame<IQGPU_FMT_CS16>(raw, i, sc, gain); break;
                        case IQGPU_FMT_CU16: v = load_frame<IQGPU_FMT_CU16>(raw, i, sc, gain); break;
                        case IQGPU_FMT_CS8: v = load_frame<IQGPU_FMT_CS8>(raw, i, sc, gain); break;
                        case IQGPU_FMT_CU8: v = load_frame<IQGPU_FMT_CU8>(raw, i, sc, gain); break;
                        default: v = load_frame<IQGPU_FMT_CF32>(raw, i, sc, gain);
                    }
                }
                x[kk] = v;
            }
        }
        float pr = x[0].x, pi = x[0].y;
#pragma unroll
        for (int kk = 1; kk < 16; kk++) { pr = fmaf(pr, d.c, x[kk].x); pi = fmaf(pi, d.c, x[kk].y); }
        // weighted tree: after the step with distance dist, lanes that are multiples of 2*dist hold
        // c^(16*dist) * (own 16*dist frames) + (the next 16*dist frames)
#pragma unroll
        for (int s = 0; s < 5; s++) {
            const int dist = 1 << s;
            const float qr = __shfl_down_sync(0xffffffffu, pr, dist);
            const float qi = __shfl_down_sync(0xffffffffu, pi, dist);
            pr = fmaf(pr, d.w[s], qr);
            pi = fmaf(pi, d.w[s], qi);
        }
        if (lane == 0) sums[tick] = make_double2((double)pr, (double)pi);
    }
}

// ---- DC carry scan over the runs: v_start[r+1] = A_r v_start[r] + S_r -------------------------------
// Two small kernels.  (1) one warp per group of DC_GROUP runs folds the group into one affine map;
// (2) every CTA folds the groups in front of it (a few thousand at most), then one warp per group
// expands the per-run start states.  All in double.
constexpr int DC_GROUP = 256;                 // runs per group (8 per lane)
struct DcScanParams {
    size_t n_runs, n_groups;
    double A, A_last;                         // c^run_len, c^(padded length of the last run)
    double undo;                              // c^-(padding of the last run)
};
struct Affine { double a, br, bi; };
__device__ __forceinline__ Affine affine_then(const Affine& first, const Affine& second)
{   // apply `first`, then `second`
    Affine r;
    r.a = second.a * first.a;
    r.br = fma(second.a, first.br, second.br);
    r.bi = fma(second.a, first.bi, second.bi);
    return r;
}
__device__ __forceinline__ Affine affine_shfl_up(const Affine& v, int d)
{
    Affine r;
    r.a = __shfl_up_sync(0xffffffffu, v.a, d);
    r.br = __shfl_up_sync(0xffffffffu, v.br, d);
    r.bi = __shfl_up_sync(0xffffffffu, v.bi, d);
    return r;
}
// lane-local fold of the lane's 8 runs of group g; returns the inclusive warp scan in `inc`
__device__ __forceinline__ void dc_group_scan(const double2* __restrict__ run_sums, const DcScanParams& p, size_t g,
                                              int lane, double2 (&s)[8], Affine& inc)
{
    const size_t r0 = g * DC_GROUP + (size_t)lane * 8;
    Affine loc{1.0, 0.0, 0.0};
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const size_t r = r0 + k;
        if (r < p.n_runs) {
            s[k] = run_sums[r];
            const double Ar = (r == p.n_runs - 1) ? p.A_last : p.A;
            loc.a *= Ar; loc.br = fma(Ar, loc.br, s[k].x); loc.bi = fma(Ar, loc.bi, s[k].y);
        } else s[k] = make_double2(0.0, 0.0);
    }
    inc = loc;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const Affine prev = affine_shfl_up(inc, d);
        if (lane >= d) inc = affine_then(prev, inc);
    }
}

__global__ void __launch_bounds__(256) dc_group_agg_kernel(const double2* __restrict__ run_sums, DcScanParams p,
                                                           const double2* __restrict__ carry, double2* __restrict__ carry_snapshot,
                                                           double* __restrict__ grp)
{
    const int lane = threadIdx.x & 31;
    const size_t warp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (blockIdx.x == 0 && threadIdx.x == 0) *carry_snapshot = *carry;
    if (warp >= p.n_groups) return;
    double2 s[8];
    Affine inc;
    dc_group_scan(run_sums, p, warp, lane, s, inc);
    if (lane == 31) { grp[3 * warp] = inc.a; grp[3 * warp + 1] = inc.br; grp[3 * warp + 2] = inc.bi; }
}

__global__ void __launch_bounds__(1024) dc_expand_kernel(const double2* __restrict__ run_sums, DcScanParams p,
                                                         const double* __restrict__ grp, const double2* __restrict__ carry_snapshot,
                                                         double2* __restrict__ carry, double2* __restrict__ run_start)
{
    __shared__ Affine sh[1024];
    __shared__ double2 gstart[32];
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    const size_t g0 = (size_t)blockIdx.x * 32;          // first group of this CTA
    // ordered fold of groups [0, g0): thread t folds a contiguous slice, then a tree over threads
    {
        const size_t per = (g0 + 1023) / 1024;
        const size_t a0 = (size_t)t * per, a1 = (a0 + per < g0) ? a0 + per : g0;
        Affine f{1.0, 0.0, 0.0};
        for (size_t g = a0; g < a1; g++) f = affine_then(f, Affine{grp[3 * g], grp[3 * g + 1], grp[3 * g + 2]});
        sh[t] = f;
    }
    __syncthreads();
    for (int d = 1; d < 1024; d <<= 1) {
        Affine f;
        const bool act = (t & (2 * d - 1)) == (2 * d - 1);
        if (act) f = affine_then(sh[t - d], sh[t]);
        __syncthreads();
        if (act) sh[t] = f;
        __syncthreads();
    }
    if (t == 0) {
        const double2 v0 = *carry_snapshot;
        const Affine pre = sh[1023];
        double vr = fma(pre.a, v0.x, pre.br), vi = fma(pre.a, v0.y, pre.bi);
        for (int k = 0; k < 32; k++) {
            gstart[k] = make_double2(vr, vi);
            const size_t g = g0 + k;
            if (g < p.n_groups) {
                const double a = grp[3 * g];
                vr = fma(a, vr, grp[3 * g + 1]); vi = fma(a, vi, grp[3 * g + 2]);
            }
        }
    }
    __syncthreads();
    const size_t g = g0 + w;
    if (g >= p.n_groups) return;
    double2 s[8];
    Affine inc;
    dc_group_scan(run_sums, p, g, lane, s, inc);
    Affine exc = affine_shfl_up(inc, 1);
    if (lane == 0) exc = Affine{1.0, 0.0, 0.0};
    const double2 gs = gstart[w];
    double vr = fma(exc.a, gs.x, exc.br), vi = fma(exc.a, gs.y, exc.bi);
    const size_t r0 = g * DC_GROUP + (size_t)lane * 8;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const size_t r = r0 + k;
        if (r < p.n_runs) {
            run_start[r] = make_double2(vr, vi);
            const double Ar = (r == p.n_runs - 1) ? p.A_last : p.A;
            vr = fma(Ar, vr, s[k].x); vi = fma(Ar, vi, s[k].y);
            if (r == p.n_runs - 1) *carry = make_double2(vr * p.undo, vi * p.undo);   // state after ALL runs, padding undone
        }
    }
}

// =============================================================================================
// K1: pre-processor chain on one call: convert -> DC -> I/Q apply -> NCO mix
//   reference src/pre_processor.c:10-55 (order), sample_convert.c:127, dc_block.c:76,
//   iq_correct.c:307-313, frequency_shift.c:86-96 (liquid nco_crcf_mix_block_up/down).
// Element-wise stages use unfused multiplies/adds so they reproduce the C arithmetic exactly.
// =============================================================================================
template <int FMT, bool DC>
__global__ void __launch_bounds__(256) pre_kernel(const void* __restrict__ raw, size_t n, PreParams p, DcDev d,
                                                  uint32_t run_len, size_t n_runs, bool aligned,
                                                  const double2* __restrict__ run_start, float2* __restrict__ out)
{
    __shared__ float lut[1024];
    if (p.nco_enable) {
        for (int i = threadIdx.x; i < 1024; i += blockDim.x) lut[i] = p.nco_table[i];
        __syncthreads();
    }
    const int lane = threadIdx.x & 31;
    const size_t warp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const size_t nwarps = ((size_t)gridDim.x * blockDim.x) >> 5;
    const float sc = in_scale<FMT>(p.gain);
    const float lanepow = DC ? d.lanepow[lane] : 0.f;
    const bool out_aligned = ((reinterpret_cast<size_t>(out) & 15) == 0);
    for (size_t run = warp; run < n_runs; run += nwarps) {
        const size_t base = run * run_len;
        const size_t end = (base + run_len < n) ? base + run_len : n;
        double vr = 0.0, vi = 0.0;
        if (DC) { const double2 v = run_start[run]; vr = v.x; vi = v.y; }
        for (size_t i0 = base; i0 < end; i0 += 128) {
            const size_t i = i0 + lane * 4;
            float2 x[4];
            load_quad<FMT>(raw, i, n, sc, p.gain, aligned, x);
            if (DC) {
                float2 E, T;
                dc_row_scan(x, d, lane, E, T);
                // v just before the lane's first sample
                float wr = fmaf(lanepow, (float)vr, E.x), wi = fmaf(lanepow, (float)vi, E.y);
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const float xr = x[k].x, xi = x[k].y;
                    x[k].x = fmaf(-d.a, wr, xr);
                    x[k].y = fmaf(-d.a, wi, xi);
                    wr = fmaf(d.c, wr, xr);
                    wi = fmaf(d.c, wi, xi);
                }
                vr = fma(d.c128, vr, (double)T.x);
                vi = fma(d.c128, vi, (double)T.y);
            }
            if (p.iq_enable) {
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const float re = x[k].x;
                    x[k].x = __fmul_rn(re, p.iq_magp1);
                    x[k].y = __fadd_rn(x[k].y, __fmul_rn(p.iq_phase, re));
                }
            }
            if (p.nco_enable) {
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const uint32_t th = p.nco_theta0 + (uint32_t)(i + k) * p.nco_dtheta;
                    x[k] = nco_mix(x[k], th, p.nco_sign, lut);
                }
            }
            if (out_aligned && i + 4 <= n) {
                float4* o = reinterpret_cast<float4*>(out + i);
                o[0] = make_float4(x[0].x, x[0].y, x[1].x, x[1].y);
                o[1] = make_float4(x[2].x, x[2].y, x[3].x, x[3].y);
            } else {
#pragma unroll
                for (int k = 0; k < 4; k++)
                    if (i + k < n) out[i + k] = x[k];
            }
        }
    }
}

static inline int grid_for_warps(size_t warps_needed, int threads)
{
    size_t blocks = (warps_needed * 32 + threads - 1) / threads;
    const size_t cap = 148 * 16;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (int)blocks;
}

#define DISPATCH_FMT(fmt, CALL)                                          \
    switch (fmt) {                                                        \
        case IQGPU_FMT_CS16:    { CALL(IQGPU_FMT_CS16); break; }          \
        case IQGPU_FMT_SC16Q11: { CALL(IQGPU_FMT_SC16Q11); break; }       \
        case IQGPU_FMT_CU16:    { CALL(IQGPU_FMT_CU16); break; }          \
        case IQGPU_FMT_CS8:     { CALL(IQGPU_FMT_CS8); break; }           \
        case IQGPU_FMT_CU8:     { CALL(IQGPU_FMT_CU8); break; }           \
        case IQGPU_FMT_CS24:    { CALL(IQGPU_FMT_CS24); break; }          \
        case IQGPU_FMT_CS32:    { CALL(IQGPU_FMT_CS32); break; }          \
        case IQGPU_FMT_CU32:    { CALL(IQGPU_FMT_CU32); break; }          \
        case IQGPU_FMT_CF32:    { CALL(IQGPU_FMT_CF32); break; }          \
        default: return cudaErrorInvalidValue;                            \
    }

cudaError_t launch_dc_run_sums(const void* raw, size_t n, const PreParams& p, uint32_t run_len,
                               double2* run_sums, cudaStream_t st)
{
    return launch_dc_run_sums_masked(raw, n, 0, p, run_len, run_sums, st);
}

cudaError_t launch_dc_run_sums_masked(const void* raw, size_t n, size_t lo, const PreParams& p, uint32_t run_len,
                                      double2* run_sums, cudaStream_t st)
{
    if (n == 0) return cudaSuccess;
    const size_t n_runs = (n + run_len - 1) / run_len;
    const DcDev d = make_dc_dev(p.dc_c, p.dc_a);
    const bool aligned = (reinterpret_cast<size_t>(raw) & 15) == 0;
    const int grid = grid_for_warps(n_runs, 256);
#define CALL(F) dc_run_sums_kernel<F><<<grid, 256, 0, st>>>(raw, n, lo, p.gain, d, run_len, n_runs, aligned, run_sums)
    DISPATCH_FMT(p.format, CALL)
#undef CALL
    return cudaGetLastError();
}

cudaError_t launch_dc_tick_sums(const void* raw, size_t n, size_t lo, const PreParams& p, double2* sums, cudaStream_t st)
{
    if (n == 0) return cudaSuccess;
    const size_t n_ticks = (n + 511) / 512;
    const DcDev16 d = make_dc_dev16(p.dc_c, p.dc_a);
    const bool aligned = (reinterpret_cast<size_t>(raw) & 15) == 0;
    const int grid = grid_for_warps(n_ticks, 256);
    dc_tick_sums_kernel<<<grid, 256, 0, st>>>(raw, n, lo, p.format, p.gain, d, n_ticks, aligned, sums);
    return cudaGetLastError();
}

cudaError_t launch_dc_scan(const double2* run_sums, size_t n_runs, uint32_t run_len, size_t n,
                           float dc_c, double2* carry_inout, double2* run_start, double* scan_ws, cudaStream_t st,
                           uint32_t row_len)
{
    if (n_runs == 0) return cudaSuccess;
    DcScanParams p{};
    p.n_runs = n_runs;
    p.n_groups = (n_runs + DC_GROUP - 1) / DC_GROUP;
    const double c = (double)dc_c;
    // rows are processed whole (128 frames); the zero padding of the last run only decays the state
    const size_t last_len = n - (n_runs - 1) * (size_t)run_len;
    const size_t last_pad = ((last_len + row_len - 1) / row_len) * row_len;
    p.A = pow(c, (double)run_len);
    p.A_last = pow(c, (double)last_pad);
    p.undo = pow(c, -(double)(last_pad - last_len));
    double2* snapshot = reinterpret_cast<double2*>(scan_ws);
    double* grp = scan_ws + 2;
    const int g1 = (int)((p.n_groups * 32 + 255) / 256);
    dc_group_agg_kernel<<<g1, 256, 0, st>>>(run_sums, p, carry_inout, snapshot, grp);
    const int g2 = (int)((p.n_groups + 31) / 32);
    dc_expand_kernel<<<g2, 1024, 0, st>>>(run_sums, p, grp, snapshot, carry_inout, run_start);
    return cudaGetLastError();
}
size_t dc_scan_workspace_doubles(size_t n_runs) { return 2 + 3 * ((n_runs + DC_GROUP - 1) / DC_GROUP) + 8; }

cudaError_t launch_pre(const void* raw, size_t n, const PreParams& p, uint32_t run_len,
                       const double2* run_start, float2* out, cudaStream_t st)
{
    if (n == 0) return cudaSuccess;
    const size_t n_runs = (n + run_len - 1) / run_len;
    const DcDev d = make_dc_dev(p.dc_enable ? p.dc_c : 0.f, p.dc_a);
    const bool aligned = (reinterpret_cast<size_t>(raw) & 15) == 0;
    const int grid = grid_for_warps(n_runs, 256);
#define CALL(F)                                                                                             \
    if (p.dc_enable) pre_kernel<F, true><<<grid, 256, 0, st>>>(raw, n, p, d, run_len, n_runs, aligned, run_start, out); \
    else pre_kernel<F, false><<<grid, 256, 0, st>>>(raw, n, p, d, run_len, n_runs, aligned, run_start, out)
    DISPATCH_FMT(p.format, CALL)
#undef CALL
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// DC blocker, REFERENCE ROUNDING (dc_mode 1): liquid's iirfilt_crcf in direct form II keeps the integrator state
// v ~ dc / alpha in fp32 and rounds it twice per sample (dc_block.c:76-85 -> iirfilt_crcf_execute_block):
//     v0 = x - a1 * v1 ;  y = (0 + b0 * v0) + b1 * v1      a1 = -1 + alpha, b = {1, -1}
// That rounding sequence is a property of the serial evaluation and only a serial evaluation reproduces it: one thread per
// component walks the stream (8 dependent cycles per sample, ~250 Msamples/s).  It exists for the module-level
// dc_block_apply drop-in (16384-frame chunks, where it costs what a launch costs) and for the parity tests; the chunk-train
// path evaluates the same difference equation in exact arithmetic (DESIGN.md, DC blocker).
// ---------------------------------------------------------------------------------------------
constexpr int DCREF_TILE = 2048;
__global__ void __launch_bounds__(256, 1) dc_reference_kernel(float2* __restrict__ x, size_t n, float a1, float2* __restrict__ state)
{
    __shared__ float tile[2 * DCREF_TILE];
    const int t = threadIdx.x;
    float v = 0.f;
    if (t < 2) v = reinterpret_cast<const float*>(state)[t];
    for (size_t base = 0; base < n; base += DCREF_TILE) {
        const size_t cnt = (n - base < (size_t)DCREF_TILE) ? n - base : (size_t)DCREF_TILE;
        float* g = reinterpret_cast<float*>(x + base);
        for (size_t i = t; i < 2 * cnt; i += 256) tile[i] = g[i];
        __syncthreads();
        if (t < 2) {
#pragma unroll 8
            for (size_t k = 0; k < cnt; k++) {
                const float xin = tile[2 * k + t];
                const float v1 = v;
                v = __fsub_rn(xin, __fmul_rn(a1, v1));
                tile[2 * k + t] = __fadd_rn(__fadd_rn(0.f, __fmul_rn(1.0f, v)), __fmul_rn(-1.0f, v1));
            }
        }
        __syncthreads();
        for (size_t i = t; i < 2 * cnt; i += 256) g[i] = tile[i];
        __syncthreads();
    }
    if (t < 2) reinterpret_cast<float*>(state)[t] = v;
}

cudaError_t launch_dc_reference(float2* x, size_t n, float dc_c, float2* state, cudaStream_t st)
{
    if (n == 0) return cudaSuccess;
    dc_reference_kernel<<<1, 256, 0, st>>>(x, n, -dc_c, state);
    return cudaGetLastError();
}

// =============================================================================================
// K2 (unfused building blocks): liquid msresamp_crcf pieces, reference src/resampler.c:49
// =============================================================================================
// halfband decimator (liquid resamp2_crcf_decim_execute):
//   y[k] = sum_{j<2m} h1[j] x[2(k-2m+1+j)] + x[2(k-m)+1]      (x by absolute stage-input index)
__global__ void __launch_bounds__(256) halfband_decim_kernel(const float2* __restrict__ x, long long a0,
                                                             const float* __restrict__ h1, unsigned m,
                                                             long long k0, size_t count, float scale,
                                                             float2* __restrict__ y)
{
    extern __shared__ float sh1[];
    for (unsigned i = threadIdx.x; i < 2 * m; i += blockDim.x) sh1[i] = h1[i];
    __syncthreads();
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < count; t += (size_t)gridDim.x * blockDim.x) {
        const long long k = k0 + (long long)t;
        const float2* xe = x + (2 * (k - 2 * (long long)m + 1) - a0);
        float sr = 0.f, si = 0.f;
        for (unsigned j = 0; j < 2 * m; j++) {
            const float2 v = xe[2 * j];
            sr = fmaf(sh1[j], v.x, sr);
            si = fmaf(sh1[j], v.y, si);
        }
        const float2 c = x[2 * (k - (long long)m) + 1 - a0];
        y[t] = make_float2((c.x + sr) * scale, (c.y + si) * scale);
    }
}

// halfband interpolator (liquid resamp2_crcf_interp_execute):
//   y[2k] = x[k-m] ;  y[2k+1] = sum_{j<2m} h1[j] x[k-2m+1+j]
__global__ void __launch_bounds__(256) halfband_interp_kernel(const float2* __restrict__ x, long long a0,
                                                              const float* __restrict__ h1, unsigned m,
                                                              long long k0, size_t count, float2* __restrict__ y)
{
    extern __shared__ float sh1[];
    for (unsigned i = threadIdx.x; i < 2 * m; i += blockDim.x) sh1[i] = h1[i];
    __syncthreads();
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < count; t += (size_t)gridDim.x * blockDim.x) {
        const long long k = k0 + (long long)t;
        const float2* xw = x + (k - 2 * (long long)m + 1 - a0);
        float sr = 0.f, si = 0.f;
        for (unsigned j = 0; j < 2 * m; j++) {
            const float2 v = xw[j];
            sr = fmaf(sh1[j], v.x, sr);
            si = fmaf(sh1[j], v.y, si);
        }
        y[2 * t] = x[k - (long long)m - a0];
        y[2 * t + 1] = make_float2(sr, si);
    }
}

// arbitrary-rate polyphase stage (liquid resamp_crcf, fixed-point phase; firpfb bank of 256):
//   output o: P = phase0 + o*step, k = kbase + (P >> 24), idx = (P & (2^24-1)) >> 16,
//   y = sum_{i<14} bank[idx][i] * x[k-13+i]
__global__ void __launch_bounds__(256) arb_kernel(const float2* __restrict__ x, long long a0,
                                                  const float* __restrict__ bank, uint32_t step, long long kbase,
                                                  uint32_t phase0, size_t count, float2* __restrict__ y)
{
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < count; t += (size_t)gridDim.x * blockDim.x) {
        const unsigned long long P = (unsigned long long)phase0 + (unsigned long long)t * step;
        const long long k = kbase + (long long)(P >> 24);
        const unsigned idx = (unsigned)((P & 0xffffffull) >> 16);
        const float* __restrict__ b = bank + idx * 14;
        const float2* xw = x + (k - 13 - a0);
        float sr = 0.f, si = 0.f;
#pragma unroll
        for (int i = 0; i < 14; i++) {
            const float2 v = xw[i];
            const float h = __ldg(b + i);
            sr = fmaf(h, v.x, sr);
            si = fmaf(h, v.y, si);
        }
        y[t] = make_float2(sr, si);
    }
}

static inline int grid_1d(size_t count, int threads)
{
    size_t blocks = (count + threads - 1) / threads;
    const size_t cap = 148 * 32;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (int)blocks;
}

cudaError_t launch_halfband_decim(const float2* x, int64_t a0, const float* h1, unsigned m, int64_t k0,
                                  size_t count, float scale, float2* y, cudaStream_t st)
{
    if (count == 0) return cudaSuccess;
    halfband_decim_kernel<<<grid_1d(count, 256), 256, 2 * m * sizeof(float), st>>>(x, a0, h1, m, k0, count, scale, y);
    return cudaGetLastError();
}
cudaError_t launch_halfband_interp(const float2* x, int64_t a0, const float* h1, unsigned m, int64_t k0,
                                   size_t count, float2* y, cudaStream_t st)
{
    if (count == 0) return cudaSuccess;
    halfband_interp_kernel<<<grid_1d(count, 256), 256, 2 * m * sizeof(float), st>>>(x, a0, h1, m, k0, count, y);
    return cudaGetLastError();
}
cudaError_t launch_arb(const float2* x, int64_t a0, const float* bank, uint32_t step, int64_t kbase,
                       uint32_t phase0, size_t count, float2* y, cudaStream_t st)
{
    if (count == 0) return cudaSuccess;
    arb_kernel<<<grid_1d(count, 256), 256, 0, st>>>(x, a0, bank, step, kbase, phase0, count, y);
    return cudaGetLastError();
}

template <int FMT> __device__ __forceinline__ void store_out(void* __restrict__ out, size_t i, float2 v);
template <int FMT> __device__ __forceinline__ void store_out4(void* __restrict__ out, size_t i, size_t n, const float2 (&v)[4], bool vec);

// =============================================================================================
// K3: tiled time-domain FIR.  reference src/filter.c:449-462 -> liquid firfilt_crcf/cccf
//   y[n] = sum_{i<N} hrev[i] x[n-(N-1)+i]   (oldest sample first, like liquid's dot product)
// Block: 128 threads x 8 consecutive outputs = 1024 outputs.  Taps are consumed in chunks of
// FIR_TC; the input window of a chunk is staged in shared memory with one pad slot per 8
// samples so that lane-strided reads (stride 8 float2) are bank-conflict free.  Each thread
// keeps an 8-sample sliding register window: one LDS.64 + 16 (real) / 32 (complex) FFMA per tap.
// =============================================================================================
constexpr int FIR_R = 8;
constexpr int FIR_THREADS = 128;
constexpr int FIR_TILE = FIR_R * FIR_THREADS;   // outputs per block
constexpr int FIR_TC = 256;                     // taps per chunk (multiple of FIR_R)
__device__ __forceinline__ int fir_pad(int j) { return j + (j >> 3); }

template <bool CPLX>
__global__ void __launch_bounds__(FIR_THREADS) fir_kernel(const float2* __restrict__ x, size_t n,
                                                          const float* __restrict__ hrev, unsigned ntaps,
                                                          float2* __restrict__ y)
{
    constexpr int WIN = FIR_TILE + FIR_TC;  // samples staged per chunk (one spare group)
    __shared__ float2 sx[WIN + WIN / 8 + 8];
    __shared__ float2 sh[FIR_TC];           // (re, im) or (re, 0)
    const int t = threadIdx.x;
    const long long tile0 = (long long)blockIdx.x * FIR_TILE;  // first output of this block
    float2 acc[FIR_R];
#pragma unroll
    for (int r = 0; r < FIR_R; r++) acc[r] = make_float2(0.f, 0.f);

    for (unsigned c0 = 0; c0 < ntaps; c0 += FIR_TC) {
        const int tc = (ntaps - c0 < (unsigned)FIR_TC) ? (int)(ntaps - c0) : FIR_TC;
        // sample needed by output o (block-relative) and tap i: x[tile0 + o - (ntaps-1) + i]
        const long long wbase = tile0 - (long long)(ntaps - 1) + c0;
        __syncthreads();
        for (int j = t; j < FIR_TILE + tc - 1; j += FIR_THREADS) {
            const long long g = wbase + j;
            sx[fir_pad(j)] = (g < (long long)n) ? x[g] : make_float2(0.f, 0.f);
        }
        for (int j = t; j < tc; j += FIR_THREADS)
            sh[j] = CPLX ? make_float2(hrev[2 * (c0 + j)], hrev[2 * (c0 + j) + 1]) : make_float2(hrev[c0 + j], 0.f);
        __syncthreads();

        float2 win[FIR_R];
        const int o0 = t * FIR_R;
#pragma unroll
        for (int r = 0; r < FIR_R; r++) win[r] = sx[fir_pad(o0 + r)];
        for (int i0 = 0; i0 < tc; i0 += FIR_R) {
#pragma unroll
            for (int u = 0; u < FIR_R; u++) {
                const float2 h = sh[i0 + u];
#pragma unroll
                for (int r = 0; r < FIR_R; r++) {
                    const float2 v = win[(r + u) % FIR_R];
                    if (CPLX) {
                        // (hr + j hi)(vr + j vi)
                        acc[r].x = fmaf(h.x, v.x, acc[r].x);
                        acc[r].x = fmaf(-h.y, v.y, acc[r].x);
                        acc[r].y = fmaf(h.x, v.y, acc[r].y);
                        acc[r].y = fmaf(h.y, v.x, acc[r].y);
                    } else {
                        acc[r].x = fmaf(h.x, v.x, acc[r].x);
                        acc[r].y = fmaf(h.x, v.y, acc[r].y);
                    }
                }
                win[u % FIR_R] = sx[fir_pad(o0 + i0 + u + FIR_R)];
            }
        }
    }
#pragma unroll
    for (int r = 0; r < FIR_R; r++) {
        const long long o = tile0 + t * FIR_R + r;
        if (o < (long long)n) y[o] = acc[r];
    }
}

// Same tiling with the taps held in the kernel-parameter constant bank: every FFMA then reads its tap
// as a uniform/constant operand (two register reads instead of three).  On this part the three-register
// FFMA issues every other cycle per scheduler; the smem-tap kernel above sits exactly at that limit
// (cfg2: 22.3 M outputs x 255 taps in 0.62 ms = 0.5 FFMA/clk/SMSP).
constexpr unsigned FIR_PARAM_TAPS = 4096;           // floats (real taps) or 2048 complex taps: 16 KB of parameters
struct FirTaps { float h[FIR_PARAM_TAPS]; };

// Samples and accumulators are packed {re, im} pairs: a real tap is one FFMA2 per output (tap as a scalar uniform
// operand), a complex tap two (the second on the swapped pair with {-hi, hi}); each half is the same IEEE fma sequence as
// the scalar form.  FFMA2 has the FLOP rate of FFMA at half the issue slots, which leaves room for the LDS next to it.
// OUTFMT != 0: the filter is the last cf32 stage of the chain (no post shift, no AGC): the epilogue converts to the
// output sample format (sample_convert.c:213-306, same code as the post kernel) and writes the final stream, so the
// filtered cf32 stream is never stored.
// FOLD: the samples x[0 .. n) lack the fused front's closed-form DC term (DcFold, kernels.hpp); it is added while the tile
// is staged (the history below x[0] is complete).  A thread's samples are 128 apart and a stretch spans thousands of
// outputs, so the stretch index costs one 64-bit division per thread and tile, then comparisons.
template <bool CPLX, int OUTFMT, bool FOLD>
__global__ void __launch_bounds__(FIR_THREADS) fir_param_kernel(const float2* __restrict__ x, size_t n, unsigned ntaps,
                                                                float2* __restrict__ y, void* __restrict__ out_conv, bool vec_out,
                                                                const __grid_constant__ FirTaps T, const __grid_constant__ DcFold F)
{
    constexpr int WIN = FIR_TILE + FIR_TC;
    __shared__ __align__(16) f32x2_t sx[WIN + WIN / 8 + 8];
    __shared__ float sG[FOLD ? 256 : 1];
    const int t = threadIdx.x;
    const long long tile0 = (long long)blockIdx.x * FIR_TILE;
    if (FOLD) {
        for (int i = t; i < 256; i += FIR_THREADS) sG[i] = F.G[i];
    }
    const float lnc = FOLD ? (float)F.geo.lnc : 0.f;
    f32x2_t acc[FIR_R];
#pragma unroll
    for (int r = 0; r < FIR_R; r++) acc[r] = 0ull;
    for (unsigned c0 = 0; c0 < ntaps; c0 += FIR_TC) {
        const int tc = (ntaps - c0 < (unsigned)FIR_TC) ? (int)(ntaps - c0) : FIR_TC;
        const long long wbase = tile0 - (long long)(ntaps - 1) + c0;
        __syncthreads();
        // per thread: the sample's o * step carried from sample to sample, the stretch it is in (w), that stretch's record
        // and first warm-up frame; all 64-bit work happens once per thread and tile
        long long w = -1, w_end = 0, w_from = 0;
        W2DcCorr cw{};
        unsigned long long Pp = FOLD ? (unsigned long long)(F.O0 + wbase + t) * F.step : 0ull;
        const unsigned long long dPp = (unsigned long long)FIR_THREADS * F.step;
        for (int j = t; j < FIR_TILE + tc - 1; j += FIR_THREADS, Pp += dPp) {
            const long long g = wbase + j;
            f32x2_t v = (g < (long long)n) ? *reinterpret_cast<const f32x2_t*>(x + g) : 0ull;
            if (FOLD && g >= 0 && g < (long long)n) {
                const long long nk = (long long)(Pp >> 24) << F.S;
                if (w < 0 || nk >= w_end) {
                    if (w < 0) { w = (nk - F.geo.B0) / F.geo.L_full; w_end = F.geo.B0 + (w + 1) * F.geo.L_full; }
                    while (nk >= w_end) { w++; w_end += F.geo.L_full; }
                    w_from = w_end - F.geo.L_full - F.geo.warm_frames;
                    if (w > 0) cw = F.corr[w];
                }
                if (w > 0) v = pk2(dc_fold_add_at(unpk2(v), Pp, (int)(nk - w_from), lnc, cw, sG));
            }
            sx[fir_pad(j)] = v;
        }
        __syncthreads();
        f32x2_t win[FIR_R];
        const f32x2_t* __restrict__ sp = sx + fir_pad(t * FIR_R);     // o0 and i0 are multiples of 8: pad(o0 + i0 + k) = pad(o0) + 9 i0/8 + k
#pragma unroll
        for (int r = 0; r < FIR_R; r++) win[r] = sp[r];
        for (int i0 = 0; i0 < tc; i0 += FIR_R) {
            sp += FIR_R + 1;
#pragma unroll
            for (int u = 0; u < FIR_R; u++) {
                const float hx = CPLX ? T.h[2 * (c0 + i0 + u)] : T.h[c0 + i0 + u];
                const float hy = CPLX ? T.h[2 * (c0 + i0 + u) + 1] : 0.f;
                const f32x2_t hh = pk2(hx, hx), hs = pk2(-hy, hy);
#pragma unroll
                for (int r = 0; r < FIR_R; r++) {
                    const f32x2_t v = win[(r + u) % FIR_R];
                    acc[r] = fma2(hh, v, acc[r]);
                    if (CPLX) {                                        // (hr + j hi)(vr + j vi)
                        const float2 f = unpk2(v);
                        acc[r] = fma2(hs, pk2(f.y, f.x), acc[r]);
                    }
                }
                win[u % FIR_R] = sp[u];
            }
        }
    }
    if (OUTFMT != 0) {
#pragma unroll
        for (int q = 0; q < FIR_R; q += 4) {
            const float2 v[4] = {unpk2(acc[q]), unpk2(acc[q + 1]), unpk2(acc[q + 2]), unpk2(acc[q + 3])};
            const long long o = tile0 + t * FIR_R + q;
            if (o < (long long)n) store_out4<OUTFMT == 0 ? IQGPU_FMT_CF32 : OUTFMT>(out_conv, (size_t)o, n, v, vec_out);
        }
        return;
    }
#pragma unroll
    for (int r = 0; r < FIR_R; r++) {
        const long long o = tile0 + t * FIR_R + r;
        if (o < (long long)n) y[o] = unpk2(acc[r]);
    }
}

bool fir_can_fold_dc(unsigned ntaps_padded, int complex_taps, bool have_host_taps)
{
    const unsigned nfloats = ntaps_padded * (complex_taps ? 2u : 1u);
    return have_host_taps && nfloats <= FIR_PARAM_TAPS && !getenv("IQGPU_FIR_SMEM_TAPS") && !getenv("IQGPU_NO_DC_FOLD");
}

bool fir_can_convert_out(int out_format, unsigned ntaps_padded, int complex_taps)
{
    const unsigned nfloats = ntaps_padded * (complex_taps ? 2u : 1u);
    if (nfloats > FIR_PARAM_TAPS || getenv("IQGPU_FIR_SMEM_TAPS") || getenv("IQGPU_FIR_NO_CONVERT")) return false;
    return out_format == IQGPU_FMT_CS16 || out_format == IQGPU_FMT_CU8 || out_format == IQGPU_FMT_CS8;
}

cudaError_t launch_fir(const float2* x, size_t n, const float* hrev, unsigned ntaps_padded, int complex_taps,
                       float2* y, cudaStream_t st, const float* hrev_host, int out_format, void* out_conv, const DcFold* fold)
{
    if (n == 0) return cudaSuccess;
    const int grid = (int)((n + FIR_TILE - 1) / FIR_TILE);
    const unsigned nfloats = ntaps_padded * (complex_taps ? 2u : 1u);
    if (out_conv && !(hrev_host && fir_can_convert_out(out_format, ntaps_padded, complex_taps))) return cudaErrorInvalidValue;
    const bool folding = fold && fold->corr;
    if (folding && !fir_can_fold_dc(ntaps_padded, complex_taps, hrev_host != nullptr)) return cudaErrorInvalidValue;
    if (hrev_host && nfloats <= FIR_PARAM_TAPS && !getenv("IQGPU_FIR_SMEM_TAPS")) {
        static thread_local FirTaps T;      // 16 KB: copied into the launch's parameter buffer
        memcpy(T.h, hrev_host, nfloats * sizeof(float));
        const bool vo = (reinterpret_cast<size_t>(out_conv) & 15) == 0;
        const DcFold F = folding ? *fold : DcFold{};
#define FIR_GO(C, O, D) fir_param_kernel<C, O, D><<<grid, FIR_THREADS, 0, st>>>(x, n, ntaps_padded, y, out_conv, vo, T, F)
#define FIR_FMT(C, D)                                                          \
        do {                                                                   \
            if (!out_conv) FIR_GO(C, 0, D);                                    \
            else if (out_format == IQGPU_FMT_CS16) FIR_GO(C, IQGPU_FMT_CS16, D); \
            else if (out_format == IQGPU_FMT_CU8) FIR_GO(C, IQGPU_FMT_CU8, D); \
            else FIR_GO(C, IQGPU_FMT_CS8, D);                                  \
        } while (0)
        if (complex_taps) { if (folding) FIR_FMT(true, true); else FIR_FMT(true, false); }
        else              { if (folding) FIR_FMT(false, true); else FIR_FMT(false, false); }
#undef FIR_FMT
#undef FIR_GO
        return cudaGetLastError();
    }
    if (complex_taps) fir_kernel<true><<<grid, FIR_THREADS, 0, st>>>(x, n, hrev, ntaps_padded, y);
    else fir_kernel<false><<<grid, FIR_THREADS, 0, st>>>(x, n, hrev, ntaps_padded, y);
    return cudaGetLastError();
}

// =============================================================================================
// K5: post-processor.  reference src/post_processor.c:9-70 (order), frequency_shift.c:86-96,
//     agc.c:86-222, sample_convert.c:213-306.
// =============================================================================================
__device__ __forceinline__ unsigned find_segment(const uint32_t* __restrict__ seg_start, unsigned nseg, uint32_t i)
{
    // largest s with seg_start[s] <= i  (seg_start[nseg] == n)
    unsigned lo = 0, hi = nseg;
    while (hi - lo > 1) {
        const unsigned mid = (lo + hi) >> 1;
        if (__ldg(seg_start + mid) <= i) lo = mid; else hi = mid;
    }
    return lo;
}

// ---- warp tiles -------------------------------------------------------------------------------
// The post-processor kernels walk the output stream in tiles of POST_TILE consecutive frames per
// warp; a lane owns 4 consecutive frames per step (2 x LDG.128 in, one vector store out) and keeps
// its segment (= reference chunk) index in a register, advancing it monotonically.
constexpr int POST_TILE = 2048;
__device__ __forceinline__ void load4(const float2* __restrict__ x, size_t i, size_t n, bool vec, float2 (&v)[4])
{
    if (vec && i + 4 <= n) {
        const float4 a = __ldg(reinterpret_cast<const float4*>(x + i));
        const float4 b = __ldg(reinterpret_cast<const float4*>(x + i) + 1);
        v[0] = make_float2(a.x, a.y); v[1] = make_float2(a.z, a.w);
        v[2] = make_float2(b.x, b.y); v[3] = make_float2(b.z, b.w);
    } else {
#pragma unroll
        for (int k = 0; k < 4; k++) v[k] = (i + k < n) ? x[i + k] : make_float2(0.f, 0.f);
    }
}

// per-segment peak |x| after the (optional) post NCO.  reference agc.c:117-124 / 168-173 uses
// cabsf (hypotf, correctly rounded = sqrt of the double sum of squares, rounded once).  sqrt and
// the float rounding are monotone, so a lane tracks max(re^2 + im^2) in double and takes one
// square root when it leaves a segment.
__device__ __forceinline__ void peak_flush(float* __restrict__ seg_peak, unsigned seg, double d)
{
    if (d > 0.0) atomicMax(reinterpret_cast<unsigned*>(seg_peak) + seg, __float_as_uint((float)sqrt(d)));
}
__global__ void __launch_bounds__(256) agc_peaks_kernel(const float2* __restrict__ x, size_t n, PostParams p,
                                                        const uint32_t* __restrict__ seg_start, unsigned nseg,
                                                        float* __restrict__ seg_peak, bool vec)
{
    __shared__ float lut[1024];
    if (p.nco_enable) {
        for (int i = threadIdx.x; i < 1024; i += blockDim.x) lut[i] = p.nco_table[i];
        __syncthreads();
    }
    const int lane = threadIdx.x & 31;
    const size_t warp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const size_t nwarps = ((size_t)gridDim.x * blockDim.x) >> 5;
    const size_t ntiles = (n + POST_TILE - 1) / POST_TILE;
    for (size_t tile = warp; tile < ntiles; tile += nwarps) {
        const size_t t0 = tile * POST_TILE;
        size_t i = t0 + (size_t)lane * 4;
        unsigned seg = (i < n) ? find_segment(seg_start, nseg, (uint32_t)i) : 0u;
        uint32_t seg_end = (i < n) ? __ldg(seg_start + seg + 1) : 0u;
        double d = 0.0;
#pragma unroll 1
        for (int it = 0; it < POST_TILE / 128; it++, i += 128) {
            if (i >= n) break;
            float2 v[4];
            load4(x, i, n, vec, v);
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const size_t ik = i + k;
                if (ik >= n) break;
                while ((uint32_t)ik >= seg_end) {           // next non-empty segment
                    peak_flush(seg_peak, seg, d); d = 0.0;
                    seg++; seg_end = __ldg(seg_start + seg + 1);
                }
                float2 w = v[k];
                if (p.nco_enable) w = nco_mix(w, p.nco_theta0 + (uint32_t)ik * p.nco_dtheta, p.nco_sign, lut);
                d = fmax(d, fma((double)w.x, (double)w.x, (double)w.y * (double)w.y));
            }
        }
        // one atomic per warp when the whole tile sits in one segment
        const unsigned seg0 = __shfl_sync(0xffffffffu, seg, 0);
        if (__all_sync(0xffffffffu, seg == seg0)) {
#pragma unroll
            for (int s = 16; s > 0; s >>= 1) d = fmax(d, __shfl_xor_sync(0xffffffffu, d, s));
            if (lane == 0) peak_flush(seg_peak, seg0, d);
        } else peak_flush(seg_peak, seg, d);
    }
}

// digital AGC state machine, one step per reference chunk (agc.c:105-222).  Wall-clock reads in
// the reference (agc.c:176,202-207) are replaced by the sample clock seen/target_rate.
// One warp walks the chunks 32 at a time.  While nothing data dependent happens inside a group
// (no ratchet, no creep, no lock transition) all 32 gains are produced in one step; otherwise the
// group is replayed chunk by chunk with warp-uniform state -- the results are those of the
// sequential reference loop in every case.
struct AgcStep {   // sequential reference step, shared by both paths
    __device__ static __forceinline__ float run(AgcState& s, float pk, unsigned cnt, float target, double rate)
    {
        float g;
        if (!s.locked) {
            if (pk > s.peak_mem) s.peak_mem = pk;
            const float safe = (s.peak_mem < 1e-4f) ? 1e-4f : s.peak_mem;
            g = __fdiv_rn(target, safe);
            const double elapsed = (double)s.seen / rate;
            if (elapsed > (double)2.0f) { s.locked = 1; s.gain = g; s.last_strong = elapsed; }
        } else {
            g = s.gain;
            const float opk = __fmul_rn(pk, g);
            const double now = (double)s.seen / rate;
            if (opk > 1.0f) { g = __fdiv_rn(0.99f, pk); s.last_strong = now; }
            else if (opk > __fmul_rn(target, 0.75f)) s.last_strong = now;
            else if (now - s.last_strong > (double)4.0f) g = __fmul_rn(g, 1.0005f);
            s.gain = g;
        }
        s.seen += cnt;
        return g;
    }
};
// Chunk-table scan.  Per tile of AGC_SCAN_TILE chunks:
//  (1) the whole CTA stages the chunk table in shared memory and evaluates everything that is not state
//      dependent in parallel: the running sample counter (block prefix sum) and each chunk's sample-clock
//      time seen/rate (one double division per chunk, off the serial path);
//  (2) "passes": from the current position the CTA evaluates ALL remaining chunks of the tile in parallel under
//      the hypothesis that no data-dependent event happens (scanning: gains follow the running peak maximum —
//      a block-wide prefix max; locked: the gain stays put and last_strong follows the latest strong chunk —
//      a block-wide prefix max of chunk times) and finds the first chunk that breaks the hypothesis (lock
//      transition, ratchet, creep).  Everything before that chunk is final.  One thread then replays the
//      reference's sequential step (agc_step_at) from that chunk until a chunk passes without an event (or
//      AGC_REPLAY_MAX chunks, so that long creep phases amortise the pass), and the next pass starts there.
// Event-free stretches of any length cost one pass per tile; the results are those of the sequential loop.
constexpr int AGC_SCAN_TILE = 2048;
constexpr int AGC_SCAN_THREADS = 512;
constexpr int AGC_REPLAY_MAX = 256;
// the reference's sequential step with the chunk's sample-clock time supplied (== (double)s.seen / rate)
__device__ __forceinline__ float agc_step_at(AgcState& s, float pk, unsigned cnt, float target, float strong_thr, double now, bool& event)
{
    float g;
    event = false;
    if (!s.locked) {
        if (pk > s.peak_mem) s.peak_mem = pk;
        const float safe = (s.peak_mem < 1e-4f) ? 1e-4f : s.peak_mem;
        g = __fdiv_rn(target, safe);
        if (now > (double)2.0f) { s.locked = 1; s.gain = g; s.last_strong = now; event = true; }
    } else {
        g = s.gain;
        const float opk = __fmul_rn(pk, g);
        if (opk > 1.0f) { g = __fdiv_rn(0.99f, pk); s.last_strong = now; event = true; }
        else if (opk > strong_thr) s.last_strong = now;
        else if (now - s.last_strong > (double)4.0f) { g = __fmul_rn(g, 1.0005f); event = true; }
        s.gain = g;
    }
    s.seen += cnt;
    return g;
}
__global__ void __launch_bounds__(AGC_SCAN_THREADS) agc_digital_scan_kernel(const uint32_t* __restrict__ seg_start, unsigned nseg,
                                                                            const float* __restrict__ seg_peak, PostParams p,
                                                                            AgcState* __restrict__ st, float* __restrict__ seg_gain,
                                                                            const int* __restrict__ skip_flag)
{
    if (skip_flag && *skip_flag) return;        // the grid-wide quiet test (below) already advanced the state over this table
    __shared__ unsigned s_cnt[AGC_SCAN_TILE];
    __shared__ float s_pk[AGC_SCAN_TILE];
    __shared__ float s_gain[AGC_SCAN_TILE];
    __shared__ double s_now[AGC_SCAN_TILE];         // seen_before / rate of every chunk
    __shared__ unsigned long long s_warp_tot[AGC_SCAN_THREADS / 32];
    __shared__ double s_warp_max[AGC_SCAN_THREADS / 32];
    __shared__ AgcState s_state;
    __shared__ unsigned s_first, s_pos;
    __shared__ unsigned long long s_sum;
    __shared__ double s_upd;                        // peak memory / last_strong at the chunk before the first event
    const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_state = *st;
    __syncthreads();
    const float target = p.agc_target;
    const float strong_thr = __fmul_rn(target, 0.75f);
    constexpr int PER_THREAD = AGC_SCAN_TILE / AGC_SCAN_THREADS;
    if (!seg_gain && s_state.locked) {
        // State only (the chunks of a lower shard) and already locked: the common case is that NOTHING happens in the
        // whole table — no chunk ratchets (peak * gain <= 1) and no weak chunk comes more than 4 s after the latest strong
        // one (no creep).  That is checked for the whole table in parallel, with the doubles the sequential loop would
        // compare: every thread walks a contiguous range of chunks; sample counts and "latest strong chunk so far" cross the
        // ranges through two block scans.  If the table is quiet the gain stays and last_strong becomes the time of the
        // latest strong chunk; otherwise the tile walk below does the work.
        unsigned long long* q_tot = reinterpret_cast<unsigned long long*>(s_now);      // the tile arrays are idle here
        double* q_last = s_now + AGC_SCAN_THREADS;
        __shared__ int q_event;
        static_assert(2 * AGC_SCAN_THREADS <= AGC_SCAN_TILE, "scratch fits the chunk-time array");
        const AgcState s0 = s_state;
        const unsigned per = (nseg + AGC_SCAN_THREADS - 1) / AGC_SCAN_THREADS;
        const unsigned i0 = min(nseg, tid * per), i1 = min(nseg, i0 + per);
        unsigned long long mine = 0;
        for (unsigned i = i0; i < i1; i++) mine += __ldg(seg_start + i + 1) - __ldg(seg_start + i);
        q_tot[tid] = mine;
        if (tid == 0) q_event = 0;
        __syncthreads();
        for (unsigned d = 1; d < AGC_SCAN_THREADS; d <<= 1) {             // inclusive scan of the range totals
            const unsigned long long v = (tid >= d) ? q_tot[tid - d] : 0ull;
            __syncthreads();
            q_tot[tid] += v;
            __syncthreads();
        }
        unsigned long long seen = s0.seen + q_tot[tid] - mine;            // samples seen before this thread's first chunk
        bool event = false;
        double local_last = -1.0;                                         // time of the latest strong chunk inside the range
        double weak_before = -1.0;                                        // time of the last weak chunk in front of the first strong one
        for (unsigned i = i0; i < i1; i++) {
            const unsigned c = __ldg(seg_start + i + 1) - __ldg(seg_start + i);
            if (!c) continue;
            const float opk = __fmul_rn(__ldg(seg_peak + i), s0.gain);
            const double now = (double)seen / p.target_rate;
            if (opk > 1.0f) event = true;                                 // ratchet
            else if (opk > strong_thr) local_last = now;
            else if (local_last >= 0.0) { if (now - local_last > (double)4.0f) event = true; }   // creep
            else weak_before = now;
            seen += c;
        }
        q_last[tid] = local_last;
        __syncthreads();
        for (unsigned d = 1; d < AGC_SCAN_THREADS; d <<= 1) {             // inclusive max-scan of the latest strong times
            const double v = (tid >= d) ? q_last[tid - d] : -1.0;
            __syncthreads();
            q_last[tid] = fmax(q_last[tid], v);
            __syncthreads();
        }
        const double before = fmax(s0.last_strong, tid ? q_last[tid - 1] : -1.0);   // latest strong chunk in front of the range
        if (weak_before >= 0.0 && weak_before - before > (double)4.0f) event = true;
        if (event) q_event = 1;
        __syncthreads();
        if (!q_event) {
            if (tid == AGC_SCAN_THREADS - 1) {
                AgcState s = s0;
                s.seen = s0.seen + q_tot[tid];
                s.last_strong = fmax(s0.last_strong, q_last[tid]);
                *st = s;
            }
            return;
        }
    }
    for (unsigned tile0 = 0; tile0 < nseg; tile0 += AGC_SCAN_TILE) {
        const unsigned tn = min((unsigned)AGC_SCAN_TILE, nseg - tile0);
        // ---- (1) parallel part: table, exclusive prefix of the sample counter, chunk times ----
        unsigned cnt[PER_THREAD];
        float pkv[PER_THREAD];
        double nowv[PER_THREAD];
        unsigned long long run = 0;
#pragma unroll
        for (int k = 0; k < PER_THREAD; k++) {
            const unsigned i = tid * PER_THREAD + k;
            cnt[k] = (i < tn) ? (__ldg(seg_start + tile0 + i + 1) - __ldg(seg_start + tile0 + i)) : 0u;
            pkv[k] = (i < tn) ? __ldg(seg_peak + tile0 + i) : 0.f;
            if (i < tn) { s_cnt[i] = cnt[k]; s_pk[i] = pkv[k]; }
            run += cnt[k];
        }
        unsigned long long inc = run;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned long long q = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= (unsigned)d) inc += q;
        }
        if (lane == 31) s_warp_tot[warp] = inc;
        if (tid == 0) s_pos = 0;
        __syncthreads();
        // exclusive prefix over the warp totals: every warp scans the 16 totals with shuffles (no serial walk)
        unsigned long long wt = (lane < AGC_SCAN_THREADS / 32) ? s_warp_tot[lane] : 0ull;
#pragma unroll
        for (int d = 1; d < AGC_SCAN_THREADS / 32; d <<= 1) {
            const unsigned long long q = __shfl_up_sync(0xffffffffu, wt, d);
            if (lane >= (unsigned)d) wt += q;
        }
        const unsigned long long below = __shfl_sync(0xffffffffu, wt, (warp + 31) & 31);     // inclusive total of warp - 1
        const unsigned long long base = s_state.seen + (warp ? below : 0ull);
        unsigned long long seen_before = base + inc - run;
#pragma unroll
        for (int k = 0; k < PER_THREAD; k++) {
            const unsigned i = tid * PER_THREAD + k;
            nowv[k] = (double)seen_before / p.target_rate;
            if (i < tn) s_now[i] = nowv[k];
            seen_before += cnt[k];
        }
        __syncthreads();
        // ---- (2) passes ----
        for (;;) {
            const unsigned pos = s_pos;
            if (pos >= tn) break;
            const AgcState s = s_state;
            if (tid == 0) { s_first = tn; s_sum = 0ull; }
            // keys: scanning -> peak of the chunk; locked -> time of the chunk if it is "strong" at the current gain
            double key[PER_THREAD], incl[PER_THREAD];
            bool actv[PER_THREAD], strong[PER_THREAD], ratchet[PER_THREAD];
            double trun = -1.0;
#pragma unroll
            for (int k = 0; k < PER_THREAD; k++) {
                const unsigned i = tid * PER_THREAD + k;
                actv[k] = (i >= pos) && (i < tn) && (cnt[k] != 0);            // agc_apply returns on num_samples == 0
                const float opk = __fmul_rn(pkv[k], s.gain);
                ratchet[k] = actv[k] && opk > 1.0f;
                strong[k] = actv[k] && opk > strong_thr;
                key[k] = !actv[k] ? -1.0 : (s.locked ? (strong[k] ? nowv[k] : -1.0) : (double)pkv[k]);
                trun = fmax(trun, key[k]);
                incl[k] = trun;
            }
            double wv = trun;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const double q = __shfl_up_sync(0xffffffffu, wv, d);
                if (lane >= (unsigned)d) wv = fmax(wv, q);
            }
            double tex = __shfl_up_sync(0xffffffffu, wv, 1);
            if (lane == 0) tex = -1.0;
            if (lane == 31) s_warp_max[warp] = wv;
            __syncthreads();
            {   // max of the keys of all chunks before this thread's: shuffle scan over the 16 warp maxima
                double wm = (lane < AGC_SCAN_THREADS / 32) ? s_warp_max[lane] : -1.0;
#pragma unroll
                for (int d = 1; d < AGC_SCAN_THREADS / 32; d <<= 1) {
                    const double q = __shfl_up_sync(0xffffffffu, wm, d);
                    if (lane >= (unsigned)d) wm = fmax(wm, q);
                }
                const double wb = __shfl_sync(0xffffffffu, wm, (warp + 31) & 31);
                if (warp) tex = fmax(tex, wb);
            }
            float g[PER_THREAD];
            double after[PER_THREAD];                                             // state value once chunk k has been taken
            unsigned ev = tn;
#pragma unroll
            for (int k = 0; k < PER_THREAD; k++) {
                const unsigned i = tid * PER_THREAD + k;
                const double ex = (k == 0) ? tex : fmax(tex, incl[k - 1]);
                const double in = fmax(tex, incl[k]);
                bool event;
                if (!s.locked) {
                    // scanning (agc.c:117-160): gain from the running peak maximum; lock test on the time BEFORE the chunk
                    const float mem = fmaxf(s.peak_mem, (float)in);
                    const float safe = (mem < 1e-4f) ? 1e-4f : mem;
                    g[k] = __fdiv_rn(target, safe);
                    after[k] = (double)mem;
                    event = actv[k] && (nowv[k] > (double)2.0f);
                } else {
                    const double ls_excl = fmax(s.last_strong, ex);
                    const bool creep = actv[k] && !strong[k] && (nowv[k] - ls_excl > (double)4.0f);
                    g[k] = s.gain;
                    after[k] = fmax(s.last_strong, in);
                    event = ratchet[k] || creep;
                }
                if (event && i < ev) ev = i;
            }
            if (ev < tn) atomicMin(&s_first, ev);
            __syncthreads();
            const unsigned first = s_first;
            unsigned long long part = 0;
#pragma unroll
            for (int k = 0; k < PER_THREAD; k++) {
                const unsigned i = tid * PER_THREAD + k;
                if (i >= pos && i < first) {
                    s_gain[i] = actv[k] ? g[k] : 1.0f;
                    part += cnt[k];
                    if (i + 1 == first) s_upd = after[k];
                }
            }
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) part += __shfl_xor_sync(0xffffffffu, part, d);
            if (lane == 0 && part) atomicAdd(&s_sum, part);
            __syncthreads();
            if (tid == 0) {
                AgcState t = s;
                if (first > pos) {
                    t.seen += s_sum;
                    if (!t.locked) t.peak_mem = (float)s_upd; else t.last_strong = s_upd;
                }
                // sequential replay from the first event until a chunk passes without one
                unsigned k = first, done = 0;
                while (k < tn) {
                    const unsigned ck = s_cnt[k];
                    if (ck == 0) { s_gain[k] = 1.0f; k++; continue; }
                    bool event;
                    s_gain[k] = agc_step_at(t, s_pk[k], ck, target, strong_thr, s_now[k], event);
                    k++;
                    if (!event || ++done >= AGC_REPLAY_MAX) break;
                }
                s_state = t;
                s_pos = k;
            }
            __syncthreads();
        }
        if (seg_gain)                                     // null: only the state is wanted (chunks of a lower shard)
            for (unsigned i = tid; i < tn; i += AGC_SCAN_THREADS) seg_gain[tile0 + i] = s_gain[i];
        __syncthreads();
    }
    if (tid == 0) *st = s_state;
}

// liquid agc_crcf_execute_block (agc.c:92-100): a nonlinear per-sample recurrence in (g, y2').
//
// Time-parallel evaluation that is bit-identical to the serial loop.  The stream is cut into
// blocks of B samples, one thread per block.  Every thread runs the serial recurrence over its
// block from a guessed start state and publishes its end state; then every block takes its
// predecessor's end state as its new start state, and only blocks whose start state changed run
// again.  Block 0 always starts from the carried (exact) state, so a sweep in which NO start
// state changes is a fixed point in which, by induction over the blocks, every block ran from
// the exact state: the outputs equal those of the sequential loop bit for bit.  Because the AGC
// loop forgets its state with time constant 1/alpha samples, the fixed point is reached after
// about 1 + 17/(alpha B) sweeps instead of one sweep per block.
// log(y) and exp(t) in double with short dependency chains (the recurrence is latency bound: one thread
// walks its block sample by sample).  Both are accurate to ~1 ulp of double, so rounding them to float
// gives the correctly rounded logf/expf result (checked against libm on 2e7 arguments; the rounding can
// differ only when the exact value lies within 1e-15 of a float rounding boundary).
__device__ __forceinline__ double agc_exp_small(double t)   // |t| <= 0.5 (t = -alpha/2 * log(y2'), alpha <= 1e-2)
{
    double p = 1.0 / 6227020800.0;
    p = fma(p, t, 1.0 / 479001600.0); p = fma(p, t, 1.0 / 39916800.0); p = fma(p, t, 1.0 / 3628800.0);
    p = fma(p, t, 1.0 / 362880.0);    p = fma(p, t, 1.0 / 40320.0);    p = fma(p, t, 1.0 / 5040.0);
    p = fma(p, t, 1.0 / 720.0);       p = fma(p, t, 1.0 / 120.0);      p = fma(p, t, 1.0 / 24.0);
    p = fma(p, t, 1.0 / 6.0);         p = fma(p, t, 0.5);              p = fma(p, t, 1.0);
    return fma(p, t, 1.0);
}

__constant__ AgcLogEntry agc_log_tab_c[AGC_LOG_N];
__constant__ double agc_coef_c[AGC_NCOEF] = AGC_COEF_LIST;

// The recurrence's loop-carried state: g, y2' and y2' once more as a double (its exact value: the next step needs it
// widened, and widening right after the rounding keeps that conversion off the critical path).
struct AgcRec { float g, y2p; double y2pd; };

// exact float -> double by integer arithmetic for a NORMAL float (any sign): 2 dependent ALU steps instead of a trip through
// the conversion unit (F2F: ~19 cycles on B200, tools/ubench/dlat.cu); the callers check normality themselves
__device__ __forceinline__ double agc_normal_f2d(unsigned bits)
{
    const unsigned mag = bits & 0x7fffffffu;
    return __hiloint2double((int)(((mag >> 3) + 0x38000000u) | (bits & 0x80000000u)), (int)(mag << 29));
}

// generic step (any operand: zero / subnormal / huge): the rare fall-back of agc_rms_step, kept out of line.
// V: one instance per kernel (0: agc_rms_parallel_kernel, 1: agc_rms_resume_kernel).  An out-of-line function shared by two
// kernels is compiled for both callers, and the parallel kernel then re-derives the table's shared-window address in its loop.
template <int V>
__device__ __noinline__ AgcRec agc_rms_step_slow(float ay2, float mha, double oma, const AgcLogEntry* __restrict__ ltab, AgcRec r)
{
    const float y2n = (float)fma(oma, r.y2pd, (double)ay2);
    float gn = r.g;
    if (y2n > 1e-6f) {
        const float lf = (float)agc_log_fast(y2n, ltab, agc_coef_c);
        const float tt = __fmul_rn(mha, lf);
        float ex;
        if (fabsf(tt) <= 0.125f) ex = (float)agc_exp_tiny((double)tt, agc_coef_c);
        else ex = (fabsf(tt) <= 0.5f) ? (float)agc_exp_small((double)tt) : (float)exp((double)tt);
        gn = __fmul_rn(gn, ex);
    }
    if (gn > 1e6f) gn = 1e6f;
    r.g = gn; r.y2p = y2n; r.y2pd = (double)y2n;
    return r;
}

// One sample of liquid's agc_crcf_execute (reference src/agc.c:92-100).  The recurrence is ONE dependent chain per block
// of the stream, so the step is written for latency: straight-line code for the operand ranges that occur (everything
// normal, y2' > 1e-6, |t| <= 0.125), conversions by integer arithmetic where they are exact, the three range checks folded
// into one predicate that is tested once at the end and sends the rare other cases through agc_rms_step_slow.
template <int V>
__device__ __forceinline__ float2 agc_rms_step(float2 v, size_t i, const PostParams& p, const float* __restrict__ lut,
                                               const AgcLogEntry* __restrict__ ltab, uint32_t ltab_s,
                                               float alpha, double oma, float mha, AgcRec& r)
{
    if (p.nco_enable) v = nco_mix(v, p.nco_theta0 + (uint32_t)i * p.nco_dtheta, p.nco_sign, lut);
    const float yr = __fmul_rn(v.x, r.g), yi = __fmul_rn(v.y, r.g);
    const float y2 = __fadd_rn(__fmul_rn(yr, yr), __fmul_rn(yi, yi));
    const float ay2 = __fmul_rn(alpha, y2);
    const unsigned ab = __float_as_uint(ay2);
    const bool ok_a = (ab - 0x00800000u) < 0x7f000000u;                      // positive normal
    const float y2n = (float)fma(oma, r.y2pd, agc_normal_f2d(ab));            // (1 - alpha) y2' + alpha y2, rounded to float
    const unsigned yb = __float_as_uint(y2n);
    // logf(y2n), agc_math.h (table through its shared-window address)
    const float lf = (float)agc_log_fast(y2n, ltab_s, agc_coef_c);
    const float tt = __fmul_rn(mha, lf);
    const unsigned tb = __float_as_uint(tt);
    const bool ok_t = ((tb & 0x7fffffffu) - 0x00800000u) <= (0x3e000000u - 0x00800000u);   // 2^-126 <= |t| <= 0.125
    const float ex = (float)agc_exp_tiny(agc_normal_f2d(tb), agc_coef_c);
    float gn = __fmul_rn(r.g, ex);
    if (gn > 1e6f) gn = 1e6f;
    if (ok_a && ok_t && y2n > 1e-6f) {
        r.g = gn; r.y2p = y2n; r.y2pd = agc_normal_f2d(yb);
    } else {
        r = agc_rms_step_slow<V>(ay2, mha, oma, ltab, r);
    }
    return make_float2(yr, yi);
}

// one block of the recurrence.  Samples are fetched eight at a time, one group AHEAD of the serial chain (a thread's samples
// are contiguous, lanes are a whole block apart: every group is a DRAM access of its own, ~1 us — hidden behind the ~2000
// cycles the chain spends on the previous group).
// Checkpoints: every AGC_CK samples the state (g, y2') is compared with / written to the block's checkpoint row.  A block
// that is run AGAIN (its start state changed) stops as soon as its state equals the one its previous run had at the same
// sample: from there on the two trajectories are the same bits, so the outputs and the end state already in memory stand.
// Returns true when the run stopped that way.
__device__ __forceinline__ void ld_global_nc_256(const float2* p, float2& a, float2& b, float2& c, float2& d)
{
    asm volatile("ld.global.nc.v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=f"(a.x), "=f"(a.y), "=f"(b.x), "=f"(b.y), "=f"(c.x), "=f"(c.y), "=f"(d.x), "=f"(d.y) : "l"(p));
}
__device__ __forceinline__ void st_global_256(float2* p, float2 a, float2 b, float2 c, float2 d)
{
    asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 :: "l"(p), "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y), "f"(d.x), "f"(d.y) : "memory");
}
constexpr int AGC_CK = 256;
template <int V = 0>
__device__ __forceinline__ bool agc_rms_block(const float2* __restrict__ x, size_t i0, size_t i1, const PostParams& p,
                                              const float* __restrict__ lut, const AgcLogEntry* __restrict__ ltab,
                                              float& g, float& y2p, float2* __restrict__ y, float2* __restrict__ ck, bool compare,
                                              uint32_t opaque_zero)
{
    const float alpha = p.agc_alpha;
    const double oma = 1.0 - (double)alpha;
    const float mha = __fmul_rn(-0.5f, alpha);
    AgcRec r{g, y2p, (double)y2p};
    // the table's shared-window address in a plain register: `opaque_zero` (a run-time 0 the compiler cannot see through)
    // keeps ptxas from re-deriving it as CTA-window base + offset — S2UR + ULEA in front of the load in every step
    uint32_t ltab_s = (uint32_t)__cvta_generic_to_shared(ltab) + opaque_zero;
    size_t i = i0;
    float2 nx[8];
    // A lane's samples are contiguous and the lanes of a warp are a whole block apart, so every global access of the warp
    // touches 32 different sectors.  As 64-bit accesses that was 64 LSU wavefronts per sample and warp, issued in bursts of
    // eight loads / eight stores — and the step's one shared-memory load (the log table, ON the dependent chain) queued
    // behind them: 190 cycles of the 660 per sample (profiles/r02i_agc_rms_full_cfg4.md, short-scoreboard samples at the
    // DFMA behind the LDS).  256-bit accesses (LDG.E.256 / STG.E.256, sm_100) need four instructions per group of eight.
    const bool wide = (((reinterpret_cast<size_t>(x + i0) | reinterpret_cast<size_t>(y + i0)) & 31) == 0);
    auto load8 = [&](size_t at) {
        if (wide) {
            ld_global_nc_256(x + at, nx[0], nx[1], nx[2], nx[3]);
            ld_global_nc_256(x + at + 4, nx[4], nx[5], nx[6], nx[7]);
        } else {
#pragma unroll
            for (int k = 0; k < 8; k++) nx[k] = x[at + k];
        }
    };
    if (i + 8 <= i1) load8(i);
    for (; i + 8 <= i1; i += 8) {
        if (((i - i0) & (AGC_CK - 1)) == 0) {
            float2* c = ck + ((i - i0) / AGC_CK);
            if (compare) {
                const float2 o = *c;
                if (__float_as_uint(o.x) == __float_as_uint(r.g) && __float_as_uint(o.y) == __float_as_uint(r.y2p)) return true;
            }
            *c = make_float2(r.g, r.y2p);
        }
        float2 v[8];
#pragma unroll
        for (int k = 0; k < 8; k++) v[k] = nx[k];
        if (i + 16 <= i1) load8(i + 8);
#pragma unroll
        for (int k = 0; k < 8; k++) v[k] = agc_rms_step<V>(v[k], i + k, p, lut, ltab, ltab_s, alpha, oma, mha, r);
        if (wide) {
            st_global_256(y + i, v[0], v[1], v[2], v[3]);
            st_global_256(y + i + 4, v[4], v[5], v[6], v[7]);
        } else {
#pragma unroll
            for (int k = 0; k < 8; k++) y[i + k] = v[k];
        }
    }
    for (; i < i1; i++) y[i] = agc_rms_step<V>(x[i], i, p, lut, ltab, ltab_s, alpha, oma, mha, r);
    g = r.g; y2p = r.y2p;
    return false;
}

constexpr int AGC_RMS_THREADS = 128;
__global__ void __launch_bounds__(AGC_RMS_THREADS) agc_rms_parallel_kernel(const float2* __restrict__ x, size_t n, PostParams p,
                                                                            AgcState* __restrict__ st, float2* __restrict__ y,
                                                                            size_t B, unsigned nblocks, float2* __restrict__ fin,
                                                                            unsigned* __restrict__ flags, float2* __restrict__ ckpt,
                                                                            unsigned ck_per_block)
{
    cg::grid_group grid = cg::this_grid();
    __shared__ float lut[1024];
    __shared__ AgcLogEntry ltab[AGC_LOG_N];
    if (p.nco_enable)
        for (int i = threadIdx.x; i < 1024; i += blockDim.x) lut[i] = p.nco_table[i];
    for (int i = threadIdx.x; i < AGC_LOG_N; i += blockDim.x) ltab[i] = agc_log_tab_c[i];
    __syncthreads();
    const unsigned b = blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = b < nblocks;
    const size_t i0 = (size_t)b * B, i1 = (i0 + B < n) ? i0 + B : n;
    const float2 carried = make_float2(st->rms_g, st->rms_y2);
    float2 start = carried;            // block 0: exact; others: first guess
    float2* ck = ckpt + (size_t)b * ck_per_block;
    bool run = true;
    for (unsigned it = 0; it <= nblocks; it++) {
        if (active && run) {
            float g = start.x, y2p = start.y;
            const bool merged = agc_rms_block(x, i0, i1, p, lut, ltab, g, y2p, y, ck, it > 0, (uint32_t)(B >> 48));
            if (!merged) fin[b] = make_float2(g, y2p);
        }
        grid.sync();
        run = false;
        if (active && b > 0) {
            const float2 ns = fin[b - 1];
            run = (__float_as_uint(ns.x) != __float_as_uint(start.x)) || (__float_as_uint(ns.y) != __float_as_uint(start.y));
            start = ns;
        }
        if (run) flags[it] = 1u;
        grid.sync();
        if (flags[it] == 0u) {         // no start state changed anywhere: fixed point
            if (b == 0) flags[nblocks + 1] = it + 1;   // sweeps used (diagnostics)
            break;
        }
    }
    if (b == nblocks - 1) { const float2 f = fin[b]; st->rms_g = f.x; st->rms_y2 = f.y; }
}

__device__ __forceinline__ bool same_bits(float2 a, float2 b)
{
    return __float_as_uint(a.x) == __float_as_uint(b.x) && __float_as_uint(a.y) == __float_as_uint(b.y);
}

// Resume of the last agc_rms_parallel_kernel run over the same samples from a new start state at sample `first` (a time
// shard taking over the end state of the shard in front of it).  At that run's fixed point every block's checkpoint row
// holds the exact trajectory and fin[] the block end states, so this is one more level of the same guess-and-verify
// scheme: block k (the one holding `first`) runs from `first` — a scalar head up to its next checkpoint, then the usual
// block walk comparing against the old checkpoints — and stops where the new trajectory meets the old one; a later block
// runs again only when its predecessor's end state changed (the sweep logic of the parallel kernel, blocks below k idle).
// The grid is the parallel kernel's (its occupancy sized the workspace plan): at most its 72 registers, 7 CTAs per SM.
__global__ void __launch_bounds__(AGC_RMS_THREADS, 7) agc_rms_resume_kernel(const float2* __restrict__ x, size_t n, PostParams p,
                                                                          AgcState* __restrict__ st, float2* __restrict__ y,
                                                                          size_t B, unsigned nblocks, float2* __restrict__ fin,
                                                                          unsigned* __restrict__ flags, float2* __restrict__ ckpt,
                                                                          unsigned ck_per_block, size_t first,
                                                                          const float2* __restrict__ start_state,
                                                                          AgcRmsResume* __restrict__ rr, int fresh,
                                                                          int* __restrict__ changed)
{
    cg::grid_group grid = cg::this_grid();
    __shared__ float lut[1024];
    __shared__ AgcLogEntry ltab[AGC_LOG_N];
    const unsigned b = blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned k = (unsigned)min((size_t)nblocks, first / B);
    const bool active = b < nblocks && b >= k;
    const size_t i0 = (size_t)b * B, i1 = (i0 + B < n) ? i0 + B : n;
    // everything the resume overwrites is read before the first grid-wide barrier
    const float2 s_new = *start_state;
    const bool same = !fresh && rr->valid && rr->last_first == first && same_bits(rr->last_start, s_new);
    const float2 old_end = make_float2(st->rms_g, st->rms_y2);
    float2 start = (b == k) ? s_new : (active ? fin[b - 1] : make_float2(0.f, 0.f));
    grid.sync();
    if (b == 0) { rr->last_start = s_new; rr->last_first = first; rr->valid = 1u; rr->lo = first; rr->hi = first; }
    if (same) {                        // same start as the previous resume: the trajectory in memory is already this one
        if (b == 0 && changed) *changed = 0;
        return;
    }
    if (p.nco_enable)
        for (int i = threadIdx.x; i < 1024; i += blockDim.x) lut[i] = p.nco_table[i];
    for (int i = threadIdx.x; i < AGC_LOG_N; i += blockDim.x) ltab[i] = agc_log_tab_c[i];
    __syncthreads();
    float2* ck = ckpt + (size_t)b * ck_per_block;
    const uint32_t opaque_zero = (uint32_t)(B >> 48);
    bool run = active && b == k, ran = false;
    for (unsigned it = 0; it <= nblocks; it++) {
        if (run) {
            float g = start.x, y2p = start.y;
            bool merged = false;
            // block k (it runs once): the head [first, c) up to its next checkpoint, then [c, i1); other blocks: [i0, i1).
            // One call site of the block walk: a second inlined copy would not fit the register budget above.
            size_t a = i0, c = i0;
            if (b == k) {
                a = first;
                c = i0 + (first - i0 + AGC_CK - 1) / AGC_CK * AGC_CK;
                if (c > i1) c = i1;
            }
#pragma unroll 1
            for (int part = (a < c) ? 0 : 1; part < 2 && !merged; part++) {
                const size_t s0 = part ? c : a, s1 = part ? i1 : c;
                if (s0 < s1)
                    merged = agc_rms_block<1>(x, s0, s1, p, lut, ltab, g, y2p, y, part ? ck + (c - i0) / AGC_CK : &rr->ck_scratch,
                                           part == 1, opaque_zero);
            }
            if (!merged) fin[b] = make_float2(g, y2p);
            ran = true;
        }
        grid.sync();
        run = false;
        if (active && b > k) {
            const float2 ns = fin[b - 1];
            run = !same_bits(ns, start);
            start = ns;
        }
        if (run) flags[it] = 1u;
        grid.sync();
        if (flags[it] == 0u) break;
    }
    if (ran) atomicMax(&rr->hi, (unsigned long long)i1);     // a merged run rewrote less: re-converting the rest is harmless
    if (b == nblocks - 1) {
        const float2 f = fin[b];
        st->rms_g = f.x; st->rms_y2 = f.y;
        if (changed) *changed = same_bits(f, old_end) ? 0 : 1;
    }
}

// cf32 -> output sample formats, reference sample_convert.c:40-73, 213-306
template <int FMT>
__device__ __forceinline__ void store_out(void* __restrict__ out, size_t i, float2 v)
{
    if (FMT == IQGPU_FMT_CF32) {
        reinterpret_cast<float2*>(out)[i] = v;
    } else if (FMT == IQGPU_FMT_CS16 || FMT == IQGPU_FMT_SC16Q11 || FMT == IQGPU_FMT_CS8) {
        const float S = (FMT == IQGPU_FMT_CS16) ? 32767.0f : (FMT == IQGPU_FMT_SC16Q11 ? 2048.0f : 127.0f);
        const float hi = (FMT == IQGPU_FMT_CS8) ? 127.0f : 32767.0f;
        const float lo = (FMT == IQGPU_FMT_CS8) ? -128.0f : -32768.0f;
        float a = __fmul_rn(v.x, S), b = __fmul_rn(v.y, S);
        a = (a > 0.0f) ? __fadd_rn(a, 0.5f) : __fsub_rn(a, 0.5f);
        b = (b > 0.0f) ? __fadd_rn(b, 0.5f) : __fsub_rn(b, 0.5f);
        a = (a > hi) ? hi : a; a = (a < lo) ? lo : a;
        b = (b > hi) ? hi : b; b = (b < lo) ? lo : b;
        const int ia = __float2int_rz(a), ib = __float2int_rz(b);
        if (FMT == IQGPU_FMT_CS8) reinterpret_cast<char2*>(out)[i] = make_char2((signed char)ia, (signed char)ib);
        else reinterpret_cast<short2*>(out)[i] = make_short2((short)ia, (short)ib);
    } else if (FMT == IQGPU_FMT_CU8 || FMT == IQGPU_FMT_CU16) {
        const float S = (FMT == IQGPU_FMT_CU8) ? 127.0f : 32767.0f;
        const float OFF = (FMT == IQGPU_FMT_CU8) ? 127.5f : 32767.5f;
        const float hi = (FMT == IQGPU_FMT_CU8) ? 255.0f : 65535.0f;
        float a = __fadd_rn(__fmul_rn(v.x, S), OFF), b = __fadd_rn(__fmul_rn(v.y, S), OFF);
        a = (a > hi) ? hi : a; a = (a < 0.0f) ? 0.0f : a;
        b = (b > hi) ? hi : b; b = (b < 0.0f) ? 0.0f : b;
        const unsigned ua = __float2uint_rz(__fadd_rn(a, 0.5f)), ub = __float2uint_rz(__fadd_rn(b, 0.5f));
        if (FMT == IQGPU_FMT_CU8) reinterpret_cast<uchar2*>(out)[i] = make_uchar2((unsigned char)ua, (unsigned char)ub);
        else reinterpret_cast<ushort2*>(out)[i] = make_ushort2((unsigned short)ua, (unsigned short)ub);
    } else if (FMT == IQGPU_FMT_CS24) {
        float a = __fmul_rn(v.x, 8388607.0f), b = __fmul_rn(v.y, 8388607.0f);
        int ia = __float2int_rz((a > 0.0f) ? __fadd_rn(a, 0.5f) : __fsub_rn(a, 0.5f));
        int ib = __float2int_rz((b > 0.0f) ? __fadd_rn(b, 0.5f) : __fsub_rn(b, 0.5f));
        ia = min(max(ia, -8388608), 8388607); ib = min(max(ib, -8388608), 8388607);
        unsigned char* o = reinterpret_cast<unsigned char*>(out) + i * 6;
        o[0] = ia & 0xff; o[1] = (ia >> 8) & 0xff; o[2] = (ia >> 16) & 0xff;
        o[3] = ib & 0xff; o[4] = (ib >> 8) & 0xff; o[5] = (ib >> 16) & 0xff;
    } else if (FMT == IQGPU_FMT_CS32) {
        const double hi = 2147483647.0, lo = -2147483648.0;
        double a = (double)v.x * hi, b = (double)v.y * hi;
        a = (a > 0.0) ? a + 0.5 : a - 0.5; b = (b > 0.0) ? b + 0.5 : b - 0.5;
        a = (a > hi) ? hi : a; a = (a < lo) ? lo : a;
        b = (b > hi) ? hi : b; b = (b < lo) ? lo : b;
        reinterpret_cast<int2*>(out)[i] = make_int2(__double2int_rz(a), __double2int_rz(b));
    } else if (FMT == IQGPU_FMT_CU32) {
        const double hi = 4294967295.0;
        double a = (double)v.x * 2147483647.0 + 2147483647.5, b = (double)v.y * 2147483647.0 + 2147483647.5;
        a = (a > hi) ? hi : a; a = (a < 0.0) ? 0.0 : a;
        b = (b > hi) ? hi : b; b = (b < 0.0) ? 0.0 : b;
        reinterpret_cast<uint2*>(out)[i] = make_uint2(__double2uint_rz(a + 0.5), __double2uint_rz(b + 0.5));
    }
}

// four consecutive frames -> output format; vector stores when the destination is 16-byte aligned
template <int FMT>
__device__ __forceinline__ void store_out4(void* __restrict__ out, size_t i, size_t n, const float2 (&v)[4], bool vec)
{
    if (vec && i + 4 <= n) {
        if (FMT == IQGPU_FMT_CF32) {
            float4* o = reinterpret_cast<float4*>(reinterpret_cast<float2*>(out) + i);
            o[0] = make_float4(v[0].x, v[0].y, v[1].x, v[1].y);
            o[1] = make_float4(v[2].x, v[2].y, v[3].x, v[3].y);
            return;
        }
        if (FMT == IQGPU_FMT_CS16 || FMT == IQGPU_FMT_SC16Q11 || FMT == IQGPU_FMT_CU16) {
            __align__(16) unsigned short tmp[8];
#pragma unroll
            for (int k = 0; k < 4; k++) store_out<FMT>(tmp, k, v[k]);
            *reinterpret_cast<uint4*>(reinterpret_cast<char*>(out) + i * 4) = *reinterpret_cast<const uint4*>(tmp);
            return;
        }
        if (FMT == IQGPU_FMT_CS8 || FMT == IQGPU_FMT_CU8) {
            __align__(8) unsigned char tmp[8];
#pragma unroll
            for (int k = 0; k < 4; k++) store_out<FMT>(tmp, k, v[k]);
            *reinterpret_cast<uint2*>(reinterpret_cast<char*>(out) + i * 2) = *reinterpret_cast<const uint2*>(tmp);
            return;
        }
    }
#pragma unroll
    for (int k = 0; k < 4; k++)
        if (i + k < n) store_out<FMT>(out, i + k, v[k]);
}

template <int FMT>
__global__ void __launch_bounds__(256) post_kernel(const float2* __restrict__ x, size_t n, PostParams p,
                                                   const uint32_t* __restrict__ seg_start, unsigned nseg,
                                                   const float* __restrict__ seg_gain, int nco_done,
                                                   float2* __restrict__ tap, void* __restrict__ out, bool vec_in, bool vec_out)
{
    __shared__ float lut[1024];
    const bool do_nco = p.nco_enable && !nco_done;
    if (do_nco) {
        for (int i = threadIdx.x; i < 1024; i += blockDim.x) lut[i] = p.nco_table[i];
        __syncthreads();
    }
    const int lane = threadIdx.x & 31;
    const size_t warp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const size_t nwarps = ((size_t)gridDim.x * blockDim.x) >> 5;
    const size_t ntiles = (n + POST_TILE - 1) / POST_TILE;
    for (size_t tile = warp; tile < ntiles; tile += nwarps) {
        size_t i = tile * POST_TILE + (size_t)lane * 4;
        unsigned seg = 0;
        uint32_t seg_end = 0xffffffffu;
        float g = 1.0f;
        if (seg_gain && i < n) {
            seg = find_segment(seg_start, nseg, (uint32_t)i);
            seg_end = __ldg(seg_start + seg + 1);
            g = __ldg(seg_gain + seg);
        }
#pragma unroll 1
        for (int it = 0; it < POST_TILE / 128; it++, i += 128) {
            if (i >= n) break;
            float2 v[4];
            load4(x, i, n, vec_in, v);
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const size_t ik = i + k;
                if (do_nco) v[k] = nco_mix(v[k], p.nco_theta0 + (uint32_t)ik * p.nco_dtheta, p.nco_sign, lut);
                if (seg_gain && ik < n) {
                    while ((uint32_t)ik >= seg_end) { seg++; seg_end = __ldg(seg_start + seg + 1); g = __ldg(seg_gain + seg); }
                    v[k].x = __fmul_rn(v[k].x, g); v[k].y = __fmul_rn(v[k].y, g);
                }
                if (tap && ik < n) tap[ik] = v[k];
            }
            store_out4<FMT>(out, i, n, v, vec_out);
        }
    }
}

static inline int grid_tiles(size_t n)
{
    const size_t tiles = (n + POST_TILE - 1) / POST_TILE;
    size_t blocks = (tiles + 7) / 8;            // 8 warps per CTA
    const size_t cap = 148 * 8;
    if (blocks > cap) blocks = cap;
    return (int)(blocks ? blocks : 1);
}
static inline bool aligned16(const void* p) { return (reinterpret_cast<size_t>(p) & 15) == 0; }

cudaError_t launch_agc_peaks(const float2* x, size_t n, const PostParams& p, const uint32_t* seg_start,
                             size_t nseg, float* seg_peak, cudaStream_t st)
{
    cudaError_t e = cudaMemsetAsync(seg_peak, 0, nseg * sizeof(float), st);
    if (e != cudaSuccess || n == 0) return e;
    agc_peaks_kernel<<<grid_tiles(n), 256, 0, st>>>(x, n, p, seg_start, (unsigned)nseg, seg_peak, aligned16(x));
    return cudaGetLastError();
}
// ---------------------------------------------------------------------------------------------
// Grid-wide quiet test for a STATE-ONLY advance over a long chunk table (a time shard advancing over the chunks of the
// shards below it, SURVEY 8(e)).  Once the digital AGC is locked (agc.c:165-218) a chunk changes the state only through a
// ratchet (peak * gain > 1), a creep step (weak for more than 4 s after the latest strong chunk) or by being strong
// (last_strong <- its time).  Every chunk's time follows from the closed-form table (samples before it), so whether ANY
// event happens in the table is a parallel question: part b (AGC_QUIET_PART chunks, one CTA) reports an internal event, the
// time of its latest strong chunk and the time of the last weak chunk in front of its first strong one; a single warp then
// walks the parts.  Quiet table: seen += total, last_strong <- latest strong time, and the one-CTA scan kernel is skipped
// (it used to walk the 458 752 chunks of seven lower shards in 1.03 ms on rank 7 of an 8-GPU run: the whole scaling loss of
// the cfg5 row in profiles/r02h_scale.md).  Any event, or a state that is not locked yet: the scan kernel does the work.
// ---------------------------------------------------------------------------------------------
constexpr int AGC_QUIET_PART = 4096, AGC_QUIET_THREADS = 256, AGC_QUIET_PER = AGC_QUIET_PART / AGC_QUIET_THREADS;
struct AgcQuietPart { int event; int pad; double last_strong, weak_before; };

__global__ void __launch_bounds__(AGC_QUIET_THREADS) agc_quiet_parts_kernel(const uint32_t* __restrict__ seg_start, unsigned nseg,
                                                                            const float* __restrict__ seg_peak, PostParams p,
                                                                            const AgcState* __restrict__ st, AgcQuietPart* __restrict__ parts,
                                                                            float* __restrict__ seg_gain, const int* __restrict__ done_flag)
{
    if (done_flag && *done_flag) return;        // an earlier test already settled the whole table
    __shared__ double s_last[AGC_QUIET_THREADS], s_weak[AGC_QUIET_THREADS];
    __shared__ int s_event;
    const unsigned t = threadIdx.x;
    const AgcState s0 = *st;
    const float strong_thr = __fmul_rn(p.agc_target, 0.75f);
    const unsigned i0 = min(nseg, blockIdx.x * AGC_QUIET_PART + t * AGC_QUIET_PER), i1 = min(nseg, i0 + AGC_QUIET_PER);
    if (t == 0) s_event = 0;
    bool event = false;
    double local_last = -1.0, weak_before = -1.0;
    const uint32_t base = __ldg(seg_start);
    for (unsigned i = i0; i < i1; i++) {
        const uint32_t a = __ldg(seg_start + i), b = __ldg(seg_start + i + 1);
        // the gains of a quiet table (the scan kernel rewrites every entry if the table is not quiet after all)
        if (seg_gain) seg_gain[i] = (b == a) ? 1.0f : s0.gain;
        if (b == a) continue;                                          // agc_apply returns on an empty chunk (agc.c:89)
        const float opk = __fmul_rn(__ldg(seg_peak + i), s0.gain);
        const double now = (double)(s0.seen + (unsigned long long)(uint32_t)(a - base)) / p.target_rate;
        if (opk > 1.0f) event = true;
        else if (opk > strong_thr) local_last = now;
        else if (local_last >= 0.0) { if (now - local_last > (double)4.0f) event = true; }
        else weak_before = now;
    }
    s_last[t] = local_last; s_weak[t] = weak_before;
    __syncthreads();
    if (event) s_event = 1;
    // latest strong chunk of the part in front of this thread's range (serial look-back is fine: 256 entries in shared memory,
    // and almost always the very first neighbour is strong)
    double before = -1.0;
    for (int k = (int)t - 1; k >= 0 && before < 0.0; k--) before = s_last[k];
    if (before >= 0.0 && weak_before >= 0.0 && weak_before - before > (double)4.0f) s_event = 1;
    __syncthreads();
    if (t == 0) {
        double last = -1.0, weak = -1.0;
        bool seen_strong = false;
        for (int k = 0; k < AGC_QUIET_THREADS; k++) {
            if (!seen_strong && s_weak[k] > weak) weak = s_weak[k];    // weak chunks in front of the part's first strong one
            if (s_last[k] >= 0.0) { seen_strong = true; last = s_last[k]; }
        }
        parts[blockIdx.x] = AgcQuietPart{s_event, 0, last, weak};
    }
}

__global__ void agc_quiet_finish_kernel(const AgcQuietPart* __restrict__ parts, unsigned nparts, const uint32_t* __restrict__ seg_start,
                                        unsigned nseg, AgcState* __restrict__ st, int* __restrict__ quiet_flag,
                                        const int* __restrict__ done_flag)
{
    if (threadIdx.x) return;
    if (done_flag && *done_flag) { *quiet_flag = 1; return; }
    AgcState s = *st;
    bool event = !s.locked;
    double before = s.last_strong;
    for (unsigned b = 0; b < nparts && !event; b++) {
        const AgcQuietPart q = parts[b];
        if (q.event) event = true;
        else if (q.weak_before >= 0.0 && q.weak_before - before > (double)4.0f) event = true;
        if (q.last_strong > before) before = q.last_strong;
    }
    if (!event) {
        s.seen += (unsigned long long)(uint32_t)(seg_start[nseg] - seg_start[0]);
        s.last_strong = before;
        *st = s;
    }
    *quiet_flag = event ? 0 : 1;
}

size_t agc_quiet_workspace_bytes(size_t nseg) { return ((nseg + AGC_QUIET_PART - 1) / AGC_QUIET_PART + 2) * sizeof(AgcQuietPart) + 32; }

// A table that is not quiet as a whole is usually not quiet because of its HEAD: a stream starts with the AGC's scanning
// phase and its lock (2 s of signal, agc.c:117-160), after which nothing happens for a long time.  So the table is asked
// twice: as a whole, and — if that fails — again behind a head of AGC_HEAD chunks that the scan kernel walks first.  All of
// it is queued unconditionally; flags in device memory turn the kernels that have nothing left to do into no-ops.
constexpr size_t AGC_HEAD = 8192;
cudaError_t launch_agc_digital_scan(const uint32_t* seg_start, size_t nseg, const float* seg_peak,
                                    const PostParams& p, AgcState* state, float* seg_gain, cudaStream_t st, void* quiet_ws)
{
    if (nseg == 0) return cudaSuccess;
    // the test itself costs two launches (~25 us): worth it for a state-only advance (its tables are long and mostly quiet)
    // and for tables the one-CTA scan would need more than a few tiles for (cfg1's 7324 chunks: 18 us of scan)
    if (!(quiet_ws && nseg >= (seg_gain ? 2 * AGC_HEAD : 1024))) {
        agc_digital_scan_kernel<<<1, AGC_SCAN_THREADS, 0, st>>>(seg_start, (unsigned)nseg, seg_peak, p, state, seg_gain, nullptr);
        return cudaGetLastError();
    }
    // (with gains too: a locked AGC in which nothing happens applies its one gain to every non-empty chunk)
    int* flag_all = reinterpret_cast<int*>(quiet_ws);
    int* flag_rest = flag_all + 4;
    AgcQuietPart* parts = reinterpret_cast<AgcQuietPart*>(reinterpret_cast<char*>(quiet_ws) + 32);
    const unsigned nparts = (unsigned)((nseg + AGC_QUIET_PART - 1) / AGC_QUIET_PART);
    agc_quiet_parts_kernel<<<nparts, AGC_QUIET_THREADS, 0, st>>>(seg_start, (unsigned)nseg, seg_peak, p, state, parts, seg_gain, nullptr);
    agc_quiet_finish_kernel<<<1, 32, 0, st>>>(parts, nparts, seg_start, (unsigned)nseg, state, flag_all, nullptr);
    // (a state-only advance comes in pieces that the caller already cut at the lock point, iq_tool_b200/shard.py)
    const size_t head = (seg_gain && nseg >= 3 * AGC_HEAD) ? AGC_HEAD : nseg;
    agc_digital_scan_kernel<<<1, AGC_SCAN_THREADS, 0, st>>>(seg_start, (unsigned)head, seg_peak, p, state, seg_gain, flag_all);
    if (head < nseg) {
        const size_t rest = nseg - head;
        const unsigned rparts = (unsigned)((rest + AGC_QUIET_PART - 1) / AGC_QUIET_PART);
        float* rest_gain = seg_gain ? seg_gain + head : nullptr;
        agc_quiet_parts_kernel<<<rparts, AGC_QUIET_THREADS, 0, st>>>(seg_start + head, (unsigned)rest, seg_peak + head, p, state, parts,
                                                                     rest_gain, flag_all);
        agc_quiet_finish_kernel<<<1, 32, 0, st>>>(parts, rparts, seg_start + head, (unsigned)rest, state, flag_rest, flag_all);
        agc_digital_scan_kernel<<<1, AGC_SCAN_THREADS, 0, st>>>(seg_start + head, (unsigned)rest, seg_peak + head, p, state, rest_gain,
                                                                flag_rest);
    }
    return cudaGetLastError();
}
// co-resident thread budget of the cooperative RMS-AGC kernel on the current device
static unsigned agc_rms_max_threads()
{
    static int cached[64] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && cached[dev]) return (unsigned)cached[dev];
    int per_sm = 0, sms = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, agc_rms_parallel_kernel, AGC_RMS_THREADS, 0);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    int t = std::max(1, per_sm) * std::max(1, sms) * AGC_RMS_THREADS;
    if (dev >= 0 && dev < 64) cached[dev] = t;
    return (unsigned)t;
}
static void agc_rms_plan(size_t n, float alpha, size_t& B, unsigned& nblocks)
{
    const unsigned tmax = agc_rms_max_threads();
    B = (n + tmax - 1) / tmax;
    // The loop forgets a wrong start state with time constant 2/alpha samples (|eigenvalue| = 1 - alpha/2).  With
    // blocks of ~20 time constants the second sweep already starts every block within ~e^-20 of the truth, so two
    // or three full sweeps plus a short tail of partial ones reach the fixed point; shorter blocks need one full
    // sweep per block length of convergence (measured: 25 sweeps at 493 samples, alpha = 1e-2).
    static const double tc = getenv("IQGPU_AGC_BLOCK_TC") ? atof(getenv("IQGPU_AGC_BLOCK_TC")) : 30.0;     // measured on cfg4: 40 -> 3.65 ms, 30 -> 3.51, 20 -> 3.79, 10 -> 4.82
    const size_t floorB = (size_t)std::min(65536.0, std::max(256.0, tc / std::max((double)alpha, 1e-6)));
    if (B < floorB) B = floorB;
    B = (B + 3) & ~(size_t)3;           // whole 32-byte groups per block: the 256-bit accesses of agc_rms_block stay aligned
    nblocks = (unsigned)((n + B - 1) / B);
}
size_t agc_rms_workspace_bytes(size_t n, float alpha)
{
    size_t B; unsigned nb;
    agc_rms_plan(n, alpha, B, nb);
    const size_t ckb = (B + AGC_CK - 1) / AGC_CK;
    // end states, sweep flags (rounded up so that the checkpoint rows stay 8-byte aligned), checkpoint rows
    return (size_t)nb * sizeof(float2) + (((size_t)nb + 2 + 1) & ~(size_t)1) * sizeof(unsigned) + (size_t)nb * ckb * sizeof(float2);
}
cudaError_t launch_agc_rms(const float2* x, size_t n, const PostParams& p, AgcState* state, float2* y, void* ws,
                           cudaStream_t st)
{
    if (n == 0) return cudaSuccess;
    {   // the log table, once per device
        static bool up[64] = {false};
        int dev = 0;
        cudaGetDevice(&dev);
        if (dev < 0 || dev >= 64 || !up[dev]) {
            AgcLogEntry tab[AGC_LOG_N];
            agc_log_table(tab);
            cudaError_t e0 = cudaMemcpyToSymbolAsync(agc_log_tab_c, tab, sizeof(tab), 0, cudaMemcpyHostToDevice, st);
            if (e0 != cudaSuccess) return e0;
            e0 = cudaStreamSynchronize(st);          // `tab` is on this stack frame
            if (e0 != cudaSuccess) return e0;
            if (dev >= 0 && dev < 64) up[dev] = true;
        }
    }
    size_t B; unsigned nb;
    agc_rms_plan(n, p.agc_alpha, B, nb);
    float2* fin = reinterpret_cast<float2*>(ws);
    unsigned* flags = reinterpret_cast<unsigned*>(fin + nb);
    cudaError_t e = cudaMemsetAsync(flags, 0, ((size_t)nb + 2) * sizeof(unsigned), st);
    if (e != cudaSuccess) return e;
    PostParams pp = p;
    float2* ckpt = reinterpret_cast<float2*>(flags + (((size_t)nb + 2 + 1) & ~(size_t)1));
    unsigned ckb = (unsigned)((B + AGC_CK - 1) / AGC_CK);
    void* args[] = {(void*)&x, (void*)&n, (void*)&pp, (void*)&state, (void*)&y, (void*)&B, (void*)&nb, (void*)&fin, (void*)&flags,
                    (void*)&ckpt, (void*)&ckb};
    const unsigned grid = (nb + AGC_RMS_THREADS - 1) / AGC_RMS_THREADS;
    e = cudaLaunchCooperativeKernel((void*)agc_rms_parallel_kernel, dim3(grid), dim3(AGC_RMS_THREADS), args, 0, st);
    if (e == cudaSuccess && getenv("IQGPU_DEBUG_AGC")) {
        unsigned sweeps = 0;
        cudaStreamSynchronize(st);
        cudaMemcpy(&sweeps, flags + nb + 1, sizeof(unsigned), cudaMemcpyDeviceToHost);
        fprintf(stderr, "[iqgpu] rms agc: n=%zu alpha=%g block=%zu blocks=%u sweeps=%u\n", n, (double)p.agc_alpha, B, nb, sweeps);
    }
    return e;
}
cudaError_t launch_post(const float2* x, size_t n, const PostParams& p, const uint32_t* seg_start, size_t nseg,
                        const float* seg_gain, int nco_done, float2* tap, void* out, cudaStream_t st)
{
    if (n == 0) return cudaSuccess;
    const int grid = grid_tiles(n);
    const bool vi = aligned16(x), vo = aligned16(out);
#define CALL(F) post_kernel<F><<<grid, 256, 0, st>>>(x, n, p, seg_start, (unsigned)nseg, seg_gain, nco_done, tap, out, vi, vo)
    DISPATCH_FMT(p.format, CALL)
#undef CALL
    return cudaGetLastError();
}
cudaError_t launch_agc_rms_resume(const float2* x, size_t n, const PostParams& p, AgcState* state, float2* y, void* ws,
                                  size_t first, const float2* start, AgcRmsResume* rr, bool fresh, int* changed,
                                  cudaStream_t st)
{
    if (n == 0 || first >= n) return cudaErrorInvalidValue;
    size_t B; unsigned nb;
    agc_rms_plan(n, p.agc_alpha, B, nb);        // the plan of the call being resumed: its workspace layout
    float2* fin = reinterpret_cast<float2*>(ws);
    unsigned* flags = reinterpret_cast<unsigned*>(fin + nb);
    cudaError_t e = cudaMemsetAsync(flags, 0, ((size_t)nb + 2) * sizeof(unsigned), st);
    if (e != cudaSuccess) return e;
    PostParams pp = p;
    float2* ckpt = reinterpret_cast<float2*>(flags + (((size_t)nb + 2 + 1) & ~(size_t)1));
    unsigned ckb = (unsigned)((B + AGC_CK - 1) / AGC_CK);
    int fr = fresh ? 1 : 0;
    void* args[] = {(void*)&x, (void*)&n, (void*)&pp, (void*)&state, (void*)&y, (void*)&B, (void*)&nb, (void*)&fin, (void*)&flags,
                    (void*)&ckpt, (void*)&ckb, (void*)&first, (void*)&start, (void*)&rr, (void*)&fr, (void*)&changed};
    const unsigned grid = (nb + AGC_RMS_THREADS - 1) / AGC_RMS_THREADS;
    return cudaLaunchCooperativeKernel((void*)agc_rms_resume_kernel, dim3(grid), dim3(AGC_RMS_THREADS), args, 0, st);
}

template <int FMT>
__global__ void __launch_bounds__(256) convert_range_kernel(const float2* __restrict__ y, const AgcRmsResume* __restrict__ rr,
                                                            void* __restrict__ out, bool vec_out)
{
    const size_t lo = rr->lo, hi = rr->hi;
    if (lo >= hi) return;
    // from the group of four holding `lo`: the frames in front of it are converted again to the same bits
    const size_t stride = (size_t)gridDim.x * blockDim.x * 4;
    for (size_t i = (lo & ~(size_t)3) + ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 4; i < hi; i += stride) {
        float2 v[4];
#pragma unroll
        for (int k = 0; k < 4; k++) v[k] = (i + k < hi) ? y[i + k] : make_float2(0.f, 0.f);
        store_out4<FMT>(out, i, hi, v, vec_out);
    }
}

cudaError_t launch_convert_range(const float2* y, const AgcRmsResume* rr, int format, void* out, cudaStream_t st)
{
    // a fixed grid striding over a range only the device knows; an unchanged resume leaves it empty (a few us)
    const int grid = 148 * 2;
    const bool vo = aligned16(out);
#define CALL(F) convert_range_kernel<F><<<grid, 256, 0, st>>>(y, rr, out, vo)
    DISPATCH_FMT(format, CALL)
#undef CALL
    return cudaGetLastError();
}

cudaError_t launch_convert_out(const float2* x, size_t n, int format, void* out, cudaStream_t st)
{
    PostParams p{};
    p.format = format;
    return launch_post(x, n, p, nullptr, 0, nullptr, 1, nullptr, out, st);
}

}  // namespace iqgpu
