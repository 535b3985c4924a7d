// fft_filter.cu — K4: FFT block filter, a cuFFT-free hand-written power-of-two FFT.
//
// Replaces liquid's fftfilt_crcf/cccf_execute as driven by the reference
// (src/filter.c:464-526: `_execute_fft_filter_pass` runs one fftfilt_*_execute per whole block of
// n frames; liquid's object is overlap-ADD with a carried tail w[n], FFT size 2n).  Here each
// block is evaluated in the equivalent overlap-SAVE form, which has no carried state and so lets
// every block of a train run in parallel:
//
//     window_b = x[(b-1) n .. (b+1) n)            (the n frames before block b and block b itself)
//     y[b n .. (b+1) n) = last n samples of IFFT( FFT(window_b) .* H ) / (2n),   H = FFT(h || 0)
//
// One CTA owns one 2n-point transform, resident in shared memory (2n <= 16384 -> 128 KB):
// radix-4 decimation-in-frequency forward (digit-reversed spectrum), multiply by H stored in the
// same digit-reversed order, conjugate-transposed network back (fft_core.cuh).  2n > 16384 is
// split: radix-2 DIF stages over a global scratch down to 16384-point sub-blocks, the shared
// memory kernel on each sub-block, radix-2 DIT stages back up.
#include <algorithm>
#include <cstdio>
#include <cmath>

#include "fft_core.cuh"
#include "fft_filter2.cuh"
#include "kernels.hpp"

namespace iqgpu {

using namespace fftcore;

constexpr unsigned FFT_SMEM_MAX = 16384;   // points per CTA-resident transform
constexpr unsigned FFT_MAX_POINTS = 1u << 21;

enum { FFT_WINDOW = 1, FFT_FWD = 2, FFT_MULH = 4, FFT_INV = 8 };

// src/dst: WINDOW mode: src -> first frame of block 0 (history below), dst -> y of block 0.
//          otherwise: contiguous M-point sub-blocks of N-point transforms, src may equal dst.
__global__ void __launch_bounds__(1024) fft_smem_kernel(const float2* __restrict__ src, float2* __restrict__ dst,
                                                        unsigned M, unsigned N, unsigned B,
                                                        const float2* __restrict__ tw, const float2* __restrict__ H,
                                                        int flags, float scale)
{
    extern __shared__ __align__(16) float2 buf[];
    const unsigned tid = threadIdx.x, nt = blockDim.x;
    const size_t cb = blockIdx.x;
    if (flags & FFT_WINDOW) {
        const float2* w = src + ((long long)cb - 1) * (long long)B;
        for (unsigned i = tid; i < M; i += nt) buf[i] = w[i];
    } else {
        const float2* w = src + cb * M;
        for (unsigned i = tid; i < M; i += nt) buf[i] = w[i];
    }
    __syncthreads();
    unsigned p = 0;
    for (unsigned m = M; m > 1; m >>= 1) p++;
    const unsigned Mq = (p & 1) ? (M >> 1) : M;
    if (flags & FFT_FWD) {
        if (p & 1) {
            for (unsigned t = tid; t < M / 2; t += nt) dif2(buf, M, t, tw, N / M);
            __syncthreads();
        }
        for (unsigned L = Mq; L >= 4; L >>= 2) {
            const unsigned tws = N / L;
            for (unsigned t = tid; t < M / 4; t += nt) dif4(buf, L, t, tw, tws);
            __syncthreads();
        }
    }
    if (flags & FFT_MULH) {
        const size_t g0 = (cb * M) & (size_t)(N - 1);
        for (unsigned i = tid; i < M; i += nt) buf[i] = cmul(buf[i], __ldg(H + g0 + i));
        __syncthreads();
    }
    if (flags & FFT_INV) {
        for (unsigned L = 4; L <= Mq; L <<= 2) {
            const unsigned tws = N / L;
            for (unsigned t = tid; t < M / 4; t += nt) dit4(buf, L, t, tw, tws);
            __syncthreads();
        }
        if (p & 1) {
            for (unsigned t = tid; t < M / 2; t += nt) dit2(buf, M, t, tw, N / M);
            __syncthreads();
        }
    }
    if (flags & FFT_WINDOW) {
        float2* y = dst + cb * B;
        for (unsigned i = tid; i < B; i += nt) {
            const float2 v = buf[B + i];
            y[i] = make_float2(v.x * scale, v.y * scale);
        }
    } else {
        float2* y = dst + cb * M;
        for (unsigned i = tid; i < M; i += nt) y[i] = buf[i];
    }
}

// ---- split path (2n > FFT_SMEM_MAX): global scratch [nblocks][N] ---------------------------------
__global__ void __launch_bounds__(256) fft_gather_kernel(const float2* __restrict__ x, unsigned B, size_t total,
                                                         float2* __restrict__ scratch)
{
    // scratch[b*2B + i] = x[(b-1)B + i]
    for (size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (size_t)gridDim.x * blockDim.x)
        scratch[g] = x[(long long)g - (long long)(g / (2 * (size_t)B) + 1) * (long long)B];
}
__global__ void __launch_bounds__(256) fft_scatter_kernel(const float2* __restrict__ scratch, unsigned B, size_t total,
                                                          float scale, float2* __restrict__ y)
{
    for (size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (size_t)gridDim.x * blockDim.x) {
        const size_t b = g / B, j = g - b * B;
        const float2 v = scratch[b * 2 * (size_t)B + B + j];
        y[g] = make_float2(v.x * scale, v.y * scale);
    }
}
template <bool INVERSE>
__global__ void __launch_bounds__(256) fft_global_r2_kernel(float2* __restrict__ buf, unsigned N, unsigned L, size_t total,
                                                            const float2* __restrict__ tw)
{
    const unsigned half = N >> 1;
    for (size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (size_t)gridDim.x * blockDim.x) {
        const size_t b = g / half;
        const unsigned t = (unsigned)(g - b * half);
        if (INVERSE) dit2(buf + b * N, L, t, tw, N / L);
        else dif2(buf + b * N, L, t, tw, N / L);
    }
}

static inline int grid_for(size_t total, int threads)
{
    size_t blocks = (total + threads - 1) / threads;
    if (blocks > 148 * 16) blocks = 148 * 16;
    return (int)(blocks ? blocks : 1);
}

static bool is_pow2(unsigned v) { return v && !(v & (v - 1)); }

bool fftfilt_supported(unsigned B) { return is_pow2(B) && 2ull * B <= FFT_MAX_POINTS; }

size_t fftfilt_scratch_bytes(size_t nblocks, unsigned B)
{
    return (2 * B > FFT_SMEM_MAX) ? nblocks * 2 * (size_t)B * sizeof(float2) : 0;
}

static cudaError_t launch_smem(const float2* src, float2* dst, unsigned M, unsigned N, unsigned B, size_t ctas,
                               const float2* tw, const float2* H, int flags, float scale, cudaStream_t st)
{
    // per-device attribute; cheap enough to set on every launch
    cudaError_t ea = cudaFuncSetAttribute(fft_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)(FFT_SMEM_MAX * sizeof(float2)));
    if (ea != cudaSuccess) return ea;
    unsigned threads = M / 4;
    if (threads > 1024) threads = 1024;
    if (threads < 32) threads = 32;
    fft_smem_kernel<<<(unsigned)ctas, threads, M * sizeof(float2), st>>>(src, dst, M, N, B, tw, H, flags, scale);
    return cudaGetLastError();
}

// v2 (radix-16 register butterflies, fft_filter2.cuh) serves every transform that fits one CTA
static bool v2_capable(unsigned nfft) { return nfft >= 64 && nfft <= fft2::MAX_POINTS; }
static size_t v2_smem_bytes(unsigned nfft) { return (size_t)(fft2::pad(nfft) + 8) * sizeof(float2); }

size_t fft_twiddle_entries(unsigned nfft)
{
    size_t n = nfft;
    if (v2_capable(nfft)) {
        const fft2::Plan P = fft2::make_plan(nfft);
        unsigned L = nfft;
        for (unsigned k = 0; k < P.n16; k++, L >>= 4) n += 4 * (size_t)(L >> 4);
    }
    return n;
}
void fft_fill_twiddles(unsigned nfft, float2* host)
{
    for (unsigned k = 0; k < nfft; k++) {
        const double a = -2.0 * M_PI * (double)k / (double)nfft;
        host[k] = make_float2((float)std::cos(a), (float)std::sin(a));
    }
    if (!v2_capable(nfft)) return;
    // compact records {W_L^j, W_L^2j, W_L^4j, W_L^8j}, j < L/16, for the radix-16 passes L = nfft, nfft/16, ...:
    // copies of natural entries (same floats)
    const fft2::Plan P = fft2::make_plan(nfft);
    float2* rec = host + nfft;
    unsigned L = nfft;
    for (unsigned k = 0; k < P.n16; k++, L >>= 4) {
        const unsigned s = L >> 4, tws = nfft / L;
        for (unsigned j = 0; j < s; j++)
            for (unsigned p = 1; p <= 8; p <<= 1) *rec++ = host[(size_t)p * j * tws];
    }
}

cudaError_t launch_fft_forward(const float2* in, unsigned nfft, const float2* twiddle, float2* out, cudaStream_t st)
{
    if (!is_pow2(nfft) || nfft < 2 || nfft > FFT_MAX_POINTS) return cudaErrorInvalidValue;
    if (v2_capable(nfft)) {
        cudaError_t ea = cudaFuncSetAttribute(fft2::fft2_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                              (int)(fft2::SMEM_F2 * sizeof(float2)));
        if (ea != cudaSuccess) return ea;
        fft2::fft2_forward_kernel<<<1, fft2::THREADS, v2_smem_bytes(nfft), st>>>(in, out, nfft, twiddle);
        return cudaGetLastError();
    }
    if (nfft <= FFT_SMEM_MAX) return launch_smem(in, out, nfft, nfft, 0, 1, twiddle, nullptr, FFT_FWD, 1.f, st);
    cudaError_t e = cudaMemcpyAsync(out, in, nfft * sizeof(float2), cudaMemcpyDeviceToDevice, st);
    if (e != cudaSuccess) return e;
    for (unsigned L = nfft; L > FFT_SMEM_MAX; L >>= 1) {
        fft_global_r2_kernel<false><<<grid_for(nfft / 2, 256), 256, 0, st>>>(out, nfft, L, nfft / 2, twiddle);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    return launch_smem(out, out, FFT_SMEM_MAX, nfft, 0, nfft / FFT_SMEM_MAX, twiddle, nullptr, FFT_FWD, 1.f, st);
}

cudaError_t launch_fftfilt(const float2* x, size_t nblocks, unsigned B, const float2* H, const float2* twiddle,
                           float2* y, float2* scratch, uint32_t* launches, cudaStream_t st)
{
    if (nblocks == 0) return cudaSuccess;
    if (!fftfilt_supported(B)) return cudaErrorInvalidValue;
    const unsigned N = 2 * B;
    const float scale = 1.0f / (float)N;
    if (v2_capable(N)) {
        cudaError_t ea = cudaFuncSetAttribute(fft2::fftfilt2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                              (int)(fft2::SMEM_F2 * sizeof(float2)));
        if (ea != cudaSuccess) return ea;
        if (launches) *launches += 1;
        // CTAs resident at a time: the L2 prefetch distance of the kernel (0 = off)
        static int wave = -1;
        if (wave < 0) {
            int dev = 0, sms = 0, per_sm = 0;
            cudaGetDevice(&dev);
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fft2::fftfilt2_kernel, fft2::THREADS, v2_smem_bytes(fft2::MAX_POINTS));
            wave = std::max(1, sms * std::max(1, per_sm));
        }
        const unsigned w = (N == fft2::MAX_POINTS) ? (unsigned)wave : 0u;     // smaller transforms run several CTAs per SM
        fft2::fftfilt2_kernel<<<(unsigned)nblocks, fft2::THREADS, v2_smem_bytes(N), st>>>(x, y, N, twiddle, H, scale, w);
        return cudaGetLastError();
    }
    if (N <= FFT_SMEM_MAX) {
        if (launches) *launches += 1;
        return launch_smem(x, y, N, N, B, nblocks, twiddle, H, FFT_WINDOW | FFT_FWD | FFT_MULH | FFT_INV, scale, st);
    }
    if (!scratch) return cudaErrorInvalidValue;
    const size_t total = nblocks * (size_t)N;
    cudaError_t e;
    fft_gather_kernel<<<grid_for(total, 256), 256, 0, st>>>(x, B, total, scratch);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    uint32_t nl = 1;
    for (unsigned L = N; L > FFT_SMEM_MAX; L >>= 1, nl++) {
        fft_global_r2_kernel<false><<<grid_for(total / 2, 256), 256, 0, st>>>(scratch, N, L, total / 2, twiddle);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    e = launch_smem(scratch, scratch, FFT_SMEM_MAX, N, 0, total / FFT_SMEM_MAX, twiddle, H, FFT_FWD | FFT_MULH | FFT_INV, 1.f, st);
    if (e != cudaSuccess) return e;
    nl++;
    for (unsigned L = 2 * FFT_SMEM_MAX; L <= N && L != 0; L <<= 1, nl++) {
        fft_global_r2_kernel<true><<<grid_for(total / 2, 256), 256, 0, st>>>(scratch, N, L, total / 2, twiddle);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    fft_scatter_kernel<<<grid_for(nblocks * (size_t)B, 256), 256, 0, st>>>(scratch, B, nblocks * (size_t)B, scale, y);
    nl++;
    if (launches) *launches += nl;
    return cudaGetLastError();
}

}  // namespace iqgpu
