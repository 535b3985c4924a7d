// iq_metric.cu — K6: one optimisation pass of the I/Q-imbalance corrector on a 1024-frame block.
//
// Replaces iq_correct_run_optimization + _estimate_power + _calculate_imbalance_metric +
// _calculate_power_spectrum (reference src/iq_correct.c:154-235, 315-389): 27 windowed
// 1024-point spectra (1 power estimate, 1 baseline metric, 25 hill-climb candidates) and a 5 %
// smoothing step.  The work is tiny and strictly sequential between candidates, so ONE CTA keeps
// the block, the Hamming window, the twiddles and the spectrum in shared memory and runs all 27
// evaluations back to back; the FFT is the radix-4 network of fft_core.cuh (1024 = 4^5), whose
// base-4 digit-reversed output order is undone when the dB spectrum is written.
// The reference draws the +-1 step directions from rand() (:391) seeded with time() (:92); here
// the caller supplies them (deterministic, SURVEY quirk B7).
#include <cuda_runtime.h>

#include "../../include/iqgpu.h"
#include "cuda_owned.hpp"
#include "fft_core.cuh"
#include "kernels.hpp"

namespace iqgpu {

using namespace fftcore;

constexpr int IQ_NFFT = 1024;
constexpr int IQ_THREADS = 256;
constexpr int IQ_PASSES = 25;               // IQ_MAX_PASSES, include/constants.h:160

struct IqOptResult { float mag, phase, avg_power, power_range; int optimized; };

__device__ __forceinline__ unsigned digitrev4_1024(unsigned p)
{
    // reverse the five base-4 digits of p
    unsigned r = 0;
#pragma unroll
    for (int d = 0; d < 5; d++) { r = (r << 2) | (p & 3u); p >>= 2; }
    return r;
}

// spectrum_db[(k + 512) % 1024] = 20 log10(|X[k]| / 1024 + 1e-12), X = FFT(window * correct(x))
__device__ void iq_power_spectrum(const float2* __restrict__ x, const float* __restrict__ win, const float2* __restrict__ tw,
                                  float2* __restrict__ buf, float* __restrict__ spec, float gain_adj, float phase_adj)
{
    const int t = threadIdx.x;
    const float magp1 = __fadd_rn(1.0f, gain_adj);
    for (int i = t; i < IQ_NFFT; i += IQ_THREADS) {
        const float2 v = x[i];
        const float re = __fmul_rn(v.x, magp1);
        const float im = __fadd_rn(v.y, __fmul_rn(phase_adj, v.x));
        buf[i] = make_float2(__fmul_rn(re, win[i]), __fmul_rn(im, win[i]));
    }
    __syncthreads();
    for (unsigned L = IQ_NFFT; L >= 4; L >>= 2) {
        dif4(buf, L, (unsigned)t, tw, IQ_NFFT / L);       // 256 butterflies per stage, one per thread
        __syncthreads();
    }
    for (int p = t; p < IQ_NFFT; p += IQ_THREADS) {
        const unsigned k = digitrev4_1024((unsigned)p);
        const float2 X = buf[p];
        float mag = (float)sqrt((double)X.x * (double)X.x + (double)X.y * (double)X.y);   // cabsf
        mag = __fdiv_rn(mag, (float)IQ_NFFT);
        spec[(k + IQ_NFFT / 2) & (IQ_NFFT - 1)] = __fmul_rn(20.0f, log10f(__fadd_rn(mag, 1e-12f)));
    }
    __syncthreads();
}

// +-1 step directions of the in-chain optimiser: a counter-based generator (SURVEY quirk B7: the reference draws them from
// rand() seeded with time(); here pass number and seed decide, so a run can be repeated)
__host__ __device__ inline float iq_direction(unsigned seed, unsigned long long pass, unsigned k)
{
    unsigned long long z = ((unsigned long long)seed << 32) ^ (pass * 0x9E3779B97F4A7C15ull) ^ ((unsigned long long)k * 0xBF58476D1CE4E5B9ull);
    z ^= z >> 30; z *= 0xBF58476D1CE4E5B9ull;
    z ^= z >> 27; z *= 0x94D049BB133111EBull;
    z ^= z >> 31;
    return (z & 1ull) ? 1.0f : -1.0f;
}

struct IqShared {
    float2 x[IQ_NFFT], buf[IQ_NFFT], tw[IQ_NFFT];
    float win[IQ_NFFT], spec[IQ_NFFT];
    float metric, avg, range;
};

__device__ void iq_tables(IqShared& sh)
{
    for (int i = threadIdx.x; i < IQ_NFFT; i += IQ_THREADS) {
        float s, c;
        sincospif(-2.0f * (float)i / (float)IQ_NFFT, &s, &c);
        sh.tw[i] = make_float2(c, s);
        // iq_correct.c:121-123 Hamming window, evaluated in float like the reference
        sh.win[i] = __fsub_rn(0.54f, __fmul_rn(0.46f, cosf(__fdiv_rn(__fmul_rn(__fmul_rn(2.0f, 3.14159265358979323846f), (float)i), (float)(IQ_NFFT - 1)))));
    }
}

// one optimisation pass on the block in sh.x (iq_correct_run_optimization, :154-235).  dirs != nullptr: caller-supplied
// directions (function-level entry point); otherwise iq_direction(seed, pass_no, k).  All threads return the same result.
__device__ IqOptResult iq_pass(IqShared& sh, const float* __restrict__ dirs, unsigned seed, unsigned long long pass_no,
                               float mag_in, float phase_in)
{
    const int t = threadIdx.x;
    const int half = IQ_NFFT / 2;
    const int lo = (int)(0.05f * half), hi = (int)(0.95f * half);
    // ---- _estimate_power (:361-389)
    iq_power_spectrum(sh.x, sh.win, sh.tw, sh.buf, sh.spec, 0.0f, 0.0f);
    if (t == 0) {
        float mx = -1000.0f;
        double sum = 0.0;
        int count = 0;
        for (int i = lo; i < hi; i++) {
            const float pn = sh.spec[i], pp = sh.spec[IQ_NFFT - 1 - i];
            if (pp > mx) mx = pp;
            if (pn > mx) mx = pn;
            sum += (double)__fadd_rn(pp, pn);
            count += 2;
        }
        sh.avg = count ? (float)(sum / count) : 0.0f;
        sh.range = count ? __fsub_rn(mx, sh.avg) : 0.0f;
    }
    __syncthreads();
    const float avg = sh.avg, range = sh.range;
    if (range < 20.0f) return IqOptResult{mag_in, phase_in, avg, range, 0};   // IQ_CORRECTION_POWER_THRESHOLD_DB (:168)
    // ---- hill climb (:177-201); the metric sum runs sequentially in float like the reference
    float cur_g = mag_in, cur_p = phase_in, best = 0.f;
    for (int pass = -1; pass < IQ_PASSES; pass++) {
        float cg = cur_g, cp = cur_p;
        if (pass >= 0) {
            const float d0 = dirs ? dirs[2 * pass] : iq_direction(seed, pass_no, 2u * (unsigned)pass);
            const float d1 = dirs ? dirs[2 * pass + 1] : iq_direction(seed, pass_no, 2u * (unsigned)pass + 1u);
            cg = __fadd_rn(cur_g, __fmul_rn(0.0001f, d0));
            cp = __fadd_rn(cur_p, __fmul_rn(0.0001f, d1));
        }
        iq_power_spectrum(sh.x, sh.win, sh.tw, sh.buf, sh.spec, cg, cp);
        if (t == 0) {
            float total = 0.0f;
            for (int i = lo; i < hi; i++) {
                const float pn = sh.spec[i], pp = sh.spec[IQ_NFFT - 1 - i];
                if (pp > -80.0f || pn > -80.0f) {
                    const float d = __fsub_rn(pp, pn);
                    total = __fadd_rn(total, __fmul_rn(d, d));
                }
            }
            sh.metric = total;
        }
        __syncthreads();
        const float m = sh.metric;
        if (pass < 0) best = m;
        else if (m > best) { best = m; cur_g = cg; cur_p = cp; }   // keeps a candidate when the metric INCREASES (:196, quirk B8)
        __syncthreads();
    }
    // 5 % smoothing into the inactive slot (:206-216)
    const float sg = __fadd_rn(__fmul_rn(__fsub_rn(1.0f, 0.05f), mag_in), __fmul_rn(0.05f, cur_g));
    const float sp = __fadd_rn(__fmul_rn(__fsub_rn(1.0f, 0.05f), phase_in), __fmul_rn(0.05f, cur_p));
    return IqOptResult{sg, sp, avg, range, 1};
}

__global__ void __launch_bounds__(IQ_THREADS) iq_optimize_kernel(const float2* __restrict__ block, const float* __restrict__ dirs,
                                                                 float mag_in, float phase_in, IqOptResult* __restrict__ out)
{
    extern __shared__ __align__(16) unsigned char iq_smem[];
    IqShared& sh = *reinterpret_cast<IqShared*>(iq_smem);
    for (int i = threadIdx.x; i < IQ_NFFT; i += IQ_THREADS) sh.x[i] = block[i];
    iq_tables(sh);
    __syncthreads();
    const IqOptResult r = iq_pass(sh, dirs, 0u, 0ull, mag_in, phase_in);
    if (threadIdx.x == 0) *out = r;
}

// In-chain optimiser (SURVEY 8(f) rank 3; reference src/utility_threads.c:35-47 + src/pipeline.c:468-476): the passes of one
// train, in stream order, on the probe blocks the chain extracted (first 1024 pre-processed frames of every eligible chunk).
// The factors live in device memory; every pass starts from what the previous one left (iq_correct.c:183-186 reads the
// active slot), weak blocks leave them alone (:168-171).
__global__ void __launch_bounds__(IQ_THREADS) iq_optimize_train_kernel(const float2* __restrict__ probes, int n_probes,
                                                                       IqOptState* __restrict__ state)
{
    extern __shared__ __align__(16) unsigned char iq_smem[];
    IqShared& sh = *reinterpret_cast<IqShared*>(iq_smem);
    iq_tables(sh);
    IqOptState st = *state;
    for (int b = 0; b < n_probes; b++) {
        __syncthreads();
        for (int i = threadIdx.x; i < IQ_NFFT; i += IQ_THREADS) sh.x[i] = probes[(size_t)b * IQ_NFFT + i];
        __syncthreads();
        const IqOptResult r = iq_pass(sh, nullptr, st.seed, st.attempts, st.mag, st.phase);
        st.attempts++;
        st.avg_power = r.avg_power; st.power_range = r.power_range;
        if (r.optimized) { st.mag = r.mag; st.phase = r.phase; st.passes++; }
    }
    if (threadIdx.x == 0) *state = st;
}

cudaError_t launch_iq_optimize_train(const float2* probes, int n_probes, IqOptState* state, cudaStream_t st)
{
    if (n_probes <= 0) return cudaSuccess;
    static_assert(sizeof(IqShared) <= 48 * 1024, "fits the default dynamic shared memory limit");
    iq_optimize_train_kernel<<<1, IQ_THREADS, sizeof(IqShared), st>>>(probes, n_probes, state);
    return cudaGetLastError();
}

float iq_direction_host(unsigned seed, unsigned long long pass, unsigned k) { return iq_direction(seed, pass, k); }

cudaError_t iq_optimize_device(const float* host_block1024, const float* host_dirs50, float* mag, float* phase,
                               float* avg_power, float* power_range, int* optimized)
{
    DeviceArray<float2> d_block;
    DeviceArray<float> d_dirs;
    DeviceArray<IqOptResult> d_out;
    cudaError_t e = d_block.alloc(IQ_NFFT);
    if (e == cudaSuccess) e = d_dirs.alloc(2 * IQ_PASSES);
    if (e == cudaSuccess) e = d_out.alloc(1);
    IqOptResult r{};
    if (e == cudaSuccess) e = cudaMemcpy(d_block.data(), host_block1024, IQ_NFFT * sizeof(float2), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(d_dirs.data(), host_dirs50, 2 * IQ_PASSES * sizeof(float), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        iq_optimize_kernel<<<1, IQ_THREADS, sizeof(IqShared)>>>(d_block.data(), d_dirs.data(), *mag, *phase, d_out.data());
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpy(&r, d_out.data(), sizeof(r), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return e;
    *mag = r.mag; *phase = r.phase;
    if (avg_power) *avg_power = r.avg_power;
    if (power_range) *power_range = r.power_range;
    if (optimized) *optimized = r.optimized;
    return cudaSuccess;
}

}  // namespace iqgpu
