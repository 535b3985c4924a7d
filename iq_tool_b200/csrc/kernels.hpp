// kernels.hpp — launch interface of the sm_100a kernels (kernels.cu / fused_front.cu).
// All pointers are device pointers unless noted; every launcher enqueues on `st` and
// returns the cudaError_t of the launch.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <string>

namespace iqgpu {

// ---- K1: pre-processor (convert [+DC] [+I/Q apply] [+NCO]) ---------------------------------
struct PreParams {
    int      format;        // IQGPU_FMT_*
    float    gain;
    int      dc_enable;
    float    dc_c;          // pole
    float    dc_a;          // 1 - pole
    int      iq_enable;
    float    iq_magp1;      // 1 + mag
    float    iq_phase;
    int      nco_enable;
    uint32_t nco_theta0;    // phase of the first sample of this call
    uint32_t nco_dtheta;
    float    nco_sign;      // +1 mix up, -1 mix down
    const float* nco_table; // 1024-entry sine table (device)
};
// DC pass 1: per-run weighted sums S_r = sum_k c^(len-1-k) x[k] (converted samples)
cudaError_t launch_dc_run_sums(const void* raw, size_t n, const PreParams& p, uint32_t run_len,
                               double2* run_sums, cudaStream_t st);
// DC pass 2: v at the start of every run from the carried state; updates the carry in place
// scan_ws: device workspace of dc_scan_workspace_doubles(n_runs) doubles
// row_len: granularity the sums were zero-padded to (128 for launch_dc_run_sums rows, 512 for tick sums)
cudaError_t launch_dc_scan(const double2* run_sums, size_t n_runs, uint32_t run_len, size_t n,
                           float dc_c, double2* carry_inout, double2* run_start, double* scan_ws, cudaStream_t st,
                           uint32_t row_len = 128);
// DC pre-pass of the fused front: one weighted sum per 512-frame tick (frames below lo / beyond n read as zero)
cudaError_t launch_dc_tick_sums(const void* raw, size_t n, size_t lo, const PreParams& p, double2* sums, cudaStream_t st);
size_t dc_scan_workspace_doubles(size_t n_runs);
// convert + (DC apply) + I/Q + NCO -> cf32
cudaError_t launch_pre(const void* raw, size_t n, const PreParams& p, uint32_t run_len,
                       const double2* run_start, float2* out, cudaStream_t st);

// DC blocker with the reference's fp32 state rounding (liquid iirfilt_crcf, direct form II), serial, in place on a cf32
// stream; state = v0 {re, im} carried across calls (device memory)
cudaError_t launch_dc_reference(float2* x, size_t n, float dc_c, float2* state, cudaStream_t st);

// ---- K2: resampler building blocks (unfused) -------------------------------------------------
// x points at the stream sample with absolute index a0 (history lies at negative offsets).
// Produces outputs k in [k0, k0+count): y[k-k0].  h1: 2m taps, oldest first.
cudaError_t launch_halfband_decim(const float2* x, int64_t a0, const float* h1, unsigned m,
                                  int64_t k0, size_t count, float scale, float2* y, cudaStream_t st);
// interpolator: inputs k in [k0,k0+count) -> outputs 2k, 2k+1 written at y[2(k-k0)], y[2(k-k0)+1]
cudaError_t launch_halfband_interp(const float2* x, int64_t a0, const float* h1, unsigned m,
                                   int64_t k0, size_t count, float2* y, cudaStream_t st);
// arbitrary polyphase stage: outputs o in [0,count): P = phase0 + o*step; k = kbase + (P>>24)
// (k is an absolute input index, x points at absolute index a0); bank [256][14] oldest first.
cudaError_t launch_arb(const float2* x, int64_t a0, const float* bank, uint32_t step, int64_t kbase,
                       uint32_t phase0, size_t count, float2* y, cudaStream_t st);

// ---- K3: time-domain FIR ---------------------------------------------------------------------
// y[n] = sum_{i<ntaps} hrev[i] * x[n - (ntaps-1) + i]; x points at the first NEW sample.
// hrev: ntaps_padded complex or real taps, oldest first, zero-padded at the FRONT to a multiple of 8.
// hrev_host (optional): the same taps in host memory; when they fit the parameter bank (4096 floats) they
// travel as kernel parameters and are read as constant-bank FFMA operands.
// out_conv (optional, only when fir_can_convert_out() says so): the filter is the chain's last cf32 stage; the epilogue
// converts to `out_format` and writes the final output there instead of the cf32 stream y.
// fold (optional, only when fir_can_fold_dc() says so): the samples [0, n) still lack the fused front's closed-form DC
// term (DcFold below); the filter adds it while it stages its tiles, so the stream is not read and written once more.
struct DcFold;
cudaError_t launch_fir(const float2* x, size_t n, const float* hrev, unsigned ntaps_padded,
                       int complex_taps, float2* y, cudaStream_t st, const float* hrev_host = nullptr,
                       int out_format = 0, void* out_conv = nullptr, const DcFold* fold = nullptr);
bool fir_can_convert_out(int out_format, unsigned ntaps_padded, int complex_taps);
bool fir_can_fold_dc(unsigned ntaps_padded, int complex_taps, bool have_host_taps);

// ---- K4: FFT block filter (overlap-save form of liquid's fftfilt) --------------------------
// For each block b in [0,nblocks): window = x[(b-1)*B .. (b+1)*B), y[b*B .. (b+1)*B) =
// last B samples of IFFT(FFT(window) .* H) / (2B).  x points at block 0's first sample.
// 2B > 16384 needs a global scratch of fftfilt_scratch_bytes(nblocks, B); *launches += kernels launched.
cudaError_t launch_fftfilt(const float2* x, size_t nblocks, unsigned B, const float2* H,
                           const float2* twiddle, float2* y, float2* scratch, uint32_t* launches, cudaStream_t st);
size_t fftfilt_scratch_bytes(size_t nblocks, unsigned B);
// H = FFT(h || 0) of size 2B (forward, un-normalised, in the network's digit-reversed order);
// twiddle: exp(-j 2 pi k / 2B), k < 2B
cudaError_t launch_fft_forward(const float2* in, unsigned nfft, const float2* twiddle, float2* out,
                               cudaStream_t st);
bool fftfilt_supported(unsigned B);
// twiddle table of an nfft-point transform as the FFT kernels expect it: exp(-2 pi i k / nfft), k < nfft, followed by the
// compact per-pass records of the radix-16 kernel (fft_filter2.cuh); float2 entries in total / filled on the host
size_t fft_twiddle_entries(unsigned nfft);
void fft_fill_twiddles(unsigned nfft, float2* host);

// ---- K5: post-processor ([NCO] + AGC + convert) ---------------------------------------------
struct AgcState {           // lives in device memory
    int      locked;
    float    gain;
    float    peak_mem;
    unsigned long long seen;
    double   last_strong;   // sample-clock seconds
    float    rms_g;         // liquid agc_crcf state
    float    rms_y2;
};
struct PostParams {
    int      format;        // output IQGPU_FMT_*
    int      nco_enable;
    uint32_t nco_theta0;
    uint32_t nco_dtheta;
    float    nco_sign;
    const float* nco_table;
    int      agc_mode;      // 0 none, 1 digital, 2 rms
    float    agc_target;
    float    agc_alpha;     // rms bandwidth
    double   target_rate;
};
// segment table: seg_start[0..nseg] (prefix offsets into the n samples of this call)
cudaError_t launch_agc_peaks(const float2* x, size_t n, const PostParams& p, const uint32_t* seg_start,
                             size_t nseg, float* seg_peak, cudaStream_t st);
// quiet_ws (optional, agc_quiet_workspace_bytes(nseg) device bytes): a state-only advance (seg_gain == nullptr) over a long
// table first asks, grid-wide, whether anything happens in it at all
size_t agc_quiet_workspace_bytes(size_t nseg);
cudaError_t launch_agc_digital_scan(const uint32_t* seg_start, size_t nseg, const float* seg_peak,
                                    const PostParams& p, AgcState* state, float* seg_gain, cudaStream_t st, void* quiet_ws = nullptr);
// rms AGC (liquid agc_crcf): the sequential recurrence evaluated time-parallel to its exact fixed point
// (after NCO if enabled -> writes mixed+scaled cf32 to y); ws: agc_rms_workspace_bytes(n, alpha) device bytes
size_t agc_rms_workspace_bytes(size_t n, float alpha);
cudaError_t launch_agc_rms(const float2* x, size_t n, const PostParams& p, AgcState* state, float2* y, void* ws,
                           cudaStream_t st);
// Resume of the last launch_agc_rms call (same x, n, p, y, ws — the workspace still holds that call's block end states and
// checkpoints): the recurrence re-runs from sample `first` with the start state *start ({g, y2'}, device), stops where its
// trajectory meets the previous one bit for bit, and leaves y and *state exactly as one call from that state at `first`
// would have.  A resume at the same sample and from the same state as the previous resume (rr->last_first / last_start;
// `fresh` = no resume since the call) does nothing.  rr receives the rewritten range [lo, hi) of y; *changed (optional) =
// whether the end state changed.
struct AgcRmsResume {
    float2 last_start;
    float2 ck_scratch;              // checkpoint slot of the unaligned head of the resumed block (never compared)
    unsigned long long last_first, lo, hi;
    unsigned valid, pad;
};
cudaError_t launch_agc_rms_resume(const float2* x, size_t n, const PostParams& p, AgcState* state, float2* y, void* ws,
                                  size_t first, const float2* start, AgcRmsResume* rr, bool fresh, int* changed,
                                  cudaStream_t st);
// convert y[rr->lo, rr->hi) to `format` into out (the range a resume rewrote; both bounds read on the device)
cudaError_t launch_convert_range(const float2* y, const AgcRmsResume* rr, int format, void* out, cudaStream_t st);
// y_cf32 (optional tap) and converted out
cudaError_t launch_post(const float2* x, size_t n, const PostParams& p, const uint32_t* seg_start,
                        size_t nseg, const float* seg_gain, int nco_already_applied, float2* tap_cf32,
                        void* out, cudaStream_t st);

// ---- conversions for the module-level API ---------------------------------------------------
cudaError_t launch_convert_out(const float2* x, size_t n, int format, void* out, cudaStream_t st);

// ---- K6: I/Q optimiser pass on one 1024-frame block (host pointers; synchronous) ---------------
cudaError_t iq_optimize_device(const float* host_block1024, const float* host_dirs50, float* mag, float* phase,
                               float* avg_power, float* power_range, int* optimized);

// in-chain form: the optimiser's factors and counters in device memory; one launch runs the passes of a train over
// n_probes blocks of 1024 frames (stream order), +-1 directions from a counter-based generator (seed, attempt number)
struct IqOptState { float mag, phase, avg_power, power_range; unsigned long long passes, attempts; unsigned seed, pad; };
cudaError_t launch_iq_optimize_train(const float2* probes, int n_probes, IqOptState* state, cudaStream_t st);
float iq_direction_host(unsigned seed, unsigned long long pass, unsigned k);

// ---- fused front: raw -> [convert, DC, I/Q, NCO] -> halfband cascade -> polyphase stage -------
// The kernel (fused_front2.cuh) is compiled for the cascades S = 0..W2_MAXS with semi-lengths 3...3,5,10; fused_supported()
// says whether a cascade is one of them.  Any other cascade runs the stage-by-stage kernels above.
constexpr int W2_MAXS = 6;          // deepest cascade with a compiled plan
struct ResamplerDesc {
    unsigned S;                                // halfband stages
    unsigned m_exec[W2_MAXS];                  // semi-length by EXECUTION depth (depth 0 = full input rate)
    const float* h1_exec[W2_MAXS];             // host pointers to the 2m dot-product taps per depth
    float zeta;
    uint32_t step;
};
// Local DC state of the warp-streaming front (fused_front2.cuh): every warp ran its stretch of the stream from v = 0, the
// term it could not know is a decaying exponential per stretch that is added afterwards in closed form.
// Polyphase position of the outputs o >= o_base of one launch.  P(o) = o * step needs up to 87 bits (positions below 2^62),
// k(o) = P >> 24 is the input sample the window ends at, (P >> 16) & 255 the bank row.  With p_base = o_base * step mod 2^64
// rounded down to a multiple of 2^24, D = o * step - p_base (mod 2^64) equals P(o) - k_base * 2^24 exactly while
// (o - o_base) * step stays below 2^63 (any launch), so k(o) = k_base + (D >> 24) and the row is (D >> 16) & 255.
struct ArbBase {
    long long k_base;
    unsigned long long p_base;
};
inline ArbBase arb_base(unsigned long long o_base, uint32_t step)
{
    const unsigned __int128 P = (unsigned __int128)o_base * step;
    return ArbBase{(long long)(P >> 24), (unsigned long long)P & ~0xffffffull};
}
struct W2DcCorr { float2 c_out, c_pre; };      // -a V0 Atot (cascade output) and -a V0 (cascade input, for the cf32 tail)
struct W2DcGeom {
    int n_stretch;
    long long B0, L_full, L_last, warm_frames, pad_frames;     // pad: zero frames between N1 and the end of the last tick
    double lnc, alpha, atot;
    long long O0;              // first output of the launch and its polyphase position
    ArbBase pos;
};
// what a consumer of the resampled stream needs to add that term itself to sample i (absolute output index O0 + i)
struct DcFold {
    const W2DcCorr* corr;      // device: one record per stretch
    const float* G;            // device: 256 polyphase row gains
    W2DcGeom geo;              // geo.O0: the launch's first output
    uint32_t step;
    int S;
};
struct FusedFront;
bool fused_supported(int format, const ResamplerDesc& r);
FusedFront* fused_create(int format, const ResamplerDesc& r, bool nco, const float* d_bank, int num_sms, std::string& err);
void fused_destroy(FusedFront* f);
cudaError_t fused_reset(FusedFront* f, cudaStream_t st);
uint32_t fused_halo_frames(const FusedFront* f);
// outputs per lane of the polyphase variant the last launch ran (1, 2 or 4; 0 before the first launch)
uint32_t fused_polyphase_variant(const FusedFront* f);
const double2* fused_dc_state_at(const FusedFront* f, int slot, int64_t n0, int64_t pos);
// raw[0] has absolute index n0; produces outputs [O0, O0+n_out) into y; d_dc_carry is the DC state at n0
// (updated to the state at n0+n).  *launches is incremented by the kernels launched.
// dc_slot (0/1): DC table slot; if fused_prepare_dc() filled it (possibly on another stream, ordered by
// the caller) the launch uses it, otherwise the pre-pass runs inline on `st`.
// fold (optional): when the launch used the local DC state, the closed-form term is NOT added to y; *fold describes it
// (fold->corr != nullptr) for a consumer that adds it on the fly, and fused_dc_correct_range() adds it in memory to the part
// of y that stays behind as somebody's history.  The cf32 tail of the pre-processed stream is corrected in any case.
cudaError_t fused_launch(FusedFront* f, const void* raw, int64_t n0, size_t n, const PreParams& pre, double2* d_dc_carry,
                         int64_t O0, size_t n_out, float2* y, uint32_t* launches, int dc_slot, cudaStream_t st,
                         DcFold* fold = nullptr);
cudaError_t fused_dc_correct_range(const DcFold& fold, float2* y, size_t first, size_t count, cudaStream_t st);
cudaError_t fused_prepare_dc(FusedFront* f, int slot, const void* raw, int64_t n0, size_t n, const PreParams& pre,
                             double2* d_dc_carry, uint32_t* launches, cudaStream_t st);

}  // namespace iqgpu
