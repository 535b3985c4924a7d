// chain.cu — the chain engine and the C ABI (include/iqgpu.h).
//
// One iqgpu_chain owns the DSP state of a full reference pipeline
// (src/pipeline.c:138-147: dc_block, iq_correct, freq_shift, resampler, filter, agc) and runs
// "trains" of reference chunks through it.  Everything that is not data dependent — NCO phase,
// halfband alignment, arbitrary-resampler phase, per-chunk output counts, FFT-filter block
// bookkeeping — is closed-form integer arithmetic on the absolute stream position and is
// evaluated on the host; the device only carries data-dependent state (DC-blocker carry, filter
// histories, AGC state).
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstddef>
#include <cstdio>
#include <cstring>
#include <string>
#include <exception>
#include <memory>
#include <new>
#include <vector>

#include "../../include/iqgpu.h"
#include "cuda_owned.hpp"
#include "design.hpp"
#include "kernels.hpp"

using namespace iqgpu;

static thread_local std::string g_err;
static int fail(int code, const std::string& msg)
{
    g_err = msg;
    return code;
}
#define CK(call)                                                                                       \
    do {                                                                                               \
        cudaError_t e_ = (call);                                                                       \
        if (e_ != cudaSuccess) {                                                                       \
            g_err = std::string(#call) + ": " + cudaGetErrorString(e_);                                \
            return IQGPU_ECUDA;                                                                        \
        }                                                                                              \
    } while (0)

namespace {

size_t bytes_per_sample(int fmt)
{
    switch (fmt) {  // reference src/sample_convert.c:102-123
        case IQGPU_FMT_S8: case IQGPU_FMT_U8: return 1;
        case IQGPU_FMT_S16: case IQGPU_FMT_U16: return 2;
        case IQGPU_FMT_S32: case IQGPU_FMT_U32: case IQGPU_FMT_F32: return 4;
        case IQGPU_FMT_CS8: case IQGPU_FMT_CU8: return 2;
        case IQGPU_FMT_CS16: case IQGPU_FMT_CU16: case IQGPU_FMT_SC16Q11: return 4;
        case IQGPU_FMT_CS24: return 6;
        case IQGPU_FMT_CS32: case IQGPU_FMT_CU32: case IQGPU_FMT_CF32: return 8;
        default: return 0;
    }
}
bool is_complex_format(int fmt) { return fmt >= IQGPU_FMT_CU8 && fmt <= IQGPU_FMT_SC16Q11; }

// cf32 stream segment with history head-room.  New data of a call is written at base+pos; the
// previous `hist` samples sit right below it.
struct DevStream {
    DeviceArray<float2> buf;
    size_t hist = 0, pos = 0, max_n = 0, slack = 0;   // slack: readable (zeroable) room kept beyond the new data
    cudaError_t alloc(size_t hist_, size_t max_n_, size_t slack_ = 0)
    {
        hist = (hist_ + 3) & ~(size_t)3;
        max_n = std::max(max_n_, hist) + 4;
        slack = slack_;
        return buf.alloc(hist + 2 * max_n + slack);
    }
    cudaError_t reset(cudaStream_t st)
    {
        pos = hist;
        return hist ? cudaMemsetAsync(buf.data(), 0, hist * sizeof(float2), st) : cudaSuccess;
    }
    // stream discontinuity that keeps the newest `keep` samples where they are and clears the history below them
    cudaError_t reset_keep_tail(cudaStream_t st, size_t keep)
    {
        if (keep >= hist) return cudaSuccess;
        return cudaMemsetAsync(buf.data() + pos - hist, 0, (hist - keep) * sizeof(float2), st);
    }
    // make room for n new samples; returns pointer to the first new sample
    cudaError_t begin(size_t n, cudaStream_t st, float2** p)
    {
        if (n > max_n) return cudaErrorInvalidValue;
        float2* base = buf.data();
        if (pos + n + slack > buf.size()) {
            // move the history to the front (ranges cannot overlap: pos - hist >= hist)
            cudaError_t e = cudaMemcpyAsync(base, base + pos - hist, hist * sizeof(float2), cudaMemcpyDeviceToDevice, st);
            if (e != cudaSuccess) return e;
            pos = hist;
        }
        *p = base + pos;
        return cudaSuccess;
    }
    void commit(size_t n) { pos += n; }
};

struct TapBuf {
    DeviceArray<float2> buf;
    size_t len = 0;
    cudaError_t append(const float2* src, size_t n, cudaStream_t st)
    {
        if (len + n > buf.size()) {
            DeviceArray<float2> nb;
            cudaError_t e = nb.alloc(std::max(buf.size() * 2, len + n + 1024));
            if (e != cudaSuccess) return e;
            if (len) {
                e = cudaMemcpyAsync(nb.data(), buf.data(), len * sizeof(float2), cudaMemcpyDeviceToDevice, st);
                if (e != cudaSuccess) return e;
                cudaStreamSynchronize(st);
            }
            buf = std::move(nb);
        }
        cudaError_t e = cudaMemcpyAsync(buf.data() + len, src, n * sizeof(float2), cudaMemcpyDeviceToDevice, st);
        len += n;
        return e;
    }
};

struct FusedDelete { void operator()(FusedFront* f) const { fused_destroy(f); } };

}  // namespace

struct iqgpu_chain {
    iqgpu_chain_config cfg{};
    int device = -1;
    bool plan_only = false;
    int in_rate = 0;
    double target_rate = 0;
    float ratio = 1.f;
    size_t in_bps = 0, out_bps = 0;

    DcPlan dc;
    ResamplerPlan rs;
    FilterPlan filt;
    bool nco_pre = false, nco_post = false;
    uint32_t nco_dtheta = 0;
    float nco_sign = 1.f;
    float iq_mag = 0.f, iq_phase = 0.f;
    int agc_mode = 0;  // 0 none, 1 digital, 2 rms
    float agc_target = 0.f, agc_alpha = 0.f;

    // options
    size_t subtrain_frames = (size_t)1 << 22;
    uint32_t chunk_frames = IQGPU_CHUNK_SAMPLES;
    bool want_fused = true;
    // 0: DC blocker in exact arithmetic (blocked affine scan, double carries); 1: the reference's fp32 direct-form-II state
    // rounding, evaluated serially (launch_dc_reference) — module-level dc_block_apply and parity tests
    int dc_mode = 0;
    bool record_taps = false;
    bool record_tap0 = false;   // tap 0 (pre-processor output) only exists on the unfused path
    bool fused_used = false;
    bool fused_active = false;  // decided when the work buffers are created; fixed for the chain's life

    // ---- stream position (host, closed form) ----
    uint64_t n_in = 0;        // input frames since reset
    uint64_t n_nco_post = 0;  // samples that went through the post NCO
    uint64_t n_out = 0;
    uint32_t fft_rem = 0;     // FFT filter remainder length (frames waiting for a full block)
    // F5: filter_reset (src/filter.c:417-436) clears the liquid object but NOT pre/post_fft_remainder_len, so the frames that
    // were waiting for a full block re-enter the new stream in front of its first chunk.  A pre-resample remainder then
    // counts as resampler input of the new stream: fft_rem_carry = its length at the reset.
    uint32_t fft_rem_carry = 0;
    uint32_t launches = 0;

    // ---- device state ----
    Stream stream, h2d, d2h;
    // second compute stream: the DC pre-pass of sub-train k+1 (HBM bound) runs underneath the fused front
    // kernel of sub-train k (issue bound); ordered with events
    Stream aux;
    Event ev_pre[2], ev_front[2], ev_call, ev_reset;
    cudaStream_t reset_stream = nullptr;   // stream a not yet consumed reset was queued on
    int order_after_reset(cudaStream_t st);
    PinnedArray<uint32_t> seg_pin[2];   // pinned staging of the chunk table (digital AGC)
    Event ev_seg[2];
    int seg_pin_slot = 0;
    template <typename Fill> int stage_chunk_table(uint32_t* dst, size_t n_chunks, cudaStream_t st, Fill fill);
    // chunk tables of lower shards (iqgpu_chain_agc_advance_device), kept per (first frame, frames): a shard plan is
    // replayed step after step, and the table is closed form in those two numbers
    struct PrefixTab { uint64_t first = 0, frames = 0; DeviceArray<uint32_t> d_seg; };
    std::vector<PrefixTab> prefix_tabs;
    bool front_recorded[2] = {false, false};
    int dc_slot = 0;                    // table slot of the sub-train run_subtrain is about to launch
    bool dc_prepared = false;           // ... and whether its pre-pass was issued on `aux`
    cudaStream_t last_stream = nullptr;   // stream of the most recent process call
    DeviceArray<float> d_lut;
    DeviceArray<double2> d_dc_carry;
    DeviceArray<float2> d_dc_ref;        // dc_mode 1: liquid's v0 {re, im} in fp32
    DeviceArray<double2> d_run_sums, d_run_start;
    DeviceArray<double> d_scan_ws;
    std::vector<DeviceArray<float>> d_hb_taps;  // per design index
    DeviceArray<float> d_bank;
    DeviceArray<float> d_fir_taps;
    std::vector<float> h_fir_taps;      // host copy (kernel-parameter taps)
    unsigned fir_taps_padded = 0;
    DeviceArray<float2> d_fft_H, d_fft_tw, d_fft_scratch;
    cudaError_t ensure_fft_scratch(size_t blocks, unsigned block, cudaStream_t st)
    {
        const size_t need = fftfilt_scratch_bytes(blocks, block) / sizeof(float2);
        return d_fft_scratch.grow(need, need + need / 2, [st] { return cudaStreamSynchronize(st); });
    }
    int fft_block_pass(const float2* src, size_t n, DevStream& out, cudaStream_t st, const float2** y, size_t* ny);
    // in-chain I/Q optimiser (SURVEY 8(f) rank 3): gate on the sample clock, passes on the device, factors applied from the
    // next sub-train on
    bool iq_optimize = false;
    double iq_interval_ms = 500.0;          // IQ_CORRECTION_INTERVAL_MS, include/constants.h:159
    uint32_t iq_seed = 20261017u;
    double iq_last_attempt_s = -1e18;       // sample-clock time of the last probe
    DeviceArray<IqOptState> d_iq_state;
    PinnedArray<IqOptState> h_iq_state;
    DeviceArray<float2> d_iq_probe;         // 1024 frames per probe
    Event ev_iq, ev_iq_probe;
    bool iq_pending = false;
    int iq_sync_state();
    int iq_push_state(cudaStream_t st);
    int iq_run_probes(const void* d_rawp, const float2* pre_out, uint64_t N0, const uint32_t* chunks, size_t n_chunks, int slot,
                      cudaStream_t st);
    DeviceArray<AgcState> d_agc;
    DeviceArray<uint32_t> d_seg_start;  // one entry more than the chunks of d_seg_peak / d_seg_gain
    DeviceArray<float> d_seg_peak, d_seg_gain;
    DeviceArray<float2> d_agc_scratch;
    DeviceArray<unsigned char> d_agc_quiet;     // digital AGC: workspace of the grid-wide quiet test (state-only advance)
    cudaError_t ensure_agc_quiet(size_t n_chunks, cudaStream_t st)
    {
        const size_t need = agc_quiet_workspace_bytes(n_chunks);
        return d_agc_quiet.grow(need, need * 2, [st] { return cudaStreamSynchronize(st); });
    }
    DeviceArray<unsigned char> d_agc_ws;        // RMS-AGC time-parallel workspace (block end states + sweep flags)
    // RMS AGC of the last call when it was one sub-train: input, parameters and (in d_agc_scratch / d_agc_ws) output and
    // checkpoints, which iqgpu_chain_agc_rms_resume_device re-runs from a later start state (time shards)
    const float2* rms_src = nullptr;
    size_t rms_n = 0;
    PostParams rms_qp{};
    bool rms_ready = false, rms_fresh = false;
    DeviceArray<AgcRmsResume> d_rms_resume;
    // d_rms_rerun[0]: {g, y2'} the last call started from (its rms_g / rms_y2), [1]: the state of a re-run of that call
    // (which so leaves d_agc alone); rms_resume_max: the latest resume frame since the call or its last re-run.  A resume
    // in front of that frame first re-runs the call (iqgpu_chain_agc_rms_resume_device).
    DeviceArray<AgcState> d_rms_rerun;
    size_t rms_resume_max = 0;
    // streams: s_in = pre output; s_stage[d] = output of executed halfband stage d; s_rs = resampler
    // output; s_f = post-filter output (or pre-filter output when the filter is pre-resample)
    DevStream s_in, s_pref, s_arb_in, s_rs, s_f;
    std::vector<DevStream> s_stage;
    TapBuf tap[3];
    std::unique_ptr<FusedFront, FusedDelete> fused;
    int num_sms = 148;
    // host-path staging (bytes)
    DeviceArray<char> d_raw[2], d_out[2];
    Event ev_h2d[2], ev_done[2], ev_d2h[2];
    bool buffers_ready = false;

    // optional per-kernel-class device timing (CUDA events on the launch stream)
    bool time_kernels = false;
    struct TimedSpan { int cls; Event a, b; };
    std::vector<TimedSpan> spans;
    std::vector<Event> ev_pool;
    double class_ms[IQGPU_KCLASS_COUNT] = {0};
    uint32_t class_launches[IQGPU_KCLASS_COUNT] = {0};
    Event get_event()
    {
        Event e;
        if (!ev_pool.empty()) { e = std::move(ev_pool.back()); ev_pool.pop_back(); }
        else create(e, cudaEventDefault);
        return e;
    }
    void span_begin(int cls, cudaStream_t st)
    {
        class_launches[cls]++;
        if (!time_kernels) return;
        TimedSpan sp{cls, get_event(), get_event()};
        cudaEventRecord(sp.a, st);
        spans.push_back(std::move(sp));
    }
    void span_end(cudaStream_t st)
    {
        if (!time_kernels || spans.empty()) return;
        cudaEventRecord(spans.back().b, st);
    }
    void collect_spans()
    {
        for (auto& sp : spans) {
            float ms = 0.f;
            if (cudaEventSynchronize(sp.b) == cudaSuccess && cudaEventElapsedTime(&ms, sp.a, sp.b) == cudaSuccess)
                class_ms[sp.cls] += ms;
            ev_pool.push_back(std::move(sp.a)); ev_pool.push_back(std::move(sp.b));
        }
        spans.clear();
    }

    ~iqgpu_chain();
    int init_device();
    int ensure_buffers();
    // keep_fft_remainder: the reference's stream-discontinuity semantics (F5); false = the state right after create
    int reset_state(bool keep_fft_remainder = false);
    size_t max_out_for(size_t n_frames) const;
    // closed-form per-chunk output frame counts from the current position (no state change)
    size_t count_outputs(const uint32_t* chunks, size_t n_chunks, uint32_t* per_chunk) const;
    // phase: 0 = whole sub-train; 1 = front only (everything up to the per-chunk AGC peaks; the
    // rest is left pending for run_back) — the split point of the sharded digital-AGC exchange
    int run_subtrain(const void* d_rawp, size_t n, const uint32_t* chunks, size_t n_chunks, void* d_outp,
                     size_t* out_frames, uint32_t* per_chunk, cudaStream_t st, int phase = 0);
    int run_back(void* d_outp, size_t skip_chunks, size_t* out_frames, cudaStream_t st);
    PreParams pre_params(uint64_t N0) const;
    int prepare_dc(int slot, const void* d_rawp, uint64_t N0, size_t n, cudaStream_t st);
    bool fir_wrote_output = false;    // this sub-train's FIR epilogue converted and stored the final output
    DcFold dc_fold{};                 // the front's closed-form DC term, when the FIR behind it adds it on the fly
    // long post-resample FIRs are evaluated by the FFT block filter kernel (overlap-save, same causal convolution): the
    // time-domain kernel runs at 85 % of FMA peak, so beyond a few hundred taps only fewer FLOPs help
    bool fir_via_fft = false;
    unsigned fir_fft_block = 0;
    bool dc_overlap = true;           // DC pre-pass of sub-train k+1 on the second stream while sub-train k runs
    uint32_t prepass_launches = 0;
    // pending back half (between process_device_begin and process_device_finish)
    struct Pending {
        bool active = false;
        const float2* src = nullptr;
        size_t n = 0, n_chunks = 0;
        std::vector<uint32_t> seg, counts;
        PostParams qp{};
        bool peaks_done = false;
    } pend;
};

// the members free their resources after this body, once nothing runs on the chain's streams any more
iqgpu_chain::~iqgpu_chain()
{
    if (plan_only) return;
    cudaSetDevice(device);
    if (stream) cudaStreamSynchronize(stream);
    if (aux) cudaStreamSynchronize(aux);
    collect_spans();
}

static bool filter_is_fft(const FilterPlan& f)
{
    return f.impl == IQGPU_FILTER_IMPL_FFT_SYM || f.impl == IQGPU_FILTER_IMPL_FFT_ASYM;
}
static bool filter_is_fir(const FilterPlan& f)
{
    return f.impl == IQGPU_FILTER_IMPL_FIR_SYM || f.impl == IQGPU_FILTER_IMPL_FIR_ASYM;
}

// chain output frames after `k` input frames since a restart: the resampler's count (pipeline.c:523), block-quantised by an
// FFT filter (filter.c:491-526).  The quantisation carries its remainder from chunk to chunk, so the sum of count_outputs'
// per-chunk counts from a restart is this closed form at every chunk boundary.
static uint64_t chain_outputs_after(const iqgpu_chain* c, uint64_t k)
{
    if (!filter_is_fft(c->filt)) return resampler_outputs_after(c->rs, k);
    const uint64_t B = c->filt.block;
    if (!c->filt.post_resample) return resampler_outputs_after(c->rs, k / B * B);
    return resampler_outputs_after(c->rs, k) / B * B;
}

size_t iqgpu_chain::max_out_for(size_t n) const
{
    double r = rs.passthrough ? 1.0 : (double)ratio;
    size_t m = (size_t)std::ceil((double)n * std::max(r, 0.0)) + 4096;
    if (rs.is_interp) m += ((size_t)2 << rs.num_halfband);
    if (filter_is_fft(filt)) m += filt.block;
    return m;
}

size_t iqgpu_chain::count_outputs(const uint32_t* chunks, size_t n_chunks, uint32_t* per_chunk) const
{
    // mirrors the reference's per-chunk bookkeeping: resampler frames_to_write (pipeline.c:523),
    // FFT-filter block quantisation (filter.c:491-526), empty chunks skipped (post_processor.c:12)
    const bool fft = filter_is_fft(filt);
    const bool pre_fft = fft && !filt.post_resample, post_fft = fft && filt.post_resample;
    uint32_t rem = fft_rem;
    uint64_t pos = pre_fft ? n_in + fft_rem_carry - fft_rem : n_in;
    uint64_t before = resampler_outputs_after(rs, pos), total = 0;
    if (!fft && !per_chunk) {       // only the total is wanted and nothing quantises per chunk: closed form over the whole train
        uint64_t sum = 0;
        for (size_t c = 0; c < n_chunks; c++) sum += chunks[c];
        return (size_t)(resampler_outputs_after(rs, pos + sum) - before);
    }
    for (size_t c = 0; c < n_chunks; c++) {
        uint32_t f = chunks[c];
        if (pre_fft) { const uint32_t tot = rem + f, b = tot / filt.block; f = b * filt.block; rem = tot - f; }
        pos += f;
        const uint64_t after = resampler_outputs_after(rs, pos);
        uint32_t r = (uint32_t)(after - before);
        before = after;
        if (post_fft && r) { const uint32_t tot = rem + r, b = tot / filt.block; r = b * filt.block; rem = tot - r; }
        if (per_chunk) per_chunk[c] = r;
        total += r;
    }
    return (size_t)total;
}

int iqgpu_chain::init_device()
{
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(IQGPU_ENODEVICE, "no CUDA device available");
    if (device >= ndev) return fail(IQGPU_EINVAL, "device index out of range");
    CK(cudaSetDevice(device));
    for (Stream* s : {&stream, &h2d, &d2h, &aux}) CK(create(*s));
    for (Event* e : {&ev_call, &ev_reset, &ev_pre[0], &ev_pre[1], &ev_front[0], &ev_front[1], &ev_seg[0], &ev_seg[1], &ev_h2d[0],
                     &ev_h2d[1], &ev_done[0], &ev_done[1], &ev_d2h[0], &ev_d2h[1]})
        CK(create(*e));
    // constant tables
    float lut[1024];
    nco_sine_table(lut);
    CK(d_lut.alloc(1024));
    CK(cudaMemcpy(d_lut.data(), lut, sizeof(lut), cudaMemcpyHostToDevice));
    CK(d_dc_carry.alloc(1));
    CK(d_dc_ref.alloc(1));
    CK(d_agc.alloc(1));
    if (agc_mode == 2) CK(d_rms_rerun.alloc(2));
    if (!rs.passthrough) {
        d_hb_taps.resize(rs.num_halfband);
        for (unsigned i = 0; i < rs.num_halfband; i++) {
            CK(d_hb_taps[i].alloc(rs.stages[i].h1.size()));
            CK(cudaMemcpy(d_hb_taps[i].data(), rs.stages[i].h1.data(), rs.stages[i].h1.size() * sizeof(float), cudaMemcpyHostToDevice));
        }
        CK(d_bank.alloc(rs.bank.size()));
        CK(cudaMemcpy(d_bank.data(), rs.bank.data(), rs.bank.size() * sizeof(float), cudaMemcpyHostToDevice));
    }
    {
        cudaDeviceProp prop{};
        if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) num_sms = prop.multiProcessorCount;
    }
    const bool pre_filter0 = filt.impl != IQGPU_FILTER_IMPL_NONE && !filt.post_resample;
    if (!rs.passthrough && !rs.is_interp && !pre_filter0) {
        ResamplerDesc rd{};
        rd.S = rs.num_halfband; rd.zeta = rs.zeta; rd.step = rs.step;
        bool ok = rs.num_halfband <= (unsigned)W2_MAXS;
        for (unsigned d = 0; ok && d < rs.num_halfband; d++) {
            const unsigned g = rs.num_halfband - 1 - d;
            rd.m_exec[d] = rs.stages[g].m;
            rd.h1_exec[d] = rs.stages[g].h1.data();
        }
        if (ok && fused_supported(cfg.input_format, rd)) {
            std::string ferr;
            fused.reset(fused_create(cfg.input_format, rd, nco_pre, d_bank.data(), num_sms, ferr));
            if (!fused) return fail(IQGPU_ECUDA, ferr);
        }
    }
    if (filter_is_fir(filt)) {
        const unsigned N = (unsigned)filt.taps.size();
        fir_taps_padded = (N + 7) & ~7u;
        const unsigned pad = fir_taps_padded - N;
        const bool cplx = filt.impl == IQGPU_FILTER_IMPL_FIR_ASYM;
        std::vector<float> h((size_t)fir_taps_padded * (cplx ? 2 : 1), 0.f);
        for (unsigned i = 0; i < N; i++) {  // oldest-first order: hrev[i] = h[N-1-i]
            const cfloat t = filt.taps[N - 1 - i];
            if (cplx) { h[2 * (pad + i)] = t.real(); h[2 * (pad + i) + 1] = t.imag(); }
            else h[pad + i] = t.real();
        }
        CK(d_fir_taps.alloc(h.size()));
        CK(cudaMemcpy(d_fir_taps.data(), h.data(), h.size() * sizeof(float), cudaMemcpyHostToDevice));
        h_fir_taps = h;
    }
    if (filter_is_fir(filt) && filt.post_resample && filt.taps.size() >= 512 && filt.taps.size() <= 8192 &&
        !getenv("IQGPU_FIR_TIME_DOMAIN")) {
        fir_via_fft = true;
        fir_fft_block = 8192;
    }
    if (filter_is_fft(filt) || fir_via_fft) {
        const unsigned blk = fir_via_fft ? fir_fft_block : filt.block;
        if (!fftfilt_supported(blk)) return fail(IQGPU_EINVAL, "FFT filter block size not supported by the GPU FFT kernel");
        const unsigned nfft = 2 * blk;
        std::vector<float2> tw(fft_twiddle_entries(nfft)), hpad(nfft, make_float2(0.f, 0.f));
        fft_fill_twiddles(nfft, tw.data());
        for (size_t i = 0; i < filt.taps.size(); i++) hpad[i] = make_float2(filt.taps[i].real(), filt.taps[i].imag());
        DeviceArray<float2> d_h;
        CK(d_fft_tw.alloc(tw.size()));
        CK(d_fft_H.alloc(nfft));
        CK(d_h.alloc(nfft));
        CK(cudaMemcpy(d_fft_tw.data(), tw.data(), tw.size() * sizeof(float2), cudaMemcpyHostToDevice));
        CK(cudaMemcpy(d_h.data(), hpad.data(), nfft * sizeof(float2), cudaMemcpyHostToDevice));
        CK(launch_fft_forward(d_h.data(), nfft, d_fft_tw.data(), d_fft_H.data(), stream));
        CK(cudaStreamSynchronize(stream));
    }
    return IQGPU_OK;
}

int iqgpu_chain::ensure_buffers()
{
    if (buffers_ready) return IQGPU_OK;
    CK(cudaSetDevice(device));
    const size_t n = subtrain_frames + chunk_frames;  // a sub-train never exceeds this
    const bool pre_filter = filt.impl != IQGPU_FILTER_IMPL_NONE && !filt.post_resample;
    const bool post_filter = filt.impl != IQGPU_FILTER_IMPL_NONE && filt.post_resample;
    const size_t filt_hist = filter_is_fir(filt) ? fir_taps_padded : (filter_is_fft(filt) ? 2 * (size_t)filt.block : 0);

    fused_active = fused && want_fused && !record_tap0 && !(dc.enable && dc_mode == 1);
    // s_in: consumer is the pre-filter, else the first resampler stage, else nothing
    size_t in_hist = 0;
    if (pre_filter) in_hist = filt_hist;
    else if (!rs.passthrough && !rs.is_interp) in_hist = rs.num_halfband ? 4 * rs.stages[rs.num_halfband - 1].m : 16;
    else if (!rs.passthrough) in_hist = 16;
    if (!fused_active && s_in.alloc(in_hist, n) != 0) return fail(IQGPU_ENOMEM, "device allocation failed (s_in)");
    if (pre_filter) {
        size_t h = 16;
        if (!rs.passthrough && !rs.is_interp && rs.num_halfband) h = 4 * rs.stages[rs.num_halfband - 1].m;
        if (s_pref.alloc(h, n + filt.block) != 0) return fail(IQGPU_ENOMEM, "device allocation failed (s_pref)");
    }
    size_t rs_max = n;
    if (fused_active) {
        rs_max = (size_t)std::ceil((double)(n >> rs.num_halfband) * (double)rs.rate_arbitrary) + 16;
    } else if (!rs.passthrough) {
        const unsigned S = rs.num_halfband;
        s_stage.resize(S);
        if (!rs.is_interp) {
            // executed stage d (design index S-1-d) halves the rate; its output feeds stage d+1 or the arb stage
            for (unsigned d = 0; d < S; d++) {
                const size_t cnt = (n >> (d + 1)) + 2;
                const size_t h = (d + 1 < S) ? 4 * rs.stages[S - 2 - d].m : 16;
                if (s_stage[d].alloc(h, cnt) != 0) return fail(IQGPU_ENOMEM, "device allocation failed (stage)");
            }
            rs_max = (size_t)std::ceil((double)(n >> S) * (double)rs.rate_arbitrary) + 16;
        } else {
            // arbitrary first (on s_in), then interpolators by design index 0..S-1
            const size_t arb_cnt = (size_t)std::ceil((double)n * (double)rs.rate_arbitrary) + 16;
            if (s_arb_in.alloc(S ? 2 * rs.stages[0].m : 0, arb_cnt) != 0) return fail(IQGPU_ENOMEM, "device allocation failed (arb)");
            for (unsigned s = 0; s < S; s++) {
                const size_t cnt = (arb_cnt << (s + 1));
                const size_t h = (s + 1 < S) ? 2 * rs.stages[s + 1].m : 0;
                if (s + 1 < S && s_stage[s].alloc(h, cnt) != 0) return fail(IQGPU_ENOMEM, "device allocation failed (stage)");
            }
            rs_max = arb_cnt << S;
        }
    }
    if (fir_via_fft) {
        // the block kernel reads one block of history below the first new sample and up to one block (zeroed) beyond the last
        if (s_rs.alloc(fir_fft_block, rs_max, fir_fft_block) != 0) return fail(IQGPU_ENOMEM, "device allocation failed (s_rs)");
    } else
    if (s_rs.alloc(post_filter ? filt_hist : 0, rs_max + (post_filter ? filt.block : 0)) != 0)
        return fail(IQGPU_ENOMEM, "device allocation failed (s_rs)");
    if (post_filter && s_f.alloc(0, rs_max + 2 * (size_t)std::max<unsigned>(filt.block, fir_fft_block)) != 0)
        return fail(IQGPU_ENOMEM, "device allocation failed (s_f)");

    const size_t max_runs = n / 128 + 2;
    CK(d_run_sums.alloc(max_runs));
    CK(d_scan_ws.alloc(dc_scan_workspace_doubles(max_runs)));
    CK(d_run_start.alloc(max_runs));
    const size_t max_segs = n / std::max<uint32_t>(1, std::min<uint32_t>(chunk_frames, 1024)) + 8;
    CK(d_seg_start.alloc(max_segs + 1));
    CK(d_seg_peak.alloc(max_segs));
    CK(d_seg_gain.alloc(max_segs));
    buffers_ready = true;
    return reset_state();
}

__global__ void agc_state_init_kernel(AgcState* st, AgcState v) { *st = v; }
// RMS-AGC resume at the end of the call: the end state becomes *s; *changed (optional) = whether it moved
__global__ void agc_rms_set_end_kernel(AgcState* st, const float2* s, int* changed)
{
    const float2 v = *s;
    if (changed)
        *changed = (__float_as_uint(v.x) != __float_as_uint(st->rms_g) || __float_as_uint(v.y) != __float_as_uint(st->rms_y2)) ? 1 : 0;
    st->rms_g = v.x; st->rms_y2 = v.y;
}

// Stream discontinuity.  All device state lives behind the stream the chain last ran on, so the reset is QUEUED there
// (memsets + one tiny kernel, no host synchronisation: the host may go on enqueueing the next train while the previous
// one still runs); a later call on another stream first waits for ev_reset.
int iqgpu_chain::reset_state(bool keep_fft_remainder)
{
    const bool pre_fft = filter_is_fft(filt) && !filt.post_resample, post_fft = filter_is_fft(filt) && filt.post_resample;
    const uint32_t keep = (keep_fft_remainder && (pre_fft || post_fft)) ? fft_rem : 0;
    n_in = 0; n_nco_post = 0; n_out = 0; fft_rem = keep;
    iq_last_attempt_s = -1e18;              // the sample clock restarts with the stream
    fft_rem_carry = pre_fft ? keep : 0;
    rms_ready = false;
    if (plan_only || !buffers_ready) return IQGPU_OK;
    CK(cudaSetDevice(device));
    cudaStream_t S = last_stream ? last_stream : stream;
    dc_prepared = false;
    front_recorded[0] = front_recorded[1] = false;
    CK(cudaMemsetAsync(d_dc_carry.data(), 0, sizeof(double2), S));
    CK(cudaMemsetAsync(d_dc_ref.data(), 0, sizeof(float2), S));
    AgcState a{};
    a.locked = 0; a.gain = 1.0f; a.seen = 0; a.last_strong = 0.0;
    a.peak_mem = (agc_mode == 1) ? 0.05f : 0.001f;   // agc.c:66,78
    a.rms_g = 1.0f; a.rms_y2 = 1.0f;                  // agc.c:58-62 (set_signal_level then set_gain(1))
    agc_state_init_kernel<<<1, 1, 0, S>>>(d_agc.data(), a);
    CK(cudaGetLastError());
    if (fused) CK(fused_reset(fused.get(), S));
    if (s_in.buf.data()) CK((keep && pre_fft) ? s_in.reset_keep_tail(S, keep) : s_in.reset(S));
    if (s_pref.buf.data()) CK(s_pref.reset(S));
    if (s_arb_in.buf.data()) CK(s_arb_in.reset(S));
    for (auto& s : s_stage) if (s.buf.data()) CK(s.reset(S));
    CK((keep && post_fft) ? s_rs.reset_keep_tail(S, keep) : s_rs.reset(S));
    if (s_f.buf.data()) CK(s_f.reset(S));
    CK(cudaEventRecord(ev_reset, S));
    reset_stream = S;
    return IQGPU_OK;
}

// a call on stream `st` after a reset that was queued on another stream
int iqgpu_chain::order_after_reset(cudaStream_t st)
{
    if (reset_stream && reset_stream != st) CK(cudaStreamWaitEvent(st, ev_reset, 0));
    reset_stream = nullptr;
    return IQGPU_OK;
}

PreParams iqgpu_chain::pre_params(uint64_t N0) const
{
    PreParams pp{};
    pp.format = cfg.input_format; pp.gain = cfg.gain;
    pp.dc_enable = dc.enable; pp.dc_c = dc.c; pp.dc_a = dc.one_minus_c;
    pp.iq_enable = cfg.iq_correction_enable; pp.iq_magp1 = 1.0f + iq_mag; pp.iq_phase = iq_phase;
    pp.nco_enable = nco_pre; pp.nco_dtheta = nco_dtheta; pp.nco_sign = nco_sign; pp.nco_table = d_lut.data();
    pp.nco_theta0 = (uint32_t)((uint64_t)(uint32_t)N0 * nco_dtheta);
    return pp;
}

// DC pre-pass of the sub-train that starts at absolute frame N0, on the second stream, into table `slot`.
// `st` is the stream the front kernels run on: the slot's previous reader must have finished first.
int iqgpu_chain::prepare_dc(int slot, const void* d_rawp, uint64_t N0, size_t n, cudaStream_t st)
{
    (void)st;
    if (front_recorded[slot]) CK(cudaStreamWaitEvent(aux, ev_front[slot], 0));
    const PreParams pp = pre_params(N0);
    uint32_t l = 0;
    CK(fused_prepare_dc(fused.get(), slot, d_rawp, (int64_t)N0, n, pp, d_dc_carry.data(), &l, aux));
    prepass_launches += l;                      // 0 when the front kernel carries the DC state itself (no pre-pass)
    CK(cudaEventRecord(ev_pre[slot], aux));
    return IQGPU_OK;
}

// ---------------------------------------------------------------------------------------------
// in-chain I/Q optimiser.  Reference: the pre thread copies the first 1024 frames of every pre-processed chunk to a side
// queue (src/pipeline.c:468-476), a side thread runs iq_correct_run_optimization on them at most every 500 ms of WALL time
// with rand() directions (src/utility_threads.c:35-47, src/iq_correct.c:154-235).  Here (SURVEY App. B7, deliberate): the
// gate runs on the SAMPLE clock (input frames / input rate; an attempt on a weak block also restarts it), the directions
// come from a counter-based generator, the passes of a sub-train run back to back on the device behind the front kernel, and
// the factors they leave are applied from the next sub-train on (the reference's apply sees them one chunk later).
// ---------------------------------------------------------------------------------------------
int iqgpu_chain::iq_sync_state()
{
    if (!iq_pending) return IQGPU_OK;
    CK(cudaEventSynchronize(ev_iq));
    iq_pending = false;
    iq_mag = h_iq_state.data()->mag; iq_phase = h_iq_state.data()->phase;
    return IQGPU_OK;
}

int iqgpu_chain::iq_push_state(cudaStream_t st)
{
    if (!d_iq_state.data()) {       // first use; d_iq_state comes last, so that a set-up that failed is redone as a whole
        CK(h_iq_state.alloc(1));
        memset(h_iq_state.data(), 0, sizeof(IqOptState));
        CK(create(ev_iq));
        CK(create(ev_iq_probe));
        CK(d_iq_state.alloc(1));
    }
    { int rc_ = iq_sync_state(); if (rc_) return rc_; }
    IqOptState* h = h_iq_state.data();
    h->mag = iq_mag; h->phase = iq_phase; h->seed = iq_seed;
    CK(cudaMemcpyAsync(d_iq_state.data(), h, sizeof(IqOptState), cudaMemcpyHostToDevice, st));
    CK(cudaStreamSynchronize(st));          // h_iq_state is also the read-back buffer
    return IQGPU_OK;
}

// pre_out: the pre-processor output of this sub-train when it exists in memory (unfused path), else nullptr: the probe
// blocks are then re-computed from the raw frames (convert, DC from the tick table, I/Q apply, NCO — the K1 kernel on 1024
// frames per eligible chunk)
int iqgpu_chain::iq_run_probes(const void* d_rawp, const float2* pre_out, uint64_t N0, const uint32_t* chunks, size_t n_chunks,
                               int slot, cudaStream_t st)
{
    if (!iq_optimize || !cfg.iq_correction_enable) return IQGPU_OK;
    std::vector<uint64_t> pos_list;
    uint64_t pos = N0;
    for (size_t c = 0; c < n_chunks; c++) {
        const double t = (double)pos / (double)in_rate;
        if (chunks[c] >= 1024 && (t - iq_last_attempt_s) * 1000.0 >= iq_interval_ms) {       // pipeline.c:469, iq_correct.c:157-162
            bool ok = true;
            if (!pre_out && dc.enable && !fused_dc_state_at(fused.get(), slot, (int64_t)N0, (int64_t)pos)) ok = false;
            if (ok) { pos_list.push_back(pos); iq_last_attempt_s = t; }
        }
        pos += chunks[c];
    }
    if (pos_list.empty()) return IQGPU_OK;
    if (!d_iq_state.data()) { int rc_ = iq_push_state(st); if (rc_) return rc_; }
    CK(d_iq_probe.grow(pos_list.size() * 1024, (pos_list.size() * 2 + 8) * 1024, [&] {
        const cudaError_t e = cudaStreamSynchronize(st);
        return e != cudaSuccess ? e : cudaStreamSynchronize(aux);
    }));
    if (iq_pending) CK(cudaStreamWaitEvent(st, ev_iq, 0));      // the previous train's passes still read the probe buffer
    for (size_t i = 0; i < pos_list.size(); i++) {
        const uint64_t p0 = pos_list[i];
        float2* dst = d_iq_probe.data() + i * 1024;
        if (pre_out) {
            CK(cudaMemcpyAsync(dst, pre_out + (p0 - N0), 1024 * sizeof(float2), cudaMemcpyDeviceToDevice, st));
        } else {
            const PreParams pp = pre_params(p0);
            const double2* v = dc.enable ? fused_dc_state_at(fused.get(), slot, (int64_t)N0, (int64_t)p0) : nullptr;
            CK(launch_pre(reinterpret_cast<const char*>(d_rawp) + (p0 - N0) * in_bps, 1024, pp, 1024, v, dst, st));
            launches++;
        }
    }
    // the passes themselves run on the second stream: the post kernels of this sub-train do not wait for them
    CK(cudaEventRecord(ev_iq_probe, st));
    CK(cudaStreamWaitEvent(aux, ev_iq_probe, 0));
    CK(launch_iq_optimize_train(d_iq_probe.data(), (int)pos_list.size(), d_iq_state.data(), aux));
    launches++;
    CK(cudaMemcpyAsync(h_iq_state.data(), d_iq_state.data(), sizeof(IqOptState), cudaMemcpyDeviceToHost, aux));
    CK(cudaEventRecord(ev_iq, aux));
    iq_pending = true;
    return IQGPU_OK;
}

// FFT block filter over the fft_rem frames that wait in front of `src` and the n new ones: the whole blocks go to `out`
// (*y: first output sample, *ny: their count), the rest waits for the next call
int iqgpu_chain::fft_block_pass(const float2* src, size_t n, DevStream& out, cudaStream_t st, const float2** y, size_t* ny)
{
    const uint32_t B = filt.block, tot = fft_rem + (uint32_t)n, blocks = tot / B;
    float2* yo = nullptr;
    CK(out.begin((size_t)blocks * B, st, &yo));
    if (blocks) {
        CK(ensure_fft_scratch(blocks, B, st));
        CK(launch_fftfilt(src - fft_rem, blocks, B, d_fft_H.data(), d_fft_tw.data(), yo, d_fft_scratch.data(), &launches, st));
    }
    out.commit((size_t)blocks * B);
    fft_rem = tot - blocks * B;
    *y = yo; *ny = (size_t)blocks * B;
    return IQGPU_OK;
}

// copies a chunk table of n_chunks + 1 entries, written by fill(), to `dst` on `st` through pinned staging: an async copy
// from pageable memory would first drain the stream.  Two slots, each reused once its previous copy has finished.
template <typename Fill>
int iqgpu_chain::stage_chunk_table(uint32_t* dst, size_t n_chunks, cudaStream_t st, Fill fill)
{
    const size_t need = n_chunks + 1;
    const int sl = seg_pin_slot ^= 1;
    CK(cudaEventSynchronize(ev_seg[sl]));
    CK(seg_pin[sl].grow(need, need * 2, no_drain));
    fill(seg_pin[sl].data());
    CK(cudaMemcpyAsync(dst, seg_pin[sl].data(), need * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    CK(cudaEventRecord(ev_seg[sl], st));
    return IQGPU_OK;
}

// ---------------------------------------------------------------------------------------------
// one sub-train on the device
// ---------------------------------------------------------------------------------------------
int iqgpu_chain::run_subtrain(const void* d_rawp, size_t n, const uint32_t* chunks, size_t n_chunks, void* d_outp,
                              size_t* out_frames, uint32_t* per_chunk, cudaStream_t st, int phase)
{
    const bool pre_filter = filt.impl != IQGPU_FILTER_IMPL_NONE && !filt.post_resample;
    const bool post_filter = filt.impl != IQGPU_FILTER_IMPL_NONE && filt.post_resample;
    const uint64_t N0 = n_in, N1 = n_in + n;

    // ---------------- closed-form bookkeeping: per-chunk frame counts ----------------
    std::vector<uint32_t> seg(n_chunks + 1, 0), counts(n_chunks, 0);
    count_outputs(chunks, n_chunks, counts.data());
    for (size_t c = 0; c < n_chunks; c++) {
        seg[c + 1] = seg[c] + counts[c];
        if (per_chunk) per_chunk[c] = counts[c];
    }
    const size_t total_out = seg[n_chunks];
    launches = 0;
    fir_wrote_output = false;
    rms_ready = false;
    if (iq_optimize) { int rc_iq = iq_sync_state(); if (rc_iq) return rc_iq; }      // factors the last train's passes left

    // ---------------- K1: pre-processor ----------------
    const PreParams pp = pre_params(N0);
    const bool use_fused = fused_active;
    const float2* post_src = nullptr;
    size_t post_n = 0;
    if (use_fused) {
        // ---------------- fused K1+K2: one pass over HBM ----------------
        const uint64_t O0 = resampler_outputs_after(rs, N0), O1 = resampler_outputs_after(rs, N1);
        float2* y_rs = nullptr;
        CK(s_rs.begin((size_t)(O1 - O0), st, &y_rs));
        if (dc_prepared) CK(cudaStreamWaitEvent(st, ev_pre[dc_slot], 0));   // the slot's table was built on `aux`
        span_begin(IQGPU_KCLASS_FUSED_FRONT, st);
        // a time-domain FIR right behind the resampler adds the front's closed-form DC term while it stages its tiles
        // (no extra pass over the resampled stream); whoever else reads the stream needs it in memory
        const bool fold_ok = post_filter && filter_is_fir(filt) && !fir_via_fft && !record_taps &&
                             fir_can_fold_dc(fir_taps_padded, filt.impl == IQGPU_FILTER_IMPL_FIR_ASYM, !h_fir_taps.empty());
        dc_fold.corr = nullptr;
        CK(fused_launch(fused.get(), d_rawp, (int64_t)N0, n, pp, d_dc_carry.data(), (int64_t)O0, (size_t)(O1 - O0), y_rs, &launches, dc_slot, st,
                        fold_ok ? &dc_fold : nullptr));
        span_end(st);
        { int rc_iq = iq_run_probes(d_rawp, nullptr, N0, chunks, n_chunks, dc_slot, st); if (rc_iq) return rc_iq; }
        if (dc.enable) { CK(cudaEventRecord(ev_front[dc_slot], st)); front_recorded[dc_slot] = true; }
        dc_prepared = false;
        s_rs.commit((size_t)(O1 - O0));
        post_src = y_rs; post_n = (size_t)(O1 - O0);
        fused_used = true;
    } else {
        float2* x_in = nullptr;
        CK(s_in.begin(n, st, &x_in));
        uint32_t rows = (uint32_t)((n + 127) / 128), rpr = 1;
        while (rpr < 32 && rows / rpr > 16384) rpr <<= 1;
        const uint32_t run_len = 128 * rpr;
        if (dc.enable && dc_mode == 1) {
            // reference rounding: convert, then liquid's fp32 recurrence literally (serial), then I/Q apply + NCO in place
            PreParams p1 = pp;
            p1.dc_enable = 0; p1.iq_enable = 0; p1.nco_enable = 0;
            span_begin(IQGPU_KCLASS_PRE, st);
            CK(launch_pre(d_rawp, n, p1, run_len, nullptr, x_in, st));
            span_end(st);
            span_begin(IQGPU_KCLASS_DC_SCAN, st);
            CK(launch_dc_reference(x_in, n, dc.c, d_dc_ref.data(), st));
            span_end(st);
            launches += 2;
            if (pp.iq_enable || pp.nco_enable) {
                PreParams p2 = pp;
                p2.format = IQGPU_FMT_CF32; p2.gain = 1.0f; p2.dc_enable = 0;
                span_begin(IQGPU_KCLASS_PRE, st);
                CK(launch_pre(x_in, n, p2, run_len, nullptr, x_in, st));
                span_end(st);
                launches++;
            }
        } else {
            if (dc.enable) {
                const size_t n_runs = (n + run_len - 1) / run_len;
                if (n_runs > d_run_sums.size()) return fail(IQGPU_EINVAL, "internal: run table too small");
                span_begin(IQGPU_KCLASS_DC_SCAN, st);
                CK(launch_dc_run_sums(d_rawp, n, pp, run_len, d_run_sums.data(), st));
                CK(launch_dc_scan(d_run_sums.data(), n_runs, run_len, n, dc.c, d_dc_carry.data(), d_run_start.data(),
                                  d_scan_ws.data(), st));
                span_end(st);
                launches += 2;
            }
            span_begin(IQGPU_KCLASS_PRE, st);
            CK(launch_pre(d_rawp, n, pp, run_len, d_run_start.data(), x_in, st));
            span_end(st);
            launches++;
        }
        s_in.commit(n);
        if (record_tap0) CK(tap[0].append(x_in, n, st));
        if (!(pre_filter && filter_is_fir(filt))) { int rc_iq = iq_run_probes(d_rawp, x_in, N0, chunks, n_chunks, 0, st); if (rc_iq) return rc_iq; }

        // ---------------- optional pre-resample filter ----------------
        const float2* rs_src = x_in;     // stream feeding the resampler (first new sample)
        size_t rs_n = n;                 // new samples in it
        uint64_t rs_pos0 = N0;           // absolute index of rs_src[0] in the resampler input stream
        if (pre_filter) {
            if (filter_is_fir(filt)) {
                float2* y = nullptr;
                CK(s_pref.begin(n, st, &y));
                CK(launch_fir(x_in, n, d_fir_taps.data(), fir_taps_padded, filt.impl == IQGPU_FILTER_IMPL_FIR_ASYM, y, st, h_fir_taps.data()));
                launches++;
                s_pref.commit(n);
                rs_src = y;
                // the reference probes buffer A after the whole pre chain, i.e. behind a pre-resample FIR (pipeline.c:466-472)
                { int rc_iq = iq_run_probes(d_rawp, y, N0, chunks, n_chunks, 0, st); if (rc_iq) return rc_iq; }
            } else {
                rs_pos0 = N0 + fft_rem_carry - fft_rem;
                int rc = fft_block_pass(x_in, n, s_pref, st, &rs_src, &rs_n);
                if (rc) return rc;
            }
        }

        // ---------------- K2: resampler ----------------
        post_src = rs_src;
        post_n = rs_n;
        if (!rs.passthrough) {
            span_begin(IQGPU_KCLASS_RESAMPLER, st);
            const unsigned S = rs.num_halfband;
            const uint64_t P0 = rs_pos0, P1 = rs_pos0 + rs_n;
            float2* y_rs = nullptr;
            if (!rs.is_interp) {
                const float2* src = rs_src;
                uint64_t a0 = P0;  // absolute index (in the current stage's input stream) of src[0]
                for (unsigned d = 0; d < S; d++) {
                    const unsigned g = S - 1 - d;
                    const uint64_t k0 = P0 >> (d + 1), k1 = P1 >> (d + 1);
                    float2* y = nullptr;
                    CK(s_stage[d].begin((size_t)(k1 - k0), st, &y));
                    CK(launch_halfband_decim(src, (int64_t)a0, d_hb_taps[g].data(), rs.stages[g].m, (int64_t)k0, (size_t)(k1 - k0),
                                             (d + 1 == S) ? rs.zeta : 1.0f, y, st));
                    launches++;
                    s_stage[d].commit((size_t)(k1 - k0));
                    src = y; a0 = k0;
                }
                const uint64_t K0 = P0 >> S, K1 = P1 >> S;
                const uint64_t O0 = arb_outputs_after(K0, rs.step), O1 = arb_outputs_after(K1, rs.step);
                const unsigned __int128 Pph = (unsigned __int128)O0 * rs.step;
                CK(s_rs.begin((size_t)(O1 - O0), st, &y_rs));
                CK(launch_arb(src, (int64_t)K0, d_bank.data(), rs.step, (int64_t)(uint64_t)(Pph >> 24), (uint32_t)(Pph & 0xffffffu),
                              (size_t)(O1 - O0), y_rs, st));
                launches++;
                post_n = (size_t)(O1 - O0);
            } else {
                const uint64_t O0 = arb_outputs_after(P0, rs.step), O1 = arb_outputs_after(P1, rs.step);
                const unsigned __int128 Pph = (unsigned __int128)O0 * rs.step;
                float2* y = nullptr;
                size_t cnt = (size_t)(O1 - O0);
                if (S == 0) CK(s_rs.begin(cnt, st, &y)); else CK(s_arb_in.begin(cnt, st, &y));
                CK(launch_arb(rs_src, (int64_t)P0, d_bank.data(), rs.step, (int64_t)(uint64_t)(Pph >> 24), (uint32_t)(Pph & 0xffffffu), cnt, y, st));
                launches++;
                if (S == 0) y_rs = y; else s_arb_in.commit(cnt);
                const float2* src = y;
                uint64_t a0 = O0;
                for (unsigned s = 0; s < S; s++) {
                    float2* yo = nullptr;
                    if (s + 1 == S) CK(s_rs.begin(2 * cnt, st, &yo)); else CK(s_stage[s].begin(2 * cnt, st, &yo));
                    CK(launch_halfband_interp(src, (int64_t)a0, d_hb_taps[s].data(), rs.stages[s].m, (int64_t)a0, cnt, yo, st));
                    launches++;
                    if (s + 1 == S) y_rs = yo; else s_stage[s].commit(2 * cnt);
                    src = yo; a0 *= 2; cnt *= 2;
                }
                post_n = cnt;
            }
            s_rs.commit(post_n);
            post_src = y_rs;
            span_end(st);
        } else if (post_filter) {
            // passthrough + post filter: the filter-only module chain of a decimating configuration (IQGPU_STAGE_FILTER
            // without IQGPU_STAGE_RESAMPLER).  Copy into s_rs, where the filter finds its history.
            float2* y = nullptr;
            CK(s_rs.begin(rs_n, st, &y));
            CK(cudaMemcpyAsync(y, rs_src, rs_n * sizeof(float2), cudaMemcpyDeviceToDevice, st));
            s_rs.commit(rs_n);
            post_src = y;
        }
    }
    if (record_taps) CK(tap[1].append(post_src, post_n, st));

    // ---------------- optional post-resample filter ----------------
    if (post_filter) {
        span_begin(IQGPU_KCLASS_FILTER, st);
        if (filter_is_fir(filt) && fir_via_fft) {
            // y[n] = sum_k h[k] x[n-k] by overlap-save blocks of 8192 outputs; the last block is completed with zeros beyond
            // the newest sample (its outputs past post_n are never read), the history below post_src is the real stream
            const size_t B = fir_fft_block, blocks = (post_n + B - 1) / B;
            float2* y = nullptr;
            CK(s_f.begin(blocks * B, st, &y));
            if (blocks) {
                if (blocks * B > post_n)
                    CK(cudaMemsetAsync(const_cast<float2*>(post_src) + post_n, 0, (blocks * B - post_n) * sizeof(float2), st));
                CK(ensure_fft_scratch(blocks, (unsigned)B, st));
                CK(launch_fftfilt(post_src, blocks, (unsigned)B, d_fft_H.data(), d_fft_tw.data(), y, d_fft_scratch.data(), &launches,
                                  st));
            }
            s_f.commit(post_n);
            post_src = y;
        } else if (filter_is_fir(filt)) {
            const int cplx = filt.impl == IQGPU_FILTER_IMPL_FIR_ASYM;
            // last cf32 stage of the chain (no post shift, no AGC, nobody records the stream, one-phase call): convert in the
            // filter's epilogue and skip the post kernel
            fir_wrote_output = phase == 0 && !record_taps && !nco_post && agc_mode == 0 && d_outp && post_n == total_out &&
                               fir_can_convert_out(cfg.output_format, fir_taps_padded, cplx);
            float2* y = nullptr;
            CK(s_f.begin(post_n, st, &y));
            const bool folding = use_fused && dc_fold.corr != nullptr;
            CK(launch_fir(post_src, post_n, d_fir_taps.data(), fir_taps_padded, cplx, y, st, h_fir_taps.data(),
                          fir_wrote_output ? cfg.output_format : 0, fir_wrote_output ? d_outp : nullptr,
                          folding ? &dc_fold : nullptr));
            launches++;
            if (folding) {
                // the newest samples stay behind as the next call's filter history: they get the term in memory now
                const size_t keep = std::min(post_n, s_rs.hist);
                CK(fused_dc_correct_range(dc_fold, const_cast<float2*>(post_src), post_n - keep, keep, st));
                if (keep) launches++;
                dc_fold.corr = nullptr;
            }
            s_f.commit(post_n);
            post_src = y;
        } else {
            int rc = fft_block_pass(post_src, post_n, s_f, st, &post_src, &post_n);
            if (rc) return rc;
        }
        span_end(st);
    }
    if (post_n != total_out) return fail(IQGPU_EINVAL, "internal: closed-form output count disagrees with the kernels' count");

    // ---------------- K5: post NCO + AGC + convert ----------------
    PostParams qp{};
    qp.format = cfg.output_format;
    qp.nco_enable = nco_post; qp.nco_dtheta = nco_dtheta; qp.nco_sign = nco_sign; qp.nco_table = d_lut.data();
    qp.nco_theta0 = (uint32_t)((uint64_t)(uint32_t)n_nco_post * nco_dtheta);
    qp.agc_mode = agc_mode; qp.agc_target = agc_target; qp.agc_alpha = agc_alpha; qp.target_rate = target_rate;
    pend.active = true;
    pend.src = post_src; pend.n = post_n; pend.n_chunks = n_chunks;
    pend.seg = seg; pend.counts = counts; pend.qp = qp; pend.peaks_done = false;
    if (post_n && agc_mode == 1) {
        // pass 1 of the digital AGC: per-chunk peaks (agc.c:117-124).  Everything after this is a
        // function of the peaks and the carried AGC state only.
        span_begin(IQGPU_KCLASS_POST, st);
        auto drain = [st] { return cudaStreamSynchronize(st); };
        CK(d_seg_start.grow(n_chunks + 1, n_chunks * 2 + 1, drain));
        CK(d_seg_peak.grow(n_chunks, n_chunks * 2, drain));
        CK(d_seg_gain.grow(n_chunks, n_chunks * 2, drain));
        { int rc = stage_chunk_table(d_seg_start.data(), n_chunks, st, [&](uint32_t* t) { std::copy(seg.begin(), seg.end(), t); }); if (rc) return rc; }
        CK(launch_agc_peaks(post_src, post_n, qp, d_seg_start.data(), n_chunks, d_seg_peak.data(), st));
        span_end(st);
        launches += 1;
        pend.peaks_done = true;
    }
    if (nco_post) n_nco_post += post_n;
    n_in = N1;
    n_out += post_n;
    *out_frames = post_n;
    if (phase == 1) return IQGPU_OK;
    return run_back(d_outp, 0, out_frames, st);
}

// back half of a sub-train: AGC state machine over the chunk peaks, scale, output conversion.
// skip_chunks: leading chunks that belong to a shard's halo — they get unit gain and do not
// advance the AGC state (their output frames are dropped by the caller).
int iqgpu_chain::run_back(void* d_outp, size_t skip_chunks, size_t* out_frames, cudaStream_t st)
{
    if (!pend.active) return fail(IQGPU_EINVAL, "no pending sub-train");
    pend.active = false;
    const float2* post_src = pend.src;
    const size_t post_n = pend.n, n_chunks = pend.n_chunks;
    const PostParams& qp = pend.qp;
    if (skip_chunks > n_chunks) return fail(IQGPU_EINVAL, "skip_chunks exceeds the chunk count");
    float2* tap2 = nullptr;
    if (record_taps && post_n) {
        // reserve room in the tap buffer and let the post kernel write straight into it
        CK(tap[2].append(post_src, post_n, st));
        tap2 = tap[2].buf.data() + tap[2].len - post_n;
    }
    if (post_n && fir_wrote_output) {
        fir_wrote_output = false;        // the FIR epilogue already produced the final stream (run_subtrain)
    } else if (post_n) {
        span_begin(IQGPU_KCLASS_POST, st);
        if (agc_mode == 1) {
            if (skip_chunks) {
                const std::vector<float> ones(skip_chunks, 1.0f);
                CK(cudaMemcpyAsync(d_seg_gain.data(), ones.data(), skip_chunks * sizeof(float), cudaMemcpyHostToDevice, st));
            }
            CK(ensure_agc_quiet(n_chunks, st));
            CK(launch_agc_digital_scan(d_seg_start.data() + skip_chunks, n_chunks - skip_chunks, d_seg_peak.data() + skip_chunks, qp,
                                       d_agc.data(), d_seg_gain.data() + skip_chunks, st, d_agc_quiet.data()));
            CK(launch_post(post_src, post_n, qp, d_seg_start.data(), n_chunks, d_seg_gain.data(), 0, tap2, d_outp, st));
            launches += 2;
        } else if (agc_mode == 2) {
            auto drain = [st] { return cudaStreamSynchronize(st); };
            CK(d_agc_scratch.grow(post_n, post_n + post_n / 2 + 1024, drain));
            float2* y = d_agc_scratch.data();
            const size_t ws_need = agc_rms_workspace_bytes(post_n, qp.agc_alpha);
            CK(d_agc_ws.grow(ws_need, ws_need * 2, drain));
            static_assert(offsetof(AgcState, rms_y2) == offsetof(AgcState, rms_g) + sizeof(float), "{g, y2'} must be adjacent");
            CK(cudaMemcpyAsync(&d_rms_rerun.data()->rms_g, &d_agc.data()->rms_g, 2 * sizeof(float), cudaMemcpyDeviceToDevice, st));
            CK(launch_agc_rms(post_src, post_n, qp, d_agc.data(), y, d_agc_ws.data(), st));
            CK(launch_post(y, post_n, qp, nullptr, 0, nullptr, 1, tap2, d_outp, st));
            launches += 2;
            rms_src = post_src; rms_n = post_n; rms_qp = qp; rms_ready = true; rms_fresh = true; rms_resume_max = 0;
        } else {
            CK(launch_post(post_src, post_n, qp, nullptr, 0, nullptr, 0, tap2, d_outp, st));
            launches++;
        }
        span_end(st);
    }
    if (out_frames) *out_frames = post_n;
    return IQGPU_OK;
}

// =============================================================================================
// C ABI
// =============================================================================================
extern "C" {

int iqgpu_abi_version(void) { return IQGPU_ABI_VERSION; }
const char* iqgpu_last_error(void) { return g_err.c_str(); }
int iqgpu_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}
void* iqgpu_host_alloc(size_t bytes)
{
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void iqgpu_host_free(void* p) { if (p) cudaFreeHost(p); }
size_t iqgpu_get_bytes_per_sample(int format) { return bytes_per_sample(format); }

static int chain_create_impl(const iqgpu_chain_config* cfgp, int device, iqgpu_chain** out)
{
    if (!cfgp || !out) return fail(IQGPU_EINVAL, "null argument");
    *out = nullptr;
    const iqgpu_chain_config& g = *cfgp;
    if (!is_complex_format(g.input_format) || !bytes_per_sample(g.input_format))
        return fail(IQGPU_EINVAL, "unhandled input format");       // sample_convert.c:207
    if (!is_complex_format(g.output_format) || !bytes_per_sample(g.output_format))
        return fail(IQGPU_EINVAL, "unhandled output format");      // sample_convert.c:304
    std::unique_ptr<iqgpu_chain> c(new iqgpu_chain());
    c->cfg = g;
    c->device = device;
    c->plan_only = device < 0;
    c->in_rate = (int)g.input_rate_hz;
    c->target_rate = g.target_rate_hz;
    c->in_bps = bytes_per_sample(g.input_format);
    c->out_bps = bytes_per_sample(g.output_format);
    std::string err;
    if (c->in_rate <= 0) return fail(IQGPU_EINVAL, "input sample rate must be positive");
    // setup.c:91-113
    if (g.no_resample) c->target_rate = (double)c->in_rate;
    c->ratio = (float)(c->target_rate / (double)c->in_rate);
    if (!std::isfinite(c->ratio) || c->ratio < 0.001f || c->ratio > 1000.0f)
        return fail(IQGPU_EINVAL, "resampling ratio invalid or outside the acceptable range");
    c->dc = design_dc(g.dc_block_enable != 0, c->in_rate);
    if (g.dc_block_enable && c->dc.alpha <= 0.0f) return fail(IQGPU_EINVAL, "DC block alpha invalid");
    c->iq_mag = g.iq_mag; c->iq_phase = g.iq_phase;
    // frequency_shift.c:24-84
    // AppResources.nco_shift_hz is a double (frequency_shift.c:32-33 widens the float CLI argument, input_wav.c:614-628
    // stores centre - (double)target): no float round trip here, callers that emulate --freq-shift cast themselves
    const double shift = g.freq_shift_hz;
    if (g.shift_after_resample && std::fabs(shift) < 1e-9)
        return fail(IQGPU_EINVAL, "--shift-after-resample used without an effective frequency shift");
    if (std::fabs(shift) >= 1e-9) {
        const double rate = g.shift_after_resample ? c->target_rate : (double)c->in_rate;
        if (std::fabs(shift) > 5.0 * rate) return fail(IQGPU_EINVAL, "frequency shift exceeds the sanity limit");
        c->nco_dtheta = nco_dtheta_for_shift(shift, rate);
        c->nco_sign = shift >= 0 ? 1.0f : -1.0f;
        c->nco_pre = !g.shift_after_resample;
        c->nco_post = g.shift_after_resample != 0;
    }
    if (!design_resampler(c->ratio, 60.0f, g.no_resample != 0, c->rs, err)) return fail(IQGPU_EINVAL, err);
    if (!design_filter(g, c->in_rate, c->target_rate, c->filt, err)) return fail(IQGPU_EINVAL, err);
    // agc.c:21-84
    if (g.agc_enable && g.agc_profile != IQGPU_AGC_OFF) {
        if (g.agc_profile == IQGPU_AGC_DIGITAL) {
            c->agc_mode = 1;
            c->agc_target = (g.agc_target_level_arg > 0) ? g.agc_target_level_arg : 0.9f;
        } else {
            c->agc_mode = 2;
            c->agc_alpha = (g.agc_profile == IQGPU_AGC_DX) ? 1e-4f : 1e-2f;
        }
    }
    if (g.stage_select) {
        // module-level chain: designed from the full configuration, runs only the selected stages cf32 -> cf32
        const int m = g.stage_select;
        c->cfg.input_format = IQGPU_FMT_CF32; c->cfg.output_format = IQGPU_FMT_CF32; c->cfg.gain = 1.0f;
        c->in_bps = c->out_bps = bytes_per_sample(IQGPU_FMT_CF32);
        if (!(m & IQGPU_STAGE_DC)) { c->dc.enable = false; c->cfg.dc_block_enable = 0; }
        if (!(m & IQGPU_STAGE_IQ)) c->cfg.iq_correction_enable = 0;
        if (!(m & IQGPU_STAGE_NCO)) { c->nco_pre = c->nco_post = false; }
        if (!(m & IQGPU_STAGE_FILTER)) c->filt = FilterPlan();
        if (!(m & IQGPU_STAGE_AGC)) c->agc_mode = 0;
        if (!(m & IQGPU_STAGE_RESAMPLER)) {
            c->rs = ResamplerPlan();
            if (!design_resampler(1.0f, 60.0f, true, c->rs, err)) return fail(IQGPU_EINVAL, err);
        }
    }
    if (!c->plan_only) {
        int rc = c->init_device();
        if (rc != IQGPU_OK) return rc;
    }
    *out = c.release();
    return IQGPU_OK;
}

// No C++ exception may cross the C ABI: a configuration whose design cannot be carried out (a tap count that does not
// fit memory, a length that went negative before its cast ...) is refused like any other invalid configuration.
int iqgpu_chain_create(const iqgpu_chain_config* cfgp, int device, iqgpu_chain** out)
{
    try {
        return chain_create_impl(cfgp, device, out);
    } catch (const std::bad_alloc&) {
        if (out) *out = nullptr;
        return fail(IQGPU_ENOMEM, "out of host memory while designing the chain");
    } catch (const std::exception& e) {
        if (out) *out = nullptr;
        return fail(IQGPU_EINVAL, std::string("configuration cannot be designed: ") + e.what());
    }
}

void iqgpu_chain_destroy(iqgpu_chain* c) { delete c; }

int iqgpu_chain_reset(iqgpu_chain* c)
{
    if (!c) return fail(IQGPU_EINVAL, "null chain");
    return c->reset_state(true);
}

int iqgpu_chain_restart(iqgpu_chain* c)
{
    if (!c) return fail(IQGPU_EINVAL, "null chain");
    return c->reset_state(false);
}

int iqgpu_chain_set_option(iqgpu_chain* c, const char* key, int64_t value)
{
    if (!c || !key) return fail(IQGPU_EINVAL, "null argument");
    const std::string k(key);
    if (k == "fused") {
        if (c->buffers_ready) return fail(IQGPU_EINVAL, "option must be set before the first process call");
        c->want_fused = value != 0;
        return IQGPU_OK;
    }
    if (k == "iq_optimize") { c->iq_optimize = value != 0; return IQGPU_OK; }
    if (k == "iq_optimize_interval_ms") { if (value < 0) return fail(IQGPU_EINVAL, "negative interval"); c->iq_interval_ms = (double)value; return IQGPU_OK; }
    if (k == "iq_optimize_seed") { c->iq_seed = (uint32_t)value; if (c->d_iq_state.data()) return c->iq_push_state(c->last_stream ? c->last_stream : c->stream); return IQGPU_OK; }
    if (k == "dc_mode") {
        if (c->buffers_ready) return fail(IQGPU_EINVAL, "option must be set before the first process call");
        if (value != 0 && value != 1) return fail(IQGPU_EINVAL, "dc_mode: 0 (exact arithmetic) or 1 (reference fp32 state rounding)");
        c->dc_mode = (int)value;
        return IQGPU_OK;
    }
    if (k == "record_taps") {
        if (c->buffers_ready && (value > 1) != c->record_tap0) return fail(IQGPU_EINVAL, "record_taps=2 must be set before the first process call");
        c->record_taps = value != 0; c->record_tap0 = value > 1;
        return IQGPU_OK;
    }
    if (k == "time_kernels") { c->time_kernels = value != 0; return IQGPU_OK; }
    if (k == "dc_overlap") { c->dc_overlap = value != 0; return IQGPU_OK; }
    if (k == "subtrain_frames" || k == "chunk_frames") {
        if (c->buffers_ready) return fail(IQGPU_EINVAL, "option must be set before the first process call");
        if (value <= 0) return fail(IQGPU_EINVAL, "value must be positive");
        if (k == "chunk_frames") c->chunk_frames = (uint32_t)value;
        else c->subtrain_frames = (size_t)value;
        return IQGPU_OK;
    }
    return fail(IQGPU_EINVAL, "unknown option");
}

int iqgpu_chain_get_kernel_times(iqgpu_chain* c, double* ms, uint32_t* launches, int reset)
{
    if (!c) return fail(IQGPU_EINVAL, "null chain");
    if (!c->plan_only) { cudaSetDevice(c->device); c->collect_spans(); }
    for (int i = 0; i < IQGPU_KCLASS_COUNT; i++) {
        if (ms) ms[i] = c->class_ms[i];
        if (launches) launches[i] = c->class_launches[i];
        if (reset) { c->class_ms[i] = 0; c->class_launches[i] = 0; }
    }
    return IQGPU_OK;
}

int iqgpu_chain_set_iq_factors(iqgpu_chain* c, float mag, float phase)
{
    if (!c) return fail(IQGPU_EINVAL, "null chain");
    if (c->d_iq_state.data()) {
        int rc = c->iq_sync_state();
        if (rc) return rc;
        c->iq_mag = mag; c->iq_phase = phase;
        return c->iq_push_state(c->last_stream ? c->last_stream : c->stream);
    }
    c->iq_mag = mag; c->iq_phase = phase;
    return IQGPU_OK;
}

int iqgpu_chain_get_iq_state(iqgpu_chain* c, float* mag, float* phase, uint64_t* passes, uint64_t* attempts)
{
    if (!c) return fail(IQGPU_EINVAL, "null chain");
    if (!c->plan_only) { CK(cudaSetDevice(c->device)); int rc = c->iq_sync_state(); if (rc) return rc; }
    if (mag) *mag = c->iq_mag;
    if (phase) *phase = c->iq_phase;
    if (passes) *passes = c->h_iq_state.data() ? c->h_iq_state.data()->passes : 0;
    if (attempts) *attempts = c->h_iq_state.data() ? c->h_iq_state.data()->attempts : 0;
    return IQGPU_OK;
}

int iqgpu_chain_get_info(iqgpu_chain* c, iqgpu_chain_info* o)
{
    if (!c || !o) return fail(IQGPU_EINVAL, "null argument");
    memset(o, 0, sizeof(*o));
    o->ratio = c->ratio;
    o->is_interp = c->rs.is_interp;
    o->num_halfband = c->rs.num_halfband;
    for (unsigned i = 0; i < c->rs.num_halfband && i < 16; i++) o->halfband_m[i] = c->rs.stages[i].m;
    o->rate_arbitrary = c->rs.rate_arbitrary;
    o->arb_step = c->rs.passthrough ? 0 : c->rs.step;
    o->filter_impl = c->filt.impl;
    o->filter_post_resample = c->filt.post_resample;
    o->filter_block_size = c->filt.block;
    o->filter_num_taps = (uint32_t)c->filt.taps.size();
    o->nco_dtheta = c->nco_dtheta;
    o->nco_is_post = c->nco_post;
    o->frames_in_total = c->n_in;
    o->frames_out_total = c->n_out;
    o->fused_front = c->fused_used ? 1 : 0;
    o->kernel_launches = c->launches;
    o->halo_frames = c->fused ? fused_halo_frames(c->fused.get()) : (uint32_t)c->rs.halo_input_frames;
    if (!c->plan_only && c->d_agc.data()) {
        AgcState a{};
        cudaSetDevice(c->device);
        if (c->last_stream) cudaStreamSynchronize(c->last_stream);
        cudaStreamSynchronize(c->stream);
        if (cudaMemcpy(&a, c->d_agc.data(), sizeof(a), cudaMemcpyDeviceToHost) == cudaSuccess) {
            o->agc_locked = a.locked; o->agc_gain = a.gain; o->agc_peak_memory = a.peak_mem; o->agc_samples_seen = a.seen;
        }
    }
    return IQGPU_OK;
}

static int build_chunks(iqgpu_chain* c, size_t n_frames, const uint32_t* chunk_frames, size_t n_chunks,
                        std::vector<uint32_t>& chunks)
{
    // the chunk table is host memory (4 B per chunk): a train beyond 2^30 chunks (1.7e13 frames) is refused rather than
    // allowed to exhaust it, and no allocation failure may leave the C ABI as a C++ exception
    constexpr size_t kMaxTrainChunks = (size_t)1 << 30;
    try {
        if (chunk_frames) {
            if (n_chunks > kMaxTrainChunks) return fail(IQGPU_EINVAL, "train too long: more than 2^30 chunks in one call");
            size_t sum = 0;
            chunks.assign(chunk_frames, chunk_frames + n_chunks);
            for (auto f : chunks) sum += f;
            if (sum != n_frames) return fail(IQGPU_EINVAL, "chunk lengths do not add up to n_frames");
        } else {
            const size_t per = std::max<uint32_t>(1, c->chunk_frames);
            if (n_frames / per >= kMaxTrainChunks) return fail(IQGPU_EINVAL, "train too long: more than 2^30 chunks in one call");
            chunks.clear();
            chunks.reserve(n_frames / per + 1);
            size_t left = n_frames;
            while (left) {
                uint32_t f = (uint32_t)std::min<size_t>(left, per);
                chunks.push_back(f);
                left -= f;
            }
        }
    } catch (const std::exception&) {
        return fail(IQGPU_ENOMEM, "out of host memory for the chunk table");
    }
    return IQGPU_OK;
}

int iqgpu_chain_resampler_outputs_after(iqgpu_chain* c, uint64_t frames_in, uint64_t* frames_out)
{
    if (!c || !frames_out) return fail(IQGPU_EINVAL, "null argument");
    *frames_out = resampler_outputs_after(c->rs, frames_in);
    return IQGPU_OK;
}

int iqgpu_chain_predict_output(iqgpu_chain* c, size_t n_frames, size_t* out_frames)
{
    if (!c || !out_frames) return fail(IQGPU_EINVAL, "null argument");
    std::vector<uint32_t> chunks;
    int rc = build_chunks(c, n_frames, nullptr, 0, chunks);
    if (rc) return rc;
    *out_frames = c->count_outputs(chunks.data(), chunks.size(), nullptr);
    return IQGPU_OK;
}

int iqgpu_chain_process_device(iqgpu_chain* c, const void* dev_raw_in, size_t n_frames, const uint32_t* chunk_frames,
                               size_t n_chunks, void* dev_out, size_t out_capacity_bytes, size_t* out_frames,
                               uint32_t* per_chunk_out, void* cuda_stream)
{
    if (!c || !out_frames) return fail(IQGPU_EINVAL, "null argument");
    if (c->plan_only) return fail(IQGPU_ENODEVICE, "chain was created without a device (plan only)");
    *out_frames = 0;
    if (n_frames == 0) return IQGPU_OK;
    if (!dev_raw_in || !dev_out) return fail(IQGPU_EINVAL, "null buffer");
    CK(cudaSetDevice(c->device));
    int rc = c->ensure_buffers();
    if (rc) return rc;
    std::vector<uint32_t> chunks;
    rc = build_chunks(c, n_frames, chunk_frames, n_chunks, chunks);
    if (rc) return rc;
    for (auto f : chunks)
        if (f > c->subtrain_frames) return fail(IQGPU_EINVAL, "a chunk exceeds subtrain_frames");
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : c->stream;
    c->last_stream = st;
    rc = c->order_after_reset(st);
    if (rc) return rc;
    if (c->count_outputs(chunks.data(), chunks.size(), nullptr) * c->out_bps > out_capacity_bytes)
        return fail(IQGPU_ECAPACITY, "output buffer too small");
    for (auto& t : c->tap) t.len = 0;
    // cut the train into sub-trains up front so that the DC pre-pass can run one sub-train ahead
    struct Sub { size_t c0, c1, in_off, n; };
    std::vector<Sub> subs;
    {
        size_t ci = 0, in_off = 0;
        while (ci < chunks.size()) {
            size_t cj = ci, n = 0;
            while (cj < chunks.size() && n + chunks[cj] <= c->subtrain_frames) { n += chunks[cj]; cj++; }
            subs.push_back({ci, cj, in_off, n});
            in_off += n;
            ci = cj;
        }
    }
    const bool overlap_dc = c->fused_active && c->dc.enable && c->dc_overlap;
    const uint64_t base_in = c->n_in;
    auto raw_at = [&](const Sub& sb) { return (const void*)((const char*)dev_raw_in + sb.in_off * c->in_bps); };
    int slot = 0;
    if (overlap_dc) {
        // the second stream starts after everything already queued on the caller's stream
        CK(cudaEventRecord(c->ev_call, st));
        CK(cudaStreamWaitEvent(c->aux, c->ev_call, 0));
        rc = c->prepare_dc(slot, raw_at(subs[0]), base_in + subs[0].in_off, subs[0].n, st);
        if (rc) return rc;
    }
    size_t out_off = 0, total = 0;
    uint32_t launches = 0;
    for (size_t k = 0; k < subs.size(); k++) {
        const Sub& sb = subs[k];
        if (overlap_dc) { c->dc_slot = slot; c->dc_prepared = true; }
        else { c->dc_slot = 0; c->dc_prepared = false; }
        size_t produced = 0;
        rc = c->run_subtrain(raw_at(sb), sb.n, chunks.data() + sb.c0, sb.c1 - sb.c0,
                             (char*)dev_out + out_off, &produced, per_chunk_out ? per_chunk_out + sb.c0 : nullptr, st);
        if (rc) return rc;
        launches += c->launches;
        if (overlap_dc && k + 1 < subs.size()) {
            // The pre-pass of the NEXT sub-train (HBM bound, few FMAs) runs on the second stream next to this sub-train's
            // filter / post kernels (FMA bound, little HBM traffic); it is gated behind this sub-train's fused front kernel,
            // which it would only slow down (both lean on the LSU pipe; measured, DESIGN.md 8).
            const uint32_t keep = c->launches;
            CK(cudaStreamWaitEvent(c->aux, c->ev_front[slot], 0));
            rc = c->prepare_dc(slot ^ 1, raw_at(subs[k + 1]), base_in + subs[k + 1].in_off, subs[k + 1].n, st);
            if (rc) return rc;
            c->launches = keep;
        }
        out_off += produced * c->out_bps; total += produced;
        slot ^= 1;
    }
    c->launches = launches + c->prepass_launches;   // pre-pass kernels that really ran on the second stream
    c->prepass_launches = 0;
    if (subs.size() != 1) c->rms_ready = false;     // an RMS-AGC resume needs the whole call in one sub-train
    *out_frames = total;
    return IQGPU_OK;
}

// ---- sharded digital AGC: the process_device call split at its only data-dependent exchange point ----
int iqgpu_chain_process_device_begin(iqgpu_chain* c, const void* dev_raw_in, size_t n_frames, const uint32_t* chunk_frames,
                                     size_t n_chunks, void* cuda_stream)
{
    if (!c) return fail(IQGPU_EINVAL, "null argument");
    if (c->plan_only) return fail(IQGPU_ENODEVICE, "chain was created without a device (plan only)");
    if (n_frames == 0 || !dev_raw_in) return fail(IQGPU_EINVAL, "empty input");
    if (c->pend.active) return fail(IQGPU_EINVAL, "a begun call is still pending (call process_device_finish)");
    CK(cudaSetDevice(c->device));
    int rc = c->ensure_buffers();
    if (rc) return rc;
    std::vector<uint32_t> chunks;
    rc = build_chunks(c, n_frames, chunk_frames, n_chunks, chunks);
    if (rc) return rc;
    if (n_frames > c->subtrain_frames)
        return fail(IQGPU_EINVAL, "a begun call must fit one sub-train (raise the subtrain_frames option)");
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : c->stream;
    c->last_stream = st;
    rc = c->order_after_reset(st);
    if (rc) return rc;
    for (auto& t : c->tap) t.len = 0;
    size_t produced = 0;
    c->dc_slot = 0; c->dc_prepared = false;
    rc = c->run_subtrain(dev_raw_in, n_frames, chunks.data(), chunks.size(), nullptr, &produced, nullptr, st, 1);
    if (rc) { c->pend.active = false; return rc; }
    return IQGPU_OK;
}

int iqgpu_chain_pending_chunk_peaks(iqgpu_chain* c, float* peaks, uint32_t* counts, size_t capacity, size_t* n_chunks)
{
    if (!c || !n_chunks) return fail(IQGPU_EINVAL, "null argument");
    if (!c->pend.active) return fail(IQGPU_EINVAL, "no pending call");
    *n_chunks = c->pend.n_chunks;
    if (!peaks && !counts) return IQGPU_OK;
    if (capacity < c->pend.n_chunks) return fail(IQGPU_ECAPACITY, "peak buffer too small");
    if (counts) std::copy(c->pend.counts.begin(), c->pend.counts.end(), counts);
    if (peaks) {
        if (c->pend.peaks_done) {
            CK(cudaSetDevice(c->device));
            CK(cudaMemcpyAsync(peaks, c->d_seg_peak.data(), c->pend.n_chunks * sizeof(float), cudaMemcpyDeviceToHost, c->last_stream));
            CK(cudaStreamSynchronize(c->last_stream));
        } else std::fill(peaks, peaks + c->pend.n_chunks, 0.0f);
    }
    return IQGPU_OK;
}

int iqgpu_chain_pending_chunk_peaks_device(iqgpu_chain* c, size_t skip_chunks, float* dev_peaks, size_t capacity,
                                           size_t* n_chunks, void* cuda_stream)
{
    if (!c || !n_chunks) return fail(IQGPU_EINVAL, "null argument");
    if (!c->pend.active) return fail(IQGPU_EINVAL, "no pending call");
    if (skip_chunks > c->pend.n_chunks) return fail(IQGPU_EINVAL, "skip_chunks exceeds the chunk count");
    const size_t live = c->pend.n_chunks - skip_chunks;
    *n_chunks = live;
    if (!dev_peaks) return IQGPU_OK;
    if (capacity < live) return fail(IQGPU_ECAPACITY, "peak buffer too small");
    CK(cudaSetDevice(c->device));
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : c->stream;
    if (st != c->last_stream) CK(cudaStreamSynchronize(c->last_stream));
    if (!live) return IQGPU_OK;
    if (c->pend.peaks_done)
        CK(cudaMemcpyAsync(dev_peaks, c->d_seg_peak.data() + skip_chunks, live * sizeof(float), cudaMemcpyDeviceToDevice, st));
    else CK(cudaMemsetAsync(dev_peaks, 0, live * sizeof(float), st));
    return IQGPU_OK;
}

int iqgpu_chain_agc_advance_device(iqgpu_chain* c, const float* dev_peaks, uint64_t first_frame, uint64_t n_frames, void* cuda_stream)
{
    if (!c) return fail(IQGPU_EINVAL, "null argument");
    if (c->plan_only) return fail(IQGPU_ENODEVICE, "plan-only chain");
    if (c->agc_mode != 1) return fail(IQGPU_EINVAL, "the chain has no digital AGC");
    if (n_frames == 0) return IQGPU_OK;
    if (!dev_peaks) return fail(IQGPU_EINVAL, "null buffer");
    if (first_frame % c->chunk_frames) return fail(IQGPU_EINVAL, "first_frame must be chunk aligned");
    CK(cudaSetDevice(c->device));
    int rc = c->ensure_buffers();
    if (rc) return rc;
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : c->stream;
    if (c->last_stream && st != c->last_stream) CK(cudaStreamSynchronize(c->last_stream));
    // the chunks' output frame counts are closed form (pipeline.c:523 and the FFT filter's blocks, chain_outputs_after)
    const size_t nch = (size_t)((n_frames + c->chunk_frames - 1) / c->chunk_frames);
    const uint32_t* d_seg = nullptr;
    for (const auto& t : c->prefix_tabs)
        if (t.first == first_frame && t.frames == n_frames) { d_seg = t.d_seg.data(); break; }
    if (!d_seg) {
        if (c->prefix_tabs.size() >= 16) {                          // rare: a new plan; drop the oldest table once it is idle
            CK(cudaStreamSynchronize(st));
            c->prefix_tabs.erase(c->prefix_tabs.begin());
        }
        iqgpu_chain::PrefixTab t;
        t.first = first_frame; t.frames = n_frames;
        CK(t.d_seg.alloc(nch + 1));
        rc = c->stage_chunk_table(t.d_seg.data(), nch, st, [&](uint32_t* seg) {
            uint64_t before = chain_outputs_after(c, first_frame);
            seg[0] = 0;
            for (size_t k = 0; k < nch; k++) {
                const uint64_t end = std::min<uint64_t>(first_frame + n_frames, first_frame + (uint64_t)(k + 1) * c->chunk_frames);
                const uint64_t after = chain_outputs_after(c, end);
                seg[k + 1] = seg[k] + (uint32_t)(after - before);   // the scan uses differences only: wrap-around is harmless
                before = after;
            }
        });
        if (rc) return rc;
        d_seg = t.d_seg.data();
        c->prefix_tabs.push_back(std::move(t));
    }
    PostParams qp{};
    qp.agc_mode = c->agc_mode; qp.agc_target = c->agc_target; qp.agc_alpha = c->agc_alpha; qp.target_rate = c->target_rate;
    CK(c->ensure_agc_quiet(nch, st));
    CK(launch_agc_digital_scan(d_seg, nch, dev_peaks, qp, c->d_agc.data(), nullptr, st, c->d_agc_quiet.data()));
    return IQGPU_OK;
}

int iqgpu_chain_process_device_finish(iqgpu_chain* c, size_t skip_chunks, void* dev_out, size_t out_capacity_bytes,
                                      size_t* out_frames, uint32_t* per_chunk_out, void* cuda_stream)
{
    if (!c || !out_frames) return fail(IQGPU_EINVAL, "null argument");
    if (!c->pend.active) return fail(IQGPU_EINVAL, "no pending call");
    if (!dev_out) return fail(IQGPU_EINVAL, "null buffer");
    if (c->pend.n * c->out_bps > out_capacity_bytes) return fail(IQGPU_ECAPACITY, "output buffer too small");
    CK(cudaSetDevice(c->device));
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : c->stream;
    if (st != c->last_stream) CK(cudaStreamSynchronize(c->last_stream));
    if (per_chunk_out) std::copy(c->pend.counts.begin(), c->pend.counts.end(), per_chunk_out);
    return c->run_back(dev_out, skip_chunks, out_frames, st);
}

int iqgpu_chain_get_agc_state(iqgpu_chain* c, iqgpu_agc_state* s)
{
    if (!c || !s) return fail(IQGPU_EINVAL, "null argument");
    if (c->plan_only) return fail(IQGPU_ENODEVICE, "plan-only chain");
    CK(cudaSetDevice(c->device));
    int rc = c->ensure_buffers();
    if (rc) return rc;
    if (c->last_stream) CK(cudaStreamSynchronize(c->last_stream));
    CK(cudaStreamSynchronize(c->stream));
    AgcState a{};
    CK(cudaMemcpy(&a, c->d_agc.data(), sizeof(a), cudaMemcpyDeviceToHost));
    s->locked = (uint32_t)a.locked; s->gain = a.gain; s->peak_memory = a.peak_mem; s->samples_seen = a.seen;
    s->last_strong_s = a.last_strong;
    return IQGPU_OK;
}

int iqgpu_chain_set_agc_state(iqgpu_chain* c, const iqgpu_agc_state* s)
{
    if (!c || !s) return fail(IQGPU_EINVAL, "null argument");
    if (c->plan_only) return fail(IQGPU_ENODEVICE, "plan-only chain");
    CK(cudaSetDevice(c->device));
    int rc = c->ensure_buffers();
    if (rc) return rc;
    cudaStream_t st = c->last_stream ? c->last_stream : c->stream;
    AgcState a{};
    CK(cudaMemcpyAsync(&a, c->d_agc.data(), sizeof(a), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    a.locked = (int)s->locked; a.gain = s->gain; a.peak_mem = s->peak_memory; a.seen = s->samples_seen;
    a.last_strong = s->last_strong_s;
    CK(cudaMemcpyAsync(c->d_agc.data(), &a, sizeof(a), cudaMemcpyHostToDevice, st));
    CK(cudaStreamSynchronize(st));
    return IQGPU_OK;
}

// ---- sharded RMS AGC: the end state {g, y2'} of a shard and the resume of its successor from it ----
int iqgpu_chain_agc_rms_state_device(iqgpu_chain* c, float* dev_state, void* cuda_stream)
{
    if (!c || !dev_state) return fail(IQGPU_EINVAL, "null argument");
    if (c->plan_only) return fail(IQGPU_ENODEVICE, "plan-only chain");
    if (c->agc_mode != 2) return fail(IQGPU_EINVAL, "the chain has no RMS AGC");
    CK(cudaSetDevice(c->device));
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : c->stream;
    if (c->last_stream && st != c->last_stream) CK(cudaStreamSynchronize(c->last_stream));
    static_assert(offsetof(AgcState, rms_y2) == offsetof(AgcState, rms_g) + sizeof(float), "{g, y2'} must be adjacent");
    CK(cudaMemcpyAsync(dev_state, &c->d_agc.data()->rms_g, 2 * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return IQGPU_OK;
}

int iqgpu_chain_agc_rms_resume_device(iqgpu_chain* c, size_t first_output, const float* dev_state, void* dev_out,
                                      size_t out_capacity_bytes, int* dev_changed, void* cuda_stream)
{
    if (!c) return fail(IQGPU_EINVAL, "null chain");
    if (c->plan_only) return fail(IQGPU_ENODEVICE, "plan-only chain");
    if (c->agc_mode != 2) return fail(IQGPU_EINVAL, "the chain has no RMS AGC");
    if (!dev_state || !dev_out) return fail(IQGPU_EINVAL, "null buffer");
    if (!c->rms_ready)
        return fail(IQGPU_EINVAL, "nothing to resume: the last call must be a process_device call that fit one sub-train "
                                  "(raise the subtrain_frames option)");
    if (c->rms_n * c->out_bps > out_capacity_bytes) return fail(IQGPU_ECAPACITY, "output buffer too small");
    CK(cudaSetDevice(c->device));
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : c->stream;
    if (c->last_stream && st != c->last_stream) CK(cudaStreamSynchronize(c->last_stream));
    c->last_stream = st;
    if (first_output == c->rms_n) {            // at the end of the call: no output changes, the end state is the given one
        agc_rms_set_end_kernel<<<1, 1, 0, st>>>(c->d_agc.data(), reinterpret_cast<const float2*>(dev_state), dev_changed);
        CK(cudaGetLastError());
        c->rms_fresh = true;                    // the trajectory in memory no longer ends in the end state
        c->launches += 1;
        return IQGPU_OK;
    }
    if (first_output > c->rms_n) {             // beyond the call: nothing to do
        if (dev_changed) CK(cudaMemsetAsync(dev_changed, 0, sizeof(int), st));
        return IQGPU_OK;
    }
    if (!c->d_rms_resume.data()) CK(c->d_rms_resume.alloc(1));
    // A resume compares its trajectory with the checkpoints of the one in memory and stops where the two meet.  Behind an
    // earlier resume's frame that trajectory is the earlier resume's, while the rows in front of the frame still hold the
    // call's own: a resume in front of it would meet the call's trajectory and stop, and leave the earlier resume's
    // outputs behind.  So it first re-runs the call from the state the call started from (outputs, checkpoints and block
    // end states as the call left them; *d_agc keeps the end state the resume compares with for `dev_changed`), and then
    // converts the whole call again.  Resumes at the same or a later frame, the time-shard hand-over, need none of this.
    const bool rerun = first_output < c->rms_resume_max;
    if (rerun) {
        AgcState* s = c->d_rms_rerun.data() + 1;         // [0] keeps the start state for the next re-run
        CK(cudaMemcpyAsync(&s->rms_g, &c->d_rms_rerun.data()->rms_g, 2 * sizeof(float), cudaMemcpyDeviceToDevice, st));
        CK(launch_agc_rms(c->rms_src, c->rms_n, c->rms_qp, s, c->d_agc_scratch.data(), c->d_agc_ws.data(), st));
    }
    CK(launch_agc_rms_resume(c->rms_src, c->rms_n, c->rms_qp, c->d_agc.data(), c->d_agc_scratch.data(), c->d_agc_ws.data(), first_output,
                             reinterpret_cast<const float2*>(dev_state), c->d_rms_resume.data(), c->rms_fresh || rerun, dev_changed,
                             st));
    c->rms_fresh = false;
    c->rms_resume_max = rerun ? first_output : std::max(c->rms_resume_max, first_output);
    if (rerun) CK(launch_post(c->d_agc_scratch.data(), c->rms_n, c->rms_qp, nullptr, 0, nullptr, 1, nullptr, dev_out, st));
    else CK(launch_convert_range(c->d_agc_scratch.data(), c->d_rms_resume.data(), c->cfg.output_format, dev_out, st));
    c->launches += rerun ? 3 : 2;
    return IQGPU_OK;
}

int iqgpu_chain_get_agc_rms_state(iqgpu_chain* c, float* g, float* y2)
{
    if (!c || !g || !y2) return fail(IQGPU_EINVAL, "null argument");
    if (c->plan_only) return fail(IQGPU_ENODEVICE, "plan-only chain");
    CK(cudaSetDevice(c->device));
    if (c->last_stream) CK(cudaStreamSynchronize(c->last_stream));
    CK(cudaStreamSynchronize(c->stream));
    AgcState a{};
    CK(cudaMemcpy(&a, c->d_agc.data(), sizeof(a), cudaMemcpyDeviceToHost));
    *g = a.rms_g; *y2 = a.rms_y2;
    return IQGPU_OK;
}

void iqgpu_agc_digital_initial_state(iqgpu_agc_state* s)
{
    if (!s) return;
    s->locked = 0; s->gain = 1.0f; s->peak_memory = 0.05f; s->samples_seen = 0; s->last_strong_s = 0.0;   // agc.c:78
}

// Host restatement of the per-chunk state machine the device runs (kernels.cu AgcStep::run ==
// reference agc.c:105-222 with the sample clock in place of the wall clock).  No device needed.
int iqgpu_agc_digital_advance(iqgpu_agc_state* s, float target, double target_rate_hz, const float* peaks,
                              const uint32_t* counts, size_t n_chunks, float* gains)
{
    if (!s || (n_chunks && (!peaks || !counts))) return fail(IQGPU_EINVAL, "null argument");
    if (!(target_rate_hz > 0.0)) return fail(IQGPU_EINVAL, "target rate must be positive");
    for (size_t c = 0; c < n_chunks; c++) {
        if (counts[c] == 0) { if (gains) gains[c] = 1.0f; continue; }   // agc_apply returns on num_samples == 0
        const float pk = peaks[c];
        float g;
        if (!s->locked) {
            if (pk > s->peak_memory) s->peak_memory = pk;
            const float safe = (s->peak_memory < 1e-4f) ? 1e-4f : s->peak_memory;
            g = target / safe;
            const double elapsed = (double)s->samples_seen / target_rate_hz;
            if (elapsed > (double)2.0f) { s->locked = 1; s->gain = g; s->last_strong_s = elapsed; }
        } else {
            g = s->gain;
            const float opk = pk * g;
            const double now = (double)s->samples_seen / target_rate_hz;
            const float thr = target * 0.75f;
            if (opk > 1.0f) { g = 0.99f / pk; s->last_strong_s = now; }
            else if (opk > thr) s->last_strong_s = now;
            else if (now - s->last_strong_s > (double)4.0f) g = g * 1.0005f;
            s->gain = g;
        }
        s->samples_seen += counts[c];
        if (gains) gains[c] = g;
    }
    return IQGPU_OK;
}

int iqgpu_chain_process(iqgpu_chain* c, const void* raw_in, size_t n_frames, const uint32_t* chunk_frames, size_t n_chunks,
                        void* out, size_t out_capacity_bytes, size_t* out_frames, uint32_t* per_chunk_out)
{
    if (!c || !out_frames) return fail(IQGPU_EINVAL, "null argument");
    return iqgpu_chain_process_multi(&c, 1, raw_in, n_frames, chunk_frames, n_chunks, &out, &out_capacity_bytes, out_frames,
                                     &per_chunk_out);
}

int iqgpu_chain_process_multi(iqgpu_chain* const* chains, size_t K, const void* raw_in, size_t n_frames,
                              const uint32_t* chunk_frames, size_t n_chunks, void* const* out, const size_t* out_capacity_bytes,
                              size_t* out_frames, uint32_t* const* per_chunk_out)
{
    if (!chains || !out || !out_capacity_bytes || !out_frames) return fail(IQGPU_EINVAL, "null argument");
    if (K == 0) return fail(IQGPU_EINVAL, "n_chains must be at least 1");
    // every check that needs no device runs first, so that it fails the same way without one
    auto chan = [K](size_t k) { return K == 1 ? std::string() : "channel " + std::to_string(k) + ": "; };
    auto bad = [&](size_t k, const std::string& m) { return fail(IQGPU_EINVAL, chan(k) + m); };
    iqgpu_chain* const c0 = chains[0];
    for (size_t k = 0; k < K; k++) {
        iqgpu_chain* c = chains[k];
        if (!c) return bad(k, "null chain handle");
        for (size_t j = 0; j < k; j++)
            if (chains[j] == c) return bad(k, "chain handle already listed as channel " + std::to_string(j));
        if (c->device != c0->device) return bad(k, "device differs from channel 0's");
        if (c->cfg.input_format != c0->cfg.input_format) return bad(k, "input_format differs from channel 0's");
        if (c->cfg.input_rate_hz != c0->cfg.input_rate_hz) return bad(k, "input_rate_hz differs from channel 0's");
        if (!chunk_frames && c->chunk_frames != c0->chunk_frames) return bad(k, "chunk_frames option differs from channel 0's");
        if (c->pend.active) return bad(k, "a begun process_device call is still pending (call process_device_finish)");
    }
    for (size_t k = 0; k < K; k++)
        if (chains[k]->plan_only) return fail(IQGPU_ENODEVICE, "chain was created without a device (plan only)");
    for (size_t k = 0; k < K; k++) out_frames[k] = 0;
    if (n_frames == 0) return IQGPU_OK;
    if (!raw_in) return fail(IQGPU_EINVAL, "null buffer");
    for (size_t k = 0; k < K; k++)
        if (!out[k]) return bad(k, "null buffer");
    CK(cudaSetDevice(c0->device));
    int rc;
    size_t sub = SIZE_MAX;          // the sub-train partition every chain can take
    for (size_t k = 0; k < K; k++) {
        rc = chains[k]->ensure_buffers();
        if (rc) return rc;
        sub = std::min(sub, chains[k]->subtrain_frames);
    }
    std::vector<uint32_t> chunks;
    rc = build_chunks(c0, n_frames, chunk_frames, n_chunks, chunks);
    if (rc) return rc;
    for (auto f : chunks)
        if (f > sub) return fail(IQGPU_EINVAL, "a chunk exceeds subtrain_frames");
    for (size_t k = 0; k < K; k++) {
        iqgpu_chain* c = chains[k];
        if (c->count_outputs(chunks.data(), chunks.size(), nullptr) * c->out_bps > out_capacity_bytes[k])
            return fail(IQGPU_ECAPACITY, chan(k) + "output buffer too small");
    }
    // staging slots sized for one sub-train: the raw input in channel 0's, each channel's output in its own
    // (the previous call ended with a synchronisation: nothing still uses the slots)
    const size_t raw_need = (sub + 16) * c0->in_bps;
    for (auto& r : c0->d_raw) CK(r.grow(raw_need, raw_need, no_drain));
    for (size_t k = 0; k < K; k++) {
        iqgpu_chain* c = chains[k];
        const size_t out_need = c->max_out_for(sub) * c->out_bps;
        for (auto& o : c->d_out) CK(o.grow(out_need, out_need, no_drain));
        rc = c->order_after_reset(c->stream);
        if (rc) return rc;
        c->last_stream = c->stream;
        for (auto& t : c->tap) t.len = 0;
    }
    std::vector<size_t> out_off(K, 0), total(K, 0);
    std::vector<uint32_t> launches(K, 0);
    size_t ci = 0, in_off = 0;
    int slot = 0;
    bool used[2] = {false, false};
    while (ci < chunks.size()) {
        size_t cj = ci, n = 0;
        while (cj < chunks.size() && n + chunks[cj] <= sub) { n += chunks[cj]; cj++; }
        // H2D of this sub-train: the raw slot is rewritten only after every channel's D2H out of this slot index finished,
        // which follows that channel's compute on the slot's previous contents
        if (used[slot])
            for (size_t k = 0; k < K; k++) CK(cudaStreamWaitEvent(c0->h2d, chains[k]->ev_d2h[slot], 0));
        CK(cudaMemcpyAsync(c0->d_raw[slot].data(), (const char*)raw_in + in_off * c0->in_bps, n * c0->in_bps, cudaMemcpyHostToDevice, c0->h2d));
        CK(cudaEventRecord(c0->ev_h2d[slot], c0->h2d));
        for (size_t k = 0; k < K; k++) {
            iqgpu_chain* c = chains[k];
            CK(cudaStreamWaitEvent(c->stream, c0->ev_h2d[slot], 0));
            size_t produced = 0;
            c->dc_slot = 0; c->dc_prepared = false;      // host path is PCIe bound: DC pre-pass inline on the compute stream
            uint32_t* pc = per_chunk_out ? per_chunk_out[k] : nullptr;
            rc = c->run_subtrain(c0->d_raw[slot].data(), n, chunks.data() + ci, cj - ci, c->d_out[slot].data(), &produced,
                                 pc ? pc + ci : nullptr, c->stream);
            if (rc) return rc;
            launches[k] += c->launches;
            CK(cudaEventRecord(c->ev_done[slot], c->stream));
            CK(cudaStreamWaitEvent(c->d2h, c->ev_done[slot], 0));
            if (produced)
                CK(cudaMemcpyAsync((char*)out[k] + out_off[k], c->d_out[slot].data(), produced * c->out_bps, cudaMemcpyDeviceToHost, c->d2h));
            CK(cudaEventRecord(c->ev_d2h[slot], c->d2h));
            out_off[k] += produced * c->out_bps; total[k] += produced;
        }
        used[slot] = true;
        in_off += n;
        ci = cj; slot ^= 1;
    }
    for (size_t k = 0; k < K; k++) {
        iqgpu_chain* c = chains[k];
        CK(cudaStreamSynchronize(c->d2h));
        CK(cudaStreamSynchronize(c->stream));
        c->launches = launches[k];
        c->rms_ready = false;                        // the output went through the staging slots, not a caller's buffer
        out_frames[k] = total[k];
    }
    return IQGPU_OK;
}

int iqgpu_chain_read_tap(iqgpu_chain* c, int tapi, float* host_cf32, size_t capacity_frames, size_t* frames)
{
    if (!c || !frames || tapi < 0 || tapi > 2) return fail(IQGPU_EINVAL, "bad argument");
    if (c->plan_only) return fail(IQGPU_ENODEVICE, "plan-only chain");
    CK(cudaSetDevice(c->device));
    CK(cudaStreamSynchronize(c->stream));
    const size_t n = c->tap[tapi].len;
    *frames = n;
    if (host_cf32) {
        if (n > capacity_frames) return fail(IQGPU_ECAPACITY, "tap buffer too small");
        if (n) CK(cudaMemcpy(host_cf32, c->tap[tapi].buf.data(), n * sizeof(float2), cudaMemcpyDeviceToHost));
    }
    return IQGPU_OK;
}

int iqgpu_chain_get_filter_taps(iqgpu_chain* c, float* taps, uint32_t capacity, uint32_t* num)
{
    if (!c || !num) return fail(IQGPU_EINVAL, "null argument");
    *num = (uint32_t)c->filt.taps.size();
    for (uint32_t i = 0; taps && i < *num && i < capacity; i++) { taps[2 * i] = c->filt.taps[i].real(); taps[2 * i + 1] = c->filt.taps[i].imag(); }
    return IQGPU_OK;
}
int iqgpu_chain_get_halfband_taps(iqgpu_chain* c, uint32_t i, float* taps, uint32_t capacity, uint32_t* num)
{
    if (!c || !num) return fail(IQGPU_EINVAL, "null argument");
    if (i >= c->rs.num_halfband) return fail(IQGPU_EINVAL, "stage index out of range");
    *num = (uint32_t)c->rs.stages[i].h.size();
    for (uint32_t k = 0; taps && k < *num && k < capacity; k++) taps[k] = c->rs.stages[i].h[k];
    return IQGPU_OK;
}
int iqgpu_chain_get_arb_taps(iqgpu_chain* c, float* taps, uint32_t capacity, uint32_t* num)
{
    if (!c || !num) return fail(IQGPU_EINVAL, "null argument");
    *num = (uint32_t)c->rs.arb_h.size();
    for (uint32_t k = 0; taps && k < *num && k < capacity; k++) taps[k] = c->rs.arb_h[k];
    return IQGPU_OK;
}

int iqgpu_chain_halo_frames(iqgpu_chain* c, size_t* halo)
{
    if (!c || !halo) return fail(IQGPU_EINVAL, "null argument");
    size_t h = (size_t)c->rs.halo_input_frames;
    // a post-resample FIR needs (ntaps-1) output-rate samples = (ntaps-1)/ratio input frames
    if (filter_is_fir(c->filt) && c->filt.post_resample)
        h += (size_t)std::ceil((double)c->filt.taps.size() / (double)c->ratio) + ((size_t)1 << c->rs.num_halfband);
    else if (filter_is_fir(c->filt)) h += c->filt.taps.size();
    // post-resample FFT filter: output block b reads the resampled samples [(b-1)n, (b+1)n), so the block before the first one
    // a shard owns must lie behind the resampler's exact region: 2n output-rate samples = 2n/ratio input frames
    if (filter_is_fft(c->filt) && c->filt.post_resample)
        h += (size_t)std::ceil(2.0 * (double)c->filt.block / (double)c->ratio) + ((size_t)1 << c->rs.num_halfband);
    // DC blocker: infinite memory; 16 time constants leave e^-16 ~ 1e-7 of the integrator state
    if (c->dc.enable) h += (size_t)std::ceil(16.0 / (double)c->dc.alpha);
    *halo = h;
    return IQGPU_OK;
}

int iqgpu_chain_outputs_after(iqgpu_chain* c, uint64_t frames_in, uint64_t* frames_out)
{
    if (!c || !frames_out) return fail(IQGPU_EINVAL, "null argument");
    *frames_out = chain_outputs_after(c, frames_in);
    return IQGPU_OK;
}

int iqgpu_chain_seek(iqgpu_chain* c, uint64_t first_frame, uint64_t* out_first_frame)
{
    if (!c) return fail(IQGPU_EINVAL, "null chain");
    if (filter_is_fft(c->filt) && !c->filt.post_resample)
        return fail(IQGPU_EINVAL, "seek is not supported with a pre-resample FFT filter: its blocks are cut from the input "
                                  "stream behind the remainder that filter_reset carries into the next stream (F5), a "
                                  "position a shard cannot reproduce; only interpolating or no_resample chains filter there");
    int rc = c->plan_only ? IQGPU_OK : c->ensure_buffers();
    if (rc) return rc;
    rc = c->reset_state();
    if (rc) return rc;
    c->n_in = first_frame;
    const uint64_t r = resampler_outputs_after(c->rs, first_frame);
    uint64_t o = r;
    if (filter_is_fft(c->filt)) {
        // the single stream cuts the filter's blocks at multiples of n from its start: R(first_frame) mod n resampled frames
        // wait for a full block here.  They are halo (dropped by the caller), so they may read as the zeros reset_state
        // left in the stream's history; the blocks that follow are those of the single stream.
        c->fft_rem = (uint32_t)(r % c->filt.block);
        o = r - c->fft_rem;
    }
    c->n_out = o;
    c->n_nco_post = o;
    if (out_first_frame) *out_first_frame = o;
    return IQGPU_OK;
}

// ---- sample_convert.h on host buffers -----------------------------------------------------------
static int convert_common(const void* in, void* out, size_t n, int in_fmt, int out_fmt, float gain)
{
    if (!in || !out) return fail(IQGPU_EINVAL, "null buffer");
    if (n == 0) return IQGPU_OK;
    iqgpu_chain_config g{};
    g.input_format = in_fmt; g.output_format = out_fmt;
    g.input_rate_hz = 1e6; g.target_rate_hz = 1e6; g.gain = gain; g.no_resample = 1;
    iqgpu_chain* c = nullptr;
    int rc = iqgpu_chain_create(&g, 0, &c);
    if (rc) return rc;
    c->subtrain_frames = std::min<size_t>(std::max<size_t>(n, 1024), (size_t)1 << 22);
    const uint32_t one = (uint32_t)std::min<size_t>(n, c->subtrain_frames);
    std::vector<uint32_t> chunks;
    for (size_t left = n; left;) { uint32_t f = (uint32_t)std::min<size_t>(left, one); chunks.push_back(f); left -= f; }
    size_t produced = 0;
    rc = iqgpu_chain_process(c, in, n, chunks.data(), chunks.size(), out, n * bytes_per_sample(out_fmt), &produced, nullptr);
    std::string m = g_err;
    delete c;
    if (rc) return fail(rc, m);
    return produced == n ? IQGPU_OK : fail(IQGPU_EINVAL, "internal: conversion produced a wrong frame count");
}
int iqgpu_convert_block_to_cf32(const void* in, float* out_cf32, size_t n, int format, float gain)
{
    if (!is_complex_format(format)) return fail(IQGPU_EINVAL, "Unhandled input format");
    return convert_common(in, out_cf32, n, format, IQGPU_FMT_CF32, gain);
}
int iqgpu_convert_cf32_to_block(const float* in_cf32, void* out, size_t n, int format)
{
    if (!is_complex_format(format)) return fail(IQGPU_EINVAL, "Unhandled output format");
    return convert_common(in_cf32, out, n, IQGPU_FMT_CF32, format, 1.0f);
}

float iqgpu_iq_direction(uint32_t seed, uint64_t attempt, uint32_t k) { return iq_direction_host(seed, attempt, k); }

int iqgpu_iq_optimize(const float* block1024_cf32, const float* directions50, float* mag, float* phase,
                      float* avg_power, float* power_range)
{
    if (!block1024_cf32 || !directions50 || !mag || !phase) return fail(IQGPU_EINVAL, "null argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return fail(IQGPU_ENODEVICE, "no CUDA device available"); }
    CK(iq_optimize_device(block1024_cf32, directions50, mag, phase, avg_power, power_range, nullptr));
    return IQGPU_OK;
}

}  // extern "C"
