/*
 * iqgpu.h — C ABI of libiqgpu.so: the B200 (sm_100a) implementation of iq_tool's per-block
 * sample-processing chain.  Plain pointers and sizes only; no CUDA or torch types.
 *
 * The reference (pclov3r/iq_tool) has no FFI for this path: its boundary is the C function
 * set declared in its stage/module headers, linked statically (SURVEY.md §8(b)).  Each group
 * of entry points below names the reference interface it replaces (file:line under
 * /root/reference).  the files under iq_tool_b200/host/ provide drop-in translation units with the
 * reference's exact prototypes that forward to these entry points; INTEGRATION.md shows how a
 * maintainer links them.
 *
 * Conventions
 *   - Every function returns IQGPU_OK (0) or a negative IQGPU_E* code; the message for the last
 *     error on the calling thread is available from iqgpu_last_error().  There is NO CPU
 *     fallback: without a usable CUDA device every compute entry point fails with
 *     IQGPU_ENODEVICE.
 *   - "frames" are complex I/Q pairs.  cf32 buffers are interleaved {re, im} floats.
 *   - Host-pointer entry points copy H2D/D2H internally (pinned staging); *_device entry points
 *     take device pointers valid on the chain's device and an optional CUDA stream handle
 *     (cudaStream_t cast to void*, NULL = the chain's own stream).
 *   - A chain processes a "train" of reference chunks per call.  Per-chunk semantics of the
 *     reference (digital-AGC gain per chunk, FFT-filter output quantisation per chunk,
 *     per-chunk frames_to_write) are preserved exactly; see DESIGN.md §Chunk trains.
 */
#ifndef IQGPU_H
#define IQGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IQGPU_ABI_VERSION 1

enum {
    IQGPU_OK = 0,
    IQGPU_EINVAL = -1,     /* bad argument / unsupported configuration (reference would log_fatal) */
    IQGPU_ENODEVICE = -2,  /* no CUDA device / driver */
    IQGPU_ECUDA = -3,      /* CUDA runtime error */
    IQGPU_ENOMEM = -4,
    IQGPU_ECAPACITY = -5   /* output buffer too small */
};

/* sample formats: numeric values of the reference's format_t (include/common_types.h:33-37) */
enum {
    IQGPU_FMT_UNKNOWN = 0, IQGPU_FMT_U8, IQGPU_FMT_S8, IQGPU_FMT_U16, IQGPU_FMT_S16, IQGPU_FMT_U32,
    IQGPU_FMT_S32, IQGPU_FMT_F32, IQGPU_FMT_CU8, IQGPU_FMT_CS8, IQGPU_FMT_CU16, IQGPU_FMT_CS16,
    IQGPU_FMT_CS24, IQGPU_FMT_CU32, IQGPU_FMT_CS32, IQGPU_FMT_CF32, IQGPU_FMT_SC16Q11
};
/* FilterType (common_types.h:45-51), FilterTypeRequest (:61-65), FilterImplementationType (:53-59),
 * AgcProfile (:77-82) */
enum { IQGPU_FILTER_NONE = 0, IQGPU_FILTER_LOWPASS, IQGPU_FILTER_HIGHPASS, IQGPU_FILTER_PASSBAND, IQGPU_FILTER_STOPBAND };
enum { IQGPU_FILTER_REQ_AUTO = 0, IQGPU_FILTER_REQ_FIR, IQGPU_FILTER_REQ_FFT };
enum { IQGPU_FILTER_IMPL_NONE = 0, IQGPU_FILTER_IMPL_FIR_SYM, IQGPU_FILTER_IMPL_FIR_ASYM, IQGPU_FILTER_IMPL_FFT_SYM, IQGPU_FILTER_IMPL_FFT_ASYM };
enum { IQGPU_AGC_OFF = 0, IQGPU_AGC_DX, IQGPU_AGC_LOCAL, IQGPU_AGC_DIGITAL };

enum { IQGPU_STAGE_DC = 1, IQGPU_STAGE_IQ = 2, IQGPU_STAGE_NCO = 4, IQGPU_STAGE_FILTER = 8,
       IQGPU_STAGE_RESAMPLER = 16, IQGPU_STAGE_AGC = 32 };

#define IQGPU_MAX_FILTER_CHAIN 5      /* MAX_FILTER_CHAIN, include/constants.h:249 */
#define IQGPU_CHUNK_SAMPLES    16384  /* PIPELINE_CHUNK_BASE_SAMPLES, include/constants.h:123 */

typedef struct {
    int32_t type;      /* IQGPU_FILTER_* */
    float   freq1_hz;  /* cutoff, or centre for pass/stop band (src/config.c:192-216) */
    float   freq2_hz;  /* bandwidth for pass/stop band */
} iqgpu_filter_request;

/* The fields of AppConfig / AppResources (include/app_context.h:66-138, 205-283) that the
 * chain reads, resolved the way src/config.c and src/setup.c resolve them. */
typedef struct {
    int32_t input_format;           /* AppResources.input_format */
    int32_t output_format;          /* AppConfig.output_format */
    double  input_rate_hz;          /* source_info.samplerate (integer Hz) */
    double  target_rate_hz;         /* AppConfig.target_rate */
    float   gain;                   /* AppConfig.gain */
    int32_t dc_block_enable;        /* AppConfig.dc_block.enable */
    int32_t iq_correction_enable;   /* AppConfig.iq_correction.enable */
    float   iq_mag;                 /* initial IqCorrectionFactors.mag */
    float   iq_phase;               /* initial IqCorrectionFactors.phase */
    int32_t shift_after_resample;   /* AppConfig.shift_after_resample */
    double  freq_shift_hz;          /* AppResources.nco_shift_hz */
    int32_t no_resample;            /* AppConfig.no_resample (native-rate processing) */
    int32_t num_filter_requests;
    iqgpu_filter_request filter_requests[IQGPU_MAX_FILTER_CHAIN];
    float   transition_width_hz;    /* --transition-width, 0 = auto */
    int32_t filter_taps;            /* --filter-taps, 0 = auto */
    float   attenuation_db;         /* --attenuation, 0 = 60 dB */
    int32_t filter_type_request;    /* IQGPU_FILTER_REQ_* (AUTO == option not given) */
    int32_t filter_fft_size;        /* --filter-fft-size, 0 = auto */
    int32_t agc_enable;             /* AppConfig.output_agc.enable */
    int32_t agc_profile;            /* IQGPU_AGC_* */
    float   agc_target_level_arg;   /* --agc-target, 0 = profile default */
    int32_t stage_select;           /* 0 = the whole chain.  Otherwise a mask of IQGPU_STAGE_*: the chain
                                     * is DESIGNED from the full configuration above (identical taps, NCO
                                     * increment, ratio, AGC timing) but executes only the selected
                                     * stage(s) on cf32 input -> cf32 output: the module-level entry
                                     * points (dc_block_apply, freq_shift_apply, filter_apply,
                                     * resampler_execute, agc_apply, iq_correct_apply). */
} iqgpu_chain_config;

typedef struct {
    float    ratio;                 /* float r = (float)(target/input), src/setup.c:107 */
    int32_t  is_interp;
    uint32_t num_halfband;          /* S */
    uint32_t halfband_m[16];        /* semi-length per design index (index 0 = lowest rate) */
    float    rate_arbitrary;
    uint32_t arb_step;              /* 24-bit fixed-point phase step */
    int32_t  filter_impl;           /* IQGPU_FILTER_IMPL_* */
    int32_t  filter_post_resample;  /* AppConfig.apply_user_filter_post_resample */
    uint32_t filter_block_size;     /* AppResources.user_filter_block_size */
    uint32_t filter_num_taps;
    uint32_t nco_dtheta;            /* 32-bit NCO phase increment, 0 if no shift */
    int32_t  nco_is_post;
    uint32_t agc_locked;            /* AppResources.agc_is_locked */
    float    agc_gain;              /* AppResources.agc_current_gain */
    float    agc_peak_memory;       /* AppResources.agc_peak_memory */
    uint64_t agc_samples_seen;      /* AppResources.agc_samples_seen */
    uint64_t frames_in_total;       /* input frames consumed since create/reset */
    uint64_t frames_out_total;      /* output frames produced since create/reset */
    uint32_t fused_front;           /* 1 when the fused convert+mix+resample kernel is in use */
    uint32_t kernel_launches;       /* kernels launched by the last process call */
    uint32_t halo_frames;           /* raw-input halo the fused front re-reads per train */
    uint32_t polyphase_variant;     /* outputs per lane of the fused front's polyphase stage in its last launch (1, 2
                                       or 4; 0 before the fused front has run) */
} iqgpu_chain_info;

typedef struct iqgpu_chain iqgpu_chain;

/* ---- library ---------------------------------------------------------------------- */
int         iqgpu_abi_version(void);
const char *iqgpu_last_error(void);
int         iqgpu_device_count(void);
/* pinned host memory for chunk pools (replaces the malloc slab of src/pipeline.c:277) */
void       *iqgpu_host_alloc(size_t bytes);
void        iqgpu_host_free(void *p);

/* ---- whole chain: pre_processor_apply_chain + resampler_execute + post_processor_apply_chain
 *      (include/pre_processor.h:24, include/resampler.h:48, include/post_processor.h:24;
 *       object creation order of src/pipeline.c:138-147) --------------------------------- */
int  iqgpu_chain_create(const iqgpu_chain_config *cfg, int device, iqgpu_chain **out);
void iqgpu_chain_destroy(iqgpu_chain *c);
/* stream discontinuity: pre_processor_reset + resampler_reset + post_processor_reset
 * (include/pre_processor.h:34, include/resampler.h:43, include/post_processor.h:34).  As in the reference, filter_reset
 * (src/filter.c:417-436) clears the FFT filter's overlap state but NOT the count of frames waiting for a full block: with
 * an FFT filter those frames re-enter the new stream in front of its first chunk (SURVEY 8(a) F5). */
int  iqgpu_chain_reset(iqgpu_chain *c);
/* the state right after iqgpu_chain_create (nothing of the old stream survives): rewinding a benchmark or a test */
int  iqgpu_chain_restart(iqgpu_chain *c);
int  iqgpu_chain_get_info(iqgpu_chain *c, iqgpu_chain_info *info);
/* runtime knobs: "fused" (0/1), "subtrain_frames", "chunk_frames", "record_taps" (0/1),
 * "time_kernels" (0/1: bracket every kernel class with CUDA events on the launch stream),
 * "dc_mode" (0 = DC blocker in exact arithmetic, the chunk-train default; 1 = the reference's fp32 direct-form-II state
 * rounding of liquid's iirfilt_crcf (src/dc_block.c:76-85), evaluated serially: what the module-level dc_block_apply
 * drop-in uses on its 16384-frame chunks — set before the first process call) */
int  iqgpu_chain_set_option(iqgpu_chain *c, const char *key, int64_t value);
/* kernel classes for iqgpu_chain_get_kernel_times */
enum {
    IQGPU_KCLASS_PRE = 0,       /* K1 convert [+DC apply] [+I/Q] [+NCO]        */
    IQGPU_KCLASS_DC_SCAN,       /* DC-blocker run sums + carry scan             */
    IQGPU_KCLASS_RESAMPLER,     /* K2 halfband stages + arbitrary stage (unfused) */
    IQGPU_KCLASS_FILTER,        /* K3 FIR / K4 FFT filter                       */
    IQGPU_KCLASS_POST,          /* K5 [NCO] + AGC + convert                     */
    IQGPU_KCLASS_FUSED_FRONT,   /* fused K1+K2                                  */
    IQGPU_KCLASS_COUNT = 8
};
/* accumulated device time (ms) and launch-group counts per kernel class since the last reset
 * of the counters; arrays of IQGPU_KCLASS_COUNT entries (either may be NULL) */
int  iqgpu_chain_get_kernel_times(iqgpu_chain *c, double *ms, uint32_t *launches, int reset);
/* live update of the I/Q correction factors (iq_correct.c:206-216 double-buffer swap) */
int  iqgpu_chain_set_iq_factors(iqgpu_chain *c, float mag, float phase);
/* In-chain I/Q optimiser (option "iq_optimize" = 1; "iq_optimize_interval_ms", default 500 = IQ_CORRECTION_INTERVAL_MS;
 * "iq_optimize_seed"): replaces the side thread of src/utility_threads.c:35-47 and the probe copy of src/pipeline.c:468-476.
 * For every chunk of >= 1024 frames that starts at least the interval after the last probed one — on the SAMPLE clock,
 * input frames / input rate — the chain takes the first 1024 pre-processed frames and runs one pass of
 * iq_correct_run_optimization (src/iq_correct.c:154-235) on the device, with +-1 directions from a counter-based generator
 * (SURVEY App. B7: the reference uses wall time and rand()); the factors a sub-train's passes leave are applied from the next
 * sub-train on.  get_iq_state returns the factors in force and the number of successful passes / probed blocks. */
int  iqgpu_chain_get_iq_state(iqgpu_chain *c, float *mag, float *phase, uint64_t *passes, uint64_t *attempts);
/* the generator behind the in-chain optimiser's directions (host; lets a test or a host-side optimiser reproduce them) */
float iqgpu_iq_direction(uint32_t seed, uint64_t attempt, uint32_t k);

/* Process a train of n_frames input frames held in HOST memory.  The train is cut into
 * reference chunks of IQGPU_CHUNK_SAMPLES frames (last one short) unless chunk_frames/n_chunks
 * give explicit chunk lengths (SDR-style irregular chunks; sum must equal n_frames).
 * out receives the converted output frames; per_chunk_out (optional, one entry per chunk)
 * receives each chunk's frames_to_write (src/pipeline.c:523). */
int  iqgpu_chain_process(iqgpu_chain *c, const void *raw_in, size_t n_frames,
                         const uint32_t *chunk_frames, size_t n_chunks,
                         void *out, size_t out_capacity_bytes, size_t *out_frames,
                         uint32_t *per_chunk_out);
/* Same, with raw_in / out resident in device memory; runs asynchronously on `cuda_stream`
 * except for the final output-frame count, which is closed-form and returned immediately. */
int  iqgpu_chain_process_device(iqgpu_chain *c, const void *dev_raw_in, size_t n_frames,
                                const uint32_t *chunk_frames, size_t n_chunks,
                                void *dev_out, size_t out_capacity_bytes, size_t *out_frames,
                                uint32_t *per_chunk_out, void *cuda_stream);
/* Several channels out of one capture: K chains consume the same host-memory train, which is copied H2D once per
 * sub-train (into chains[0]'s staging) and processed by every chain, each on its own streams, into its own output.
 * out[k] / out_capacity_bytes[k] / out_frames[k] / per_chunk_out[k] (the array or an entry may be NULL) belong to
 * chains[k]; channel k's output, per-chunk counts and state are those of iqgpu_chain_process on chains[k] alone.
 * The train is cut into sub-trains of the smallest subtrain_frames of the chains.  Before any work is queued the call
 * refuses (IQGPU_EINVAL, the message names the channel and the field) zero chains, a NULL or repeated handle, chains
 * on different devices, a different input_format or input_rate_hz, a different chunk_frames option when the chunk
 * lengths are implicit, and a chain with a begun process_device call pending; then plan-only chains
 * (IQGPU_ENODEVICE) and a channel whose output does not fit (IQGPU_ECAPACITY).  iqgpu_chain_process is the K = 1
 * case. */
int  iqgpu_chain_process_multi(iqgpu_chain *const *chains, size_t n_chains, const void *raw_in, size_t n_frames,
                               const uint32_t *chunk_frames, size_t n_chunks, void *const *out,
                               const size_t *out_capacity_bytes, size_t *out_frames, uint32_t *const *per_chunk_out);
/* closed form: resampler output frames after `frames_in` input frames since reset
 * (msresamp_crcf_execute's cumulative *num_written, src/resampler.c:49) */
int  iqgpu_chain_resampler_outputs_after(iqgpu_chain *c, uint64_t frames_in, uint64_t *frames_out);
/* closed-form output frame count for the NEXT n_frames (no data touched) */
int  iqgpu_chain_predict_output(iqgpu_chain *c, size_t n_frames, size_t *out_frames);
/* copy the cf32 stream observed at an internal tap of the LAST process call to host:
 * tap 0 = after the pre-processor chain, 1 = after the resampler, 2 = before output conversion.
 * Taps 0 is only materialised when the chain runs unfused. */
int  iqgpu_chain_read_tap(iqgpu_chain *c, int tap, float *host_cf32, size_t capacity_frames, size_t *frames);
/* design introspection (filter.c master taps; msresamp design) */
int  iqgpu_chain_get_filter_taps(iqgpu_chain *c, float *cf32_taps, uint32_t capacity, uint32_t *num_taps);
int  iqgpu_chain_get_halfband_taps(iqgpu_chain *c, uint32_t design_index, float *taps, uint32_t capacity, uint32_t *num_taps);
int  iqgpu_chain_get_arb_taps(iqgpu_chain *c, float *taps, uint32_t capacity, uint32_t *num_taps);

/* ---- time-sharding (multi-GPU, SURVEY.md 8(e)): position this chain at absolute input
 *      frame `first_frame` of a longer capture with EMPTY filter histories.  NCO phase, halfband
 *      alignment, arbitrary-resampler phase and output index are set in closed form;
 *      `out_first_frame` receives the absolute output-frame index of the first output the chain
 *      will emit.  To reproduce the single-stream result a shard seeks to
 *      (shard_start - halo), processes from there and drops the outputs that precede
 *      shard_start (their count is closed form too); halo from iqgpu_chain_halo_frames.
 *      A post-resample FFT filter (every decimating chain with one) is positioned on the single
 *      stream's blocks: R(first_frame) mod n resampled frames (R = resampler outputs, n = block)
 *      wait as zeros for a full block and `out_first_frame` = floor(R(first_frame) / n) * n.  A
 *      pre-resample FFT filter (interpolating or no_resample chains) is refused.  The RMS AGC
 *      starts from its reset state; iqgpu_chain_agc_rms_resume_device hands the state over.
 *      The halo covers the resampler's history, a FIR's taps, two FFT blocks (2n / ratio frames)
 *      and 16 time constants of the DC blocker (the only approximate term).
 *      Stream positions are limited to IQGPU_MAX_STREAM_POSITION (2^62) input frames, and the
 *      resampled output index to the same bound (an interpolating chain reaches it first): a seek
 *      to first_frame >= 2^62, or one whose output index would pass it, and a process call or an
 *      iqgpu_chain_agc_advance_device range that would carry either past it are refused with
 *      IQGPU_EINVAL before any work is queued. -------------------------------------------------- */
#define IQGPU_MAX_STREAM_POSITION (1ull << 62)
int  iqgpu_chain_seek(iqgpu_chain *c, uint64_t first_frame, uint64_t *out_first_frame);
int  iqgpu_chain_halo_frames(iqgpu_chain *c, size_t *halo_frames);
/* closed form: chain output frames after `frames_in` input frames since a restart — the resampler's
 * count, block-quantised by an FFT filter.  The output index of a capture frame, for shard plans. */
int  iqgpu_chain_outputs_after(iqgpu_chain *c, uint64_t frames_in, uint64_t *frames_out);

/* ---- sharded RMS AGC (liquid agc_crcf, a nonlinear per-sample recurrence in {g, y2'}): each
 *      shard runs its halo and shard from the reset state at its lead with ONE process_device call
 *      (one sub-train: raise the subtrain_frames option), then world-1 rounds follow, in each of
 *      which every rank publishes its end state (8 bytes) and rank g >= 1 resumes from rank g-1's.
 *      After round k ranks 0..k are exact.
 *        agc_rms_state_device   copies the end state {g, y2'} (two floats) to device memory on `stream`;
 *        agc_rms_resume_device  re-runs the AGC of the last call from output frame `first_output` (the
 *                               shard's first owned output) with the state at `dev_state`, rewrites
 *                               and re-converts into `dev_out` (the last call's output buffer) only the
 *                               range that changed, and writes 1 / 0 to `dev_changed` (optional, device
 *                               int) when the end state did / did not change.  Any sequence of resumes
 *                               of one call is allowed: each leaves the outputs in front of `first_output`
 *                               as they are and makes the outputs from it on and the end state those of
 *                               the AGC run from `dev_state` at `first_output`.  A resume at the same
 *                               frame from the same state as the previous one does nothing on the device;
 *                               one in front of an earlier resume's frame first re-runs the whole call
 *                               (and converts all of it again); one at the call's end (`first_output` =
 *                               its output count) only sets the end state; beyond it, nothing happens.
 *                               All of it is queued on `stream` without a host synchronisation;
 *        get_agc_rms_state      reads {g, y2'} to the host (synchronises). ----------------------------- */
int  iqgpu_chain_agc_rms_state_device(iqgpu_chain *c, float *dev_state, void *cuda_stream);
int  iqgpu_chain_agc_rms_resume_device(iqgpu_chain *c, size_t first_output, const float *dev_state, void *dev_out,
                                       size_t out_capacity_bytes, int *dev_changed, void *cuda_stream);
int  iqgpu_chain_get_agc_rms_state(iqgpu_chain *c, float *g, float *y2);

/* ---- sharded digital AGC (SURVEY.md 8(e)): the one exchange step of a time-sharded run.
 *      The digital AGC (src/agc.c:105-222) is a scalar state machine over per-chunk peaks, so a
 *      shard needs the state left by every earlier chunk of the capture.  process_device is
 *      split at that point:
 *        begin   runs everything up to the per-chunk peaks of this call (one sub-train),
 *        pending_chunk_peaks hands the peaks (and per-chunk frame counts) to the host,
 *        -- the ranks all-gather their peaks; each advances the initial state over the chunks
 *           of all earlier shards with iqgpu_agc_digital_advance and installs it with
 *           iqgpu_chain_set_agc_state --
 *        finish  runs the state machine over this call's chunks, scales and converts.
 *      `skip_chunks` leading chunks (the shard's halo) get unit gain and leave the state alone.
 *      Works for every chain (without a digital AGC the peaks read as zero). ------------------ */
typedef struct {
    uint32_t locked;          /* AppResources.agc_is_locked            (include/app_context.h:226-231) */
    float    gain;            /* AppResources.agc_current_gain */
    float    peak_memory;     /* AppResources.agc_peak_memory */
    uint64_t samples_seen;    /* AppResources.agc_samples_seen */
    double   last_strong_s;   /* agc_last_strong_peak_time on the sample clock (seconds) */
} iqgpu_agc_state;
int  iqgpu_chain_process_device_begin(iqgpu_chain *c, const void *dev_raw_in, size_t n_frames,
                                      const uint32_t *chunk_frames, size_t n_chunks, void *cuda_stream);
int  iqgpu_chain_pending_chunk_peaks(iqgpu_chain *c, float *peaks, uint32_t *counts, size_t capacity, size_t *n_chunks);
int  iqgpu_chain_process_device_finish(iqgpu_chain *c, size_t skip_chunks, void *dev_out, size_t out_capacity_bytes,
                                       size_t *out_frames, uint32_t *per_chunk_out, void *cuda_stream);
/* Device-side form of the same exchange (no host round trip: the peaks never leave the GPUs).
 *   iqgpu_chain_pending_chunk_peaks_device  copies the begun call's per-chunk peaks [skip_chunks, n_chunks) into a device
 *                                           buffer (e.g. the send buffer of an NCCL all-gather), asynchronously on `stream`;
 *   iqgpu_chain_agc_advance_device          advances the chain's device-resident digital-AGC state over the reference chunks
 *                                           of input frames [first_frame, first_frame + n_frames) of the capture, whose
 *                                           per-chunk peaks are in device memory (e.g. a lower rank's slice of the gathered
 *                                           buffer); the chunks' frame counts are closed form.  Call it once per lower rank,
 *                                           in rank order, between ..._begin and ..._finish. */
int  iqgpu_chain_pending_chunk_peaks_device(iqgpu_chain *c, size_t skip_chunks, float *dev_peaks, size_t capacity,
                                            size_t *n_chunks, void *cuda_stream);
int  iqgpu_chain_agc_advance_device(iqgpu_chain *c, const float *dev_peaks, uint64_t first_frame, uint64_t n_frames,
                                    void *cuda_stream);
int  iqgpu_chain_get_agc_state(iqgpu_chain *c, iqgpu_agc_state *s);
int  iqgpu_chain_set_agc_state(iqgpu_chain *c, const iqgpu_agc_state *s);
/* host-only (no device): agc_create's initial state (agc.c:66-80) and the per-chunk state machine */
void iqgpu_agc_digital_initial_state(iqgpu_agc_state *s);
int  iqgpu_agc_digital_advance(iqgpu_agc_state *s, float target, double target_rate_hz, const float *peaks,
                               const uint32_t *counts, size_t n_chunks, float *gains /* optional */);

/* ---- raw-file streaming (the callers either side of the path, SURVEY.md 8(f)): replaces the Reader and
 *      Writer threads of a raw-file run (src/input_rawfile.c:188-249: sf_read_raw per 16384-frame chunk;
 *      src/output_raw_file.c:146-184: 1 MB fwrites from a ring buffer) with large reads of whole chunk
 *      trains into pinned memory, the chain, and one write per train, overlapped on three threads.  The
 *      file is cut into reference chunks exactly as the reference does (short last chunk, trailing partial
 *      frame dropped, nothing flushed at end of stream). ------------------------------------------------- */
typedef struct {
    uint64_t frames_in;       /* input frames read and processed */
    uint64_t frames_out;      /* output frames written */
    uint64_t bytes_written;
    uint64_t trains;          /* chain calls made */
} iqgpu_rawfile_stats;
int         iqgpu_rawfile_run(const iqgpu_chain_config *cfg, int device, const char *in_path, const char *out_path,
                              size_t train_chunks /* reference chunks per chain call, 0 = 64 */,
                              iqgpu_rawfile_stats *stats /* optional */);
/* Several channels out of one raw file (see iqgpu_chain_process_multi): the file is read once, chain k is built from
 * cfgs[k] and writes out_paths[k]; stats (optional) receives one record per channel.  Every output is opened before
 * anything is read: if one cannot be, the call fails naming its path and removes the outputs it had opened. */
int         iqgpu_rawfile_run_channels(const iqgpu_chain_config *cfgs, size_t n_channels, int device, const char *in_path,
                                       const char *const *out_paths, size_t train_chunks,
                                       iqgpu_rawfile_stats *stats /* [n_channels] or NULL */);
const char *iqgpu_rawfile_last_error(void);

/* ---- WAV / RF64 containers around the path (SURVEY.md 8(f) rank 4): the WAV input module
 *      (src/input_wav.c: wav_initialize :542-632, auxi metadata :146-188,294-441, file-name metadata :190-271,
 *      --wav-center-target-freq :612-629, reader loop :634-699) and the WAV / RF64 output modules
 *      (src/output_wav_common.c:54-174, src/output_wav.c, src/output_wav_rf64.c).  The reference parses and
 *      writes the container with libsndfile and the XML form of the auxi chunk with expat; both are restated
 *      here in plain C++ (no dependency), the sample payload goes through the same reader / chain / writer
 *      pass as a raw file. ------------------------------------------------------------------------------- */
enum { IQGPU_CONTAINER_RAW = 0, IQGPU_CONTAINER_WAV = 1, IQGPU_CONTAINER_RF64 = 2 };
/* SdrSoftwareType (src/input_wav.c:56-62) */
enum { IQGPU_SDR_SOFTWARE_UNKNOWN = 0, IQGPU_SDR_CONSOLE, IQGPU_SDR_SHARP, IQGPU_SDR_UNO, IQGPU_SDR_CONNECT };

typedef struct {
    /* what sf_open + SF_INFO give the reference (src/input_wav.c:552-598) */
    int32_t  container;             /* IQGPU_CONTAINER_WAV or IQGPU_CONTAINER_RF64 */
    int32_t  sample_format;         /* IQGPU_FMT_CS16 (PCM_16) or IQGPU_FMT_CU8 (PCM_U8); anything else is refused */
    int32_t  format_tag;            /* 1 = PCM, 3 = IEEE float, 0xFFFE = extensible (sub-format resolved) ... */
    int32_t  channels;
    int32_t  bits_per_sample;
    int32_t  sample_rate_hz;
    uint64_t data_offset;           /* file offset of the first sample byte */
    uint64_t data_bytes;            /* payload length, clipped to the file */
    uint64_t frames;                /* data_bytes / (channels * bytes per sample) */
    /* SdrMetadata (src/input_wav.c:64-78) */
    int32_t  metadata_present;      /* WavPrivateData.sdr_info_present */
    int32_t  source_software;       /* IQGPU_SDR_* */
    int32_t  center_freq_hz_present;
    int32_t  timestamp_unix_present;
    double   center_freq_hz;
    int64_t  timestamp_unix;
    int32_t  timestamp_str_present;
    int32_t  software_name_present;
    int32_t  software_version_present;
    int32_t  radio_model_present;
    char     timestamp_str[64];
    char     software_name[64];
    char     software_version[64];
    char     radio_model[128];
} iqgpu_wav_info;

/* wav_initialize up to the shift decision: header, first auxi chunk, then the file name.  Host only (no device).
 * Fails with IQGPU_EINVAL (message in iqgpu_rawfile_last_error) where the reference log_fatal()s: not a WAV/RF64
 * file, channels != 2, a PCM subtype other than 16-bit signed / 8-bit unsigned, sample rate <= 0. */
int  iqgpu_wav_probe(const char *path, iqgpu_wav_info *info);
/* the two metadata sources on their own (info must be zeroed or hold earlier results; return 1 if anything
 * new was parsed, 0 if not): an auxi chunk body — XML <Definition .../> attributes first (SDR Console), the
 * binary SYSTEMTIME + centre-frequency layout second (SDRuno / SDR#) — and the base name of the file. */
int  iqgpu_wav_parse_auxi(const void *chunk, size_t bytes, iqgpu_wav_info *info);
int  iqgpu_wav_parse_filename(const char *base_filename, iqgpu_wav_info *info);
/* --wav-center-target-freq (src/input_wav.c:612-629): nco_shift_hz = centre frequency - (double)target.
 * IQGPU_EINVAL if a --freq-shift was given as well or the file carries no centre frequency. */
int  iqgpu_wav_center_target_shift(const iqgpu_wav_info *info, float center_target_hz, double freq_shift_hz_arg,
                                   double *nco_shift_hz);
/* the header libsndfile leaves in front of `data_bytes` of 2-channel PCM once the file is closed
 * (44 bytes for WAV, 80 for RF64: RF64 / ds64 / fmt / data); output_format is CS16 or CU8
 * (wav_common_validate_options, src/output_wav_common.c:46-52), the rate is (int)target_rate (:96). */
size_t iqgpu_wav_header_bytes(int container);
int  iqgpu_wav_build_header(int container, int output_format, int sample_rate_hz, uint64_t data_bytes,
                            void *header, size_t capacity);
/* A whole file run: in_container RAW takes format and rate from cfg; WAV / RF64 (either value: the header
 * decides) take them from the file the way wav_initialize does, and center_target_hz != 0 turns the file's
 * centre-frequency metadata into the chain's shift.  out_container RAW writes the bare samples, WAV / RF64
 * the container.  `in_info` (optional) receives the probe result. */
int  iqgpu_wavfile_run(const iqgpu_chain_config *cfg, int device, const char *in_path, int in_container,
                       const char *out_path, int out_container, float center_target_hz, size_t train_chunks,
                       iqgpu_rawfile_stats *stats /* optional */, iqgpu_wav_info *in_info /* optional */);
/* The same with several channels out of one input (iqgpu_rawfile_run_channels): a WAV / RF64 input gives every
 * channel its format and rate, a non-zero center_target_hz[k] turns its centre frequency into channel k's shift, and
 * each container output carries its own channel's rate.  iqgpu_wavfile_run is the one-channel case. */
int  iqgpu_wavfile_run_channels(const iqgpu_chain_config *cfgs, size_t n_channels, int device, const char *in_path,
                                int in_container, const char *const *out_paths, const int *out_containers,
                                const float *center_target_hz /* [n_channels] or NULL */, size_t train_chunks,
                                iqgpu_rawfile_stats *stats /* [n_channels] or NULL */, iqgpu_wav_info *in_info /* optional */);

/* ---- sample_convert.h (include/sample_convert.h:19,35,50) — host buffers ------------- */
size_t iqgpu_get_bytes_per_sample(int format);
int    iqgpu_convert_block_to_cf32(const void *in, float *out_cf32, size_t n_frames, int format, float gain);
int    iqgpu_convert_cf32_to_block(const float *in_cf32, void *out, size_t n_frames, int format);

/* ---- I/Q optimiser metric (include/iq_correct.h:56; src/iq_correct.c:154-235,315-393) -
 * One optimisation pass on a 1024-sample cf32 block: power estimate, 1+25 metric evaluations
 * with caller-supplied +-1 directions (2*25 floats; the reference draws them from rand()),
 * 5 % smoothing.  in/out: mag, phase.  Returns average_power / power_range as the reference
 * stores them. */
int  iqgpu_iq_optimize(const float *block1024_cf32, const float *directions50,
                       float *mag, float *phase, float *avg_power, float *power_range);

/* ---- diagnostics (not on the data path) --------------------------------------------------------------------------
 * FP32 FMA peak of `device` in TFLOP/s, measured with the instruction the kernels spend their FLOPs in (packed FFMA2 with
 * a warp-uniform tap): the denominator of the FP32 roofline bench.py reports (BASELINE.md asks for the measured figure). */
int  iqgpu_ubench_fp32_peak(int device, double *tflops, double *kernel_ms /* optional */);

#ifdef __cplusplus
}
#endif
#endif /* IQGPU_H */
