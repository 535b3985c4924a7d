/* app_context.h — the members of the reference's AppConfig and AppResources
 * (include/app_context.h:66-138, 205-283) that the drop-in layer and oracle/ref_harness.c read or
 * write.  Member names and types follow the reference; members nothing here touches are left out,
 * so the layout is not the reference's.  TEST INFRASTRUCTURE. */
#ifndef REFAPI_APP_CONTEXT_H
#define REFAPI_APP_CONTEXT_H
#include <pthread.h>
#include <stdbool.h>
#include <stddef.h>
#include <stdint.h>

#include "common_types.h"
#include "constants.h"
#include "sndfile.h"

typedef struct resampler_s resampler_t;

typedef struct {
    FilterType type;
    float      freq1_hz;
    float      freq2_hz;
} FilterRequest;

typedef struct AppConfig {
    float  gain;
    bool   gain_provided;
    float  freq_shift_hz_arg;
    bool   shift_after_resample;
    bool   no_resample;
    double target_rate;
    format_t output_format;
    struct { bool enable; } iq_correction;
    struct { bool enable; } dc_block;
    struct {
        bool       enable;
        AgcProfile profile;
        float      target_level;
        float      target_level_arg;
    } output_agc;
    int           num_filter_requests;
    FilterRequest filter_requests[MAX_FILTER_CHAIN];
    float         transition_width_hz_arg;
    int           filter_taps_arg;
    float         attenuation_db_arg;
    int           filter_fft_size_arg;
    const char   *filter_type_str_arg;
    FilterTypeRequest filter_type_request;
    bool          apply_user_filter_post_resample;
} AppConfig;

typedef struct { float mag; float phase; } IqCorrectionFactors;

typedef struct { sf_count_t frames; int samplerate; } SourceInfo;

typedef struct {
    void               *fft_plan;
    pthread_mutex_t     iq_factors_mutex;
    IqCorrectionFactors factors_buffer[2];
    int                 active_buffer_idx;
    float               average_power;
    float               power_range;
    int                 samples_in_accum;
    double              last_optimization_time;
} IqCorrectionResources;

typedef struct AppResources {
    AppConfig      *config;
    SourceInfo      source_info;
    format_t        input_format;
    size_t          input_bytes_per_sample_pair;
    size_t          output_bytes_per_sample_pair;
    bool            is_passthrough;
    float           resample_ratio;
    unsigned int    max_out_samples;
    pthread_mutex_t progress_mutex;
    bool            error_occurred;

    struct { void *dc_block_filter; } dc_block;
    IqCorrectionResources iq_correction;

    double       nco_shift_hz;
    void        *pre_resample_nco;
    void        *post_resample_nco;
    resampler_t *resampler;

    void                    *user_filter_object;
    FilterImplementationType user_filter_type_actual;
    unsigned int             user_filter_block_size;
    complex_float_t         *pre_fft_remainder_buffer;
    unsigned int             pre_fft_remainder_len;
    complex_float_t         *post_fft_remainder_buffer;
    unsigned int             post_fft_remainder_len;

    void    *output_agc_object;
    bool     agc_is_locked;
    float    agc_current_gain;
    float    agc_peak_memory;
    uint64_t agc_samples_seen;
    double   agc_last_strong_peak_time;
} AppResources;

typedef struct ModuleContext { AppConfig *config; AppResources *resources; } ModuleContext;
#endif
