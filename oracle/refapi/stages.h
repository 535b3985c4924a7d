/* stages.h — the stage and module prototypes of the reference's include/{pre_processor,resampler,
 * post_processor,filter,frequency_shift,sample_convert,dc_block,iq_correct,agc}.h (SURVEY.md 8(b)),
 * which the drop-in layer implements.  The per-module headers below include this one.  TEST INFRASTRUCTURE. */
#ifndef REFAPI_STAGES_H
#define REFAPI_STAGES_H
#include "app_context.h"
#include "memory_arena.h"
#include "pipeline_types.h"

void pre_processor_apply_chain(AppResources *resources, SampleChunk *item);
void pre_processor_reset(AppResources *resources);

resampler_t *create_resampler(const struct AppConfig *config, struct AppResources *resources, float resample_ratio);
void destroy_resampler(resampler_t *resampler);
void resampler_reset(resampler_t *resampler);
void resampler_execute(resampler_t *resampler, complex_float_t *input, unsigned int num_input_frames,
                       complex_float_t *output, unsigned int *num_output_frames);

void post_processor_apply_chain(AppResources *resources, SampleChunk *item);
void post_processor_reset(AppResources *resources);

bool filter_create(AppConfig *config, AppResources *resources, MemoryArena *arena);
void filter_reset(AppResources *resources);
void filter_destroy(AppResources *resources);
unsigned int filter_apply(AppResources *resources, SampleChunk *item, bool is_post_resample);

bool freq_shift_create(AppConfig *config, AppResources *resources);
void freq_shift_apply(void *nco, double shift_hz, complex_float_t *input, complex_float_t *output, unsigned int num_frames);
void freq_shift_reset_nco(void *nco);
void freq_shift_destroy_ncos(AppResources *resources);

size_t get_bytes_per_sample(format_t format);
bool convert_block_to_cf32(const void *input_buffer, complex_float_t *output_buffer, size_t num_frames,
                           format_t input_format, float gain);
bool convert_cf32_to_block(const complex_float_t *input_buffer, void *output_buffer, size_t num_frames,
                           format_t output_format);

bool dc_block_create(AppConfig *config, AppResources *resources);
void dc_block_reset(AppResources *resources);
void dc_block_apply(AppResources *resources, complex_float_t *samples, int num_samples);
void dc_block_destroy(AppResources *resources);

bool iq_correct_init(AppConfig *config, AppResources *resources, MemoryArena *arena);
void iq_correct_apply(AppResources *resources, complex_float_t *samples, int num_samples);
void iq_correct_run_optimization(AppResources *resources, const complex_float_t *optimization_data);
void iq_correct_destroy(AppResources *resources);
bool iq_correct_run_initial_calibration(ModuleContext *ctx, SNDFILE *infile);

bool agc_create(AppConfig *config, AppResources *resources);
void agc_apply(AppResources *resources, complex_float_t *samples, unsigned int num_samples);
void agc_reset(AppResources *resources);
void agc_destroy(AppResources *resources);
#endif
