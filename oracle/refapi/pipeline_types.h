/* pipeline_types.h — the reference's SampleChunk (include/pipeline_types.h:32-55), the members the
 * drop-in layer and oracle/ref_harness.c use.  TEST INFRASTRUCTURE. */
#ifndef REFAPI_PIPELINE_TYPES_H
#define REFAPI_PIPELINE_TYPES_H
#include <stdbool.h>
#include <stddef.h>
#include <stdint.h>

#include "common_types.h"

typedef struct SampleChunk {
    void            *raw_input_data;
    complex_float_t *complex_sample_buffer_a;
    complex_float_t *complex_sample_buffer_b;
    unsigned char   *final_output_data;
    complex_float_t *current_input_buffer;
    complex_float_t *current_output_buffer;
    size_t           raw_input_capacity_bytes;
    size_t           complex_buffer_capacity_samples;
    size_t           final_output_capacity_bytes;
    size_t           input_bytes_per_sample_pair;
    int64_t          frames_read;
    unsigned int     frames_to_write;
    format_t         packet_sample_format;
    bool             is_last_chunk;
    bool             stream_discontinuity_event;
} SampleChunk;
#endif
