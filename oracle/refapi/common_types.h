/* common_types.h — the types of the reference's include/common_types.h that the drop-in layer and
 * oracle/ref_harness.c use, with the reference's numeric values (cf. oracle/iq_chain_cfg.h).
 * TEST INFRASTRUCTURE: where the reference tree is present its own headers are used instead. */
#ifndef REFAPI_COMMON_TYPES_H
#define REFAPI_COMMON_TYPES_H
#include <complex.h>
#include <stdbool.h>
#include <stddef.h>
#include <stdint.h>

typedef float complex complex_float_t;                       /* :14 */

typedef enum {                                               /* :33-37 */
    FORMAT_UNKNOWN = 0, U8, S8, U16, S16, U32, S32, F32,
    CU8, CS8, CU16, CS16, CS24, CU32, CS32, CF32, SC16Q11
} format_t;

typedef enum { FILTER_NONE = 0, FILTER_LOWPASS, FILTER_HIGHPASS, FILTER_PASSBAND, FILTER_STOPBAND } FilterType;   /* :45-51 */

typedef enum {                                               /* :53-59 */
    FILTER_IMPL_NONE = 0, FILTER_IMPL_FIR_SYMMETRIC, FILTER_IMPL_FIR_ASYMMETRIC,
    FILTER_IMPL_FFT_SYMMETRIC, FILTER_IMPL_FFT_ASYMMETRIC
} FilterImplementationType;

typedef enum { FILTER_TYPE_AUTO = 0, FILTER_TYPE_FIR, FILTER_TYPE_FFT } FilterTypeRequest;   /* :61-65 */

typedef enum { AGC_PROFILE_OFF = 0, AGC_PROFILE_DX, AGC_PROFILE_LOCAL, AGC_PROFILE_DIGITAL } AgcProfile;   /* :77-82 */
#endif
