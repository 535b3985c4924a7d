/* constants.h — the values of the reference's include/constants.h that the drop-in layer and
 * oracle/ref_harness.c use (restated with their line numbers in oracle/iq_oracle.c). TEST INFRASTRUCTURE. */
#ifndef REFAPI_CONSTANTS_H
#define REFAPI_CONSTANTS_H
#define PIPELINE_CHUNK_BASE_SAMPLES      16384      /* :123 */
#define RESAMPLER_OUTPUT_SAFETY_MARGIN   128        /* :129 */
#define DC_BLOCK_CUTOFF_HZ               10.0f      /* :149 */
#define IQ_CORRECTION_FFT_SIZE           1024       /* :157 */
#define IQ_CORRECTION_INTERVAL_MS        500        /* :159 */
#define IQ_MAX_PASSES                    25         /* :160 */
#define IQ_CORRECTION_POWER_THRESHOLD_DB 20.0f      /* :161 */
#define AGC_DIGITAL_PEAK_TARGET          0.9f       /* :184 */
#define AGC_DX_TARGET                    0.5f       /* the oracle's default for the DX and local profiles */
#define AGC_LOCAL_TARGET                 0.5f
#define MIN_ACCEPTABLE_RATIO             0.001f     /* :245 */
#define MAX_ACCEPTABLE_RATIO             1000.0f    /* :246 */
#define SHIFT_FACTOR_LIMIT               5.0        /* :248 */
#define MAX_FILTER_CHAIN                 5
#endif
