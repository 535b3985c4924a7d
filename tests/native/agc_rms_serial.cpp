// agc_rms_serial — the RMS AGC (liquid agc_crcf_execute_block, oracle/liquid_compat/liquid_compat.c:574-590) as the plain
// serial loop on the CPU: one sample after the other, in the evaluation order the GPU's step documents (kernels.cu,
// agc_rms_step / agc_rms_step_slow), with the same log / exp (agc_math.h).  The GPU's time-parallel evaluation promises
// the bits of this loop; tests/test_agc_rms_exact.py holds it to that.
// Build: g++ -O2 -shared -fPIC -ffp-contract=off (no contraction: every product and sum below is rounded on its own).
#include <stddef.h>
#include "../../iq_tool_b200/csrc/agc_math.h"

extern "C" {

// x, y: n interleaved complex floats (y == x allowed); state: {g, y2'} in, the end state out.
// stats (optional, 5 counters, added to): [0] steps whose y2' (after the update) is <= 1e-6 (gain frozen),
// [1] steps through agc_exp_small (0.125 < |t| <= 0.5), [2] steps through exp (|t| > 0.5), [3] steps that clamp g at 1e6,
// [4] steps off the GPU's straight-line path (alpha*y2 not a positive normal float, y2' <= 1e-6, or |t| not a normal float
// <= 0.125): what a test input exercises, not part of the result.
void agc_rms_serial(const float* x, float* y, size_t n, float alpha, float* state, unsigned long long* stats)
{
    static AgcLogEntry tab[AGC_LOG_N];
    static bool have_tab = false;
    if (!have_tab) { agc_log_table(tab); have_tab = true; }
    static const double K[AGC_NCOEF] = AGC_COEF_LIST;
    const double oma = 1.0 - (double)alpha;
    const float mha = -0.5f * alpha;
    float g = state[0], y2p = state[1];
    for (size_t i = 0; i < n; i++) {
        const float yr = x[2 * i] * g, yi = x[2 * i + 1] * g;
        const float rr = yr * yr, ii = yi * yi;
        const float y2 = rr + ii;
        const float ay2 = alpha * y2;
        const float y2n = (float)fma(oma, (double)y2p, (double)ay2);      // (1 - alpha) y2' + alpha y2, one rounding
        bool generic = !(ay2 >= 1.17549435e-38f && ay2 <= 3.40282347e38f);
        if (y2n > 1e-6f) {
            const float lf = (float)agc_log_fast(y2n, tab, K);
            const float tt = mha * lf;
            const float at = fabsf(tt);
            float ex;
            if (at <= 0.125f) {
                ex = (float)agc_exp_tiny((double)tt, K);
                if (at < 1.17549435e-38f) generic = true;
            } else if (at <= 0.5f) {
                ex = (float)agc_exp_small((double)tt);
                generic = true;
                if (stats) stats[1]++;
            } else {
                ex = (float)exp((double)tt);
                generic = true;
                if (stats) stats[2]++;
            }
            g = g * ex;
        } else {
            generic = true;
            if (stats) stats[0]++;
        }
        if (g > 1e6f) {
            g = 1e6f;
            if (stats) stats[3]++;
        }
        y2p = y2n;
        if (stats && generic) stats[4]++;
        y[2 * i] = yr;
        y[2 * i + 1] = yi;
    }
    state[0] = g;
    state[1] = y2p;
}

}
