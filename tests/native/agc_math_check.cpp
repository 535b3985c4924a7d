// agc_math_check — the GPU's logf / expf for the RMS AGC (iq_tool_b200/csrc/agc_math.h, plain IEEE double arithmetic)
// against long double on the CPU; run by tests/test_agc_rms_exact.py.  Usage: agc_math_check [stride]   (stride 1 = every
// float in range).  Ranges: log over [1e-6, FLT_MAX] (every argument the recurrence takes the log of: y2' > 1e-6 up to the
// ~1e12 of a full-scale burst behind a gain held at its 1e6 clamp, and on to the largest float) plus a dense sweep around
// 1.0 (the AGC's steady state); agc_exp_tiny over 1e-12 <= |t| <= 0.125; agc_exp_small over 0.125 <= |t| <= 0.5.
// Prints per function the largest pre-rounding relative error (against long double), how many float results differ from
// the correctly rounded one (the long double result rounded to float) and, for information, from this libm's (glibc's logf
// / expf are not correctly rounded: ~0.3 % / ~0.01 % of arguments are one ulp off).  Exit code 1 if a pre-rounding error
// exceeds 2e-15, i.e. if the result could differ from the correctly rounded one for more than ~1e-7 of the arguments.
#include <cfloat>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include "../../iq_tool_b200/csrc/agc_math.h"

struct Tally {
    const char* name;
    unsigned long long n = 0, off_cr = 0, off_libm = 0;
    double worst = 0.0, worst_at = 0.0;
    void add(float arg, double mine, long double exact, float libm)
    {
        if (exact != 0.0L) {
            const double rel = (double)fabsl(((long double)mine - exact) / exact);
            if (rel > worst) { worst = rel; worst_at = arg; }
        }
        n++;
        if ((float)mine != (float)exact) off_cr++;
        if ((float)mine != libm) off_libm++;
    }
    void print() const
    {
        printf("%s: %llu arguments, %llu differ from the correctly rounded float, %llu from libm, "
               "worst pre-rounding relative error %.3g at %.9g\n", name, n, off_cr, off_libm, worst, worst_at);
    }
};

static uint32_t bits(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }
static float from_bits(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }

int main(int argc, char** argv)
{
    const uint32_t stride = argc > 1 ? (uint32_t)atoi(argv[1]) : 97;
    AgcLogEntry tab[AGC_LOG_N];
    agc_log_table(tab);
    static const double K[AGC_NCOEF] = AGC_COEF_LIST;
    Tally tlog{"logf"}, ttiny{"agc_exp_tiny"}, tsmall{"agc_exp_small"};
    // log: every stride-th float in [1e-6, FLT_MAX] plus every float in [0.96, 1.04]
    for (int pass = 0; pass < 2; pass++) {
        const uint32_t lo = bits(pass ? 0.96f : 1.0e-6f), hi = bits(pass ? 1.04f : FLT_MAX), st = pass ? 1 : stride;
        for (uint64_t u = lo; u <= hi; u += st) {
            const float x = from_bits((uint32_t)u);
            tlog.add(x, agc_log_fast(x, tab, K), logl((long double)x), logf(x));
        }
    }
    // exp: both signs, every stride-th float of each range
    for (int sgn = 0; sgn < 2; sgn++) {
        for (int small = 0; small < 2; small++) {
            const uint32_t lo = bits(small ? 0.125f : 1.0e-12f), hi = bits(small ? 0.5f : 0.125f);
            for (uint64_t u = lo; u <= hi; u += stride) {
                float t = from_bits((uint32_t)u);
                if (sgn) t = -t;
                const double d = small ? agc_exp_small((double)t) : agc_exp_tiny((double)t, K);
                (small ? tsmall : ttiny).add(t, d, expl((long double)t), expf(t));
            }
        }
    }
    tlog.print();
    ttiny.print();
    tsmall.print();
    return (tlog.worst > 2e-15 || ttiny.worst > 2e-15 || tsmall.worst > 2e-15) ? 1 : 0;
}
