/* frequency_shift.h — see stages.h.  TEST INFRASTRUCTURE. */
#include "stages.h"
