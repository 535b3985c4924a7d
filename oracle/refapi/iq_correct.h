/* iq_correct.h — see stages.h.  TEST INFRASTRUCTURE. */
#include "stages.h"
