/* post_processor.h — see stages.h.  TEST INFRASTRUCTURE. */
#include "stages.h"
