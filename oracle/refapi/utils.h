/* utils.h — the call the drop-in layer makes (reference include/utils.h). TEST INFRASTRUCTURE. */
#ifndef REFAPI_UTILS_H
#define REFAPI_UTILS_H
double get_monotonic_time_sec(void);
#endif
