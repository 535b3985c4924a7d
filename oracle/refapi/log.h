/* log.h — the reference's logger interface (include/log.h) as the drop-in layer and
 * oracle/ref_harness.c call it.  TEST INFRASTRUCTURE. */
#ifndef REFAPI_LOG_H
#define REFAPI_LOG_H
enum { LOG_TRACE, LOG_DEBUG, LOG_INFO, LOG_WARN, LOG_ERROR, LOG_FATAL };

void log_set_level(int level);
void log_log(int level, const char *file, int line, const char *fmt, ...) __attribute__((format(printf, 4, 5)));

#define log_trace(...) log_log(LOG_TRACE, __FILE__, __LINE__, __VA_ARGS__)
#define log_debug(...) log_log(LOG_DEBUG, __FILE__, __LINE__, __VA_ARGS__)
#define log_info(...)  log_log(LOG_INFO,  __FILE__, __LINE__, __VA_ARGS__)
#define log_warn(...)  log_log(LOG_WARN,  __FILE__, __LINE__, __VA_ARGS__)
#define log_error(...) log_log(LOG_ERROR, __FILE__, __LINE__, __VA_ARGS__)
#define log_fatal(...) log_log(LOG_FATAL, __FILE__, __LINE__, __VA_ARGS__)
#endif
