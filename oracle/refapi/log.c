/* log.c — a stderr logger behind log.h, for the drop-in test harness. TEST INFRASTRUCTURE. */
#include "log.h"

#include <stdarg.h>
#include <stdio.h>

static int g_level = LOG_INFO;

void log_set_level(int level) { g_level = level; }

void log_log(int level, const char *file, int line, const char *fmt, ...)
{
    static const char *names[] = {"TRACE", "DEBUG", "INFO", "WARN", "ERROR", "FATAL"};
    if (level < g_level) return;
    va_list ap;
    va_start(ap, fmt);
    fprintf(stderr, "%s %s:%d: ", names[level], file, line);
    vfprintf(stderr, fmt, ap);
    fputc('\n', stderr);
    va_end(ap);
}
