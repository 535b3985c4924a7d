/* signal_handler.h — the call the drop-in layer makes (reference include/signal_handler.h). TEST INFRASTRUCTURE. */
#ifndef REFAPI_SIGNAL_HANDLER_H
#define REFAPI_SIGNAL_HANDLER_H
#include "app_context.h"
void handle_fatal_thread_error(const char *context_msg, AppResources *resources);
#endif
