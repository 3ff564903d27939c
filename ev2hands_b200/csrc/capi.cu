// Status plumbing of the C ABI (include/ev2h.h).
#include "common.cuh"
#include <string.h>

namespace ev2h {
static thread_local char g_err[512] = "";
void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
}  // namespace ev2h

extern "C" int ev2h_version(void) { return 102; }
extern "C" const char *ev2h_last_error(void) { return ev2h::g_err; }
