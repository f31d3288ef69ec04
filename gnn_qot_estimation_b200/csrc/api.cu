// Error plumbing + version for libqot_b200.
#include <stdarg.h>

#include "common.cuh"

namespace qot {
static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
}  // namespace qot

extern "C" const char* qot_last_error(void) { return qot::g_err; }
extern "C" int qot_version(void) { return 101; }
