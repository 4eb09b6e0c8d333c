// Library-level entry points: version, error string, launch counter.
#include <stdarg.h>

#include <atomic>

#include "scb_common.cuh"

namespace scb {
static thread_local char g_error[512] = "";
static std::atomic<int64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_error, sizeof(g_error), fmt, ap);
  va_end(ap);
}
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
}  // namespace scb

extern "C" int scb_version(void) { return 205; }
extern "C" const char* scb_last_error(void) { return scb::g_error; }
extern "C" int64_t scb_launch_count(void) { return scb::g_launches.load(); }
