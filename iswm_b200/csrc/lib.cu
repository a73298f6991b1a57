// lib.cu — process-wide plumbing of libiswm_b200.so: thread-local error text,
// launch counter, version.
#include "common.cuh"
#include <stdarg.h>
#include <stdlib.h>

namespace iswm {
static thread_local char t_err[512] = "";
std::atomic<int64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(t_err, sizeof(t_err), fmt, ap);
  va_end(ap);
}
std::atomic<int> g_skip_mask{0};
bool pdl_enabled() {
  static const bool on = [] {
    const char* e = getenv("ISWM_PDL");
    return !(e && e[0] == '0');
  }();
  return on;
}
}  // namespace iswm

extern "C" const char* iswm_last_error(void) { return iswm::t_err; }
extern "C" int iswm_version(void) { return 100; }
extern "C" int64_t iswm_launch_count(void) { return iswm::g_launches.load(); }
extern "C" void iswm_reset_launch_count(void) { iswm::g_launches.store(0); }
extern "C" void iswm_debug_set_skip(int mask) { iswm::g_skip_mask.store(mask); }
