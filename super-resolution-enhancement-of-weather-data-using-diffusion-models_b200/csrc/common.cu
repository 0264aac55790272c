// common.cu -- error string, version, device probe.
#include <stdarg.h>

#include "common.cuh"

namespace wsr {
static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
int g_pdl_mode = 0;
}  // namespace wsr

extern "C" const char* wsr_last_error(void) { return wsr::g_err; }
extern "C" int wsr_version(void) { return 100; }

// programmatic dependent launch on / off for the launches that follow (common.cuh); returns the previous setting
extern "C" int wsr_set_pdl(int on) {
  const int prev = wsr::g_pdl_mode;
  wsr::g_pdl_mode = on ? 1 : 0;
  return prev;
}
extern "C" int wsr_device_is_sm100(void) {
  int dev = 0, major = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return 0;
  return major == 10 ? 1 : 0;
}
