// Library-level entry points (version, last-error text) and the SM count the persistent kernels size their grids by.
#include "common.cuh"
#include <string.h>

static thread_local char g_err[512] = "";

void ssp_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int ssp_num_sms() {
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0)
      sms = 148;
  }
  return sms;
}

extern "C" const char* ssp_last_error(void) { return g_err; }
extern "C" int ssp_version(void) { return 100; }  // 0.1.0
