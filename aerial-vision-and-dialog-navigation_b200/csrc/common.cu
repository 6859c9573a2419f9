// Error plumbing and device queries for libavdn.so.
#include "common.cuh"

#include <stdlib.h>

namespace avdn {

static thread_local char g_err[512] = "ok";

char* err_buf() { return g_err; }

int set_err(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess)
    return set_err(AVDN_ERR_LAUNCH, "%s: %s", what, cudaGetErrorString(e));
  return AVDN_OK;
}

int sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    cudaDeviceProp p;
    if (cudaGetDeviceProperties(&p, dev) != cudaSuccess) return 148;
    n = p.multiProcessorCount;
  }
  return n;
}

bool pdl_enabled() {
  static const bool on = [] {
    const char* e = getenv("AVDN_PDL");
    return e && e[0] == '1';
  }();
  return on;
}

}  // namespace avdn

extern "C" const char* avdn_last_error_string(void) { return avdn::err_buf(); }

extern "C" int avdn_abi_version(void) { return 11; }

extern "C" int avdn_device_supported(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
    cudaGetLastError();
    return 0;
  }
  cudaDeviceProp p;
  if (cudaGetDeviceProperties(&p, 0) != cudaSuccess) return 0;
  return p.major == 10 ? 1 : 0;
}
