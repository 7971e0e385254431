// Error reporting and small host utilities behind include/hypernerf_b200.h.
#include <string.h>
#include "hn_api_internal.h"

namespace hn {

static thread_local char g_err[512] = "";

int set_error(int code, const char* msg) {
  strncpy(g_err, msg ? msg : "", sizeof(g_err) - 1);
  g_err[sizeof(g_err) - 1] = 0;
  return code;
}

int set_cuda_error(cudaError_t e, const char* where) {
  if (e == cudaSuccess) return 0;
  snprintf(g_err, sizeof(g_err), "%s: %s (%s)", where ? where : "cuda", cudaGetErrorString(e), cudaGetErrorName(e));
  return (int)e;
}

int num_sms() {
  static thread_local int cached_dev = -1, cached = 0;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  if (dev != cached_dev) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached = n;
    cached_dev = dev;
  }
  return cached;
}

}  // namespace hn

extern "C" int hn_abi_version(void) { return HN_ABI_VERSION; }
extern "C" const char* hn_last_error(void) { return hn::g_err; }
