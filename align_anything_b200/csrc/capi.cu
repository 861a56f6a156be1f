// capi.cu -- error plumbing and device queries behind the C ABI (include/aa_b200.h).
#include <stdarg.h>
#include <stdio.h>

#include <map>
#include <mutex>
#include <tuple>

#include "common.cuh"

namespace aa {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int check_launch(const char *what) {
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) return AA_OK;
  set_error("%s: %s (%s)", what, cudaGetErrorString(e), cudaGetErrorName(e));
  return static_cast<int>(e);
}

int sm_count() {
  static thread_local int cached_dev = -1;
  static thread_local int cached = 0;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  if (dev != cached_dev) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
      n = 148;
    cached = n;
    cached_dev = dev;
  }
  return cached;
}

int resident_ctas(const void *kernel, int threads, size_t smem) {
  int dev = 0;
  cudaGetDevice(&dev);
  static std::mutex mu;
  static std::map<std::tuple<const void *, int, size_t, int>, int> cache;
  const auto key = std::make_tuple(kernel, threads, smem, dev);
  std::lock_guard<std::mutex> lock(mu);
  auto it = cache.find(key);
  if (it != cache.end()) return it->second;
  int n = 0;
  // a failed query leaves its error for the launch's check_launch to report; the launch then runs one CTA per SM
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, threads, smem) != cudaSuccess || n < 1) return 1;
  cache.emplace(key, n);
  return n;
}

}  // namespace aa

extern "C" int aa_abi_version(void) { return AA_B200_ABI_VERSION; }

extern "C" const char *aa_last_error(void) { return aa::g_err; }

extern "C" int aa_device_info(int *sm_count, int *max_smem_optin) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) {
    aa::set_error("aa_device_info: %s", cudaGetErrorString(e));
    return static_cast<int>(e);
  }
  int major = 0, minor = 0;
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev);
  if (major != 10) {
    aa::set_error("aa_device_info: device %d is sm_%d%d; libaa_b200 is built for sm_100a only", dev,
                  major, minor);
    return AA_ERR_UNSUPPORTED;
  }
  if (sm_count) cudaDeviceGetAttribute(sm_count, cudaDevAttrMultiProcessorCount, dev);
  if (max_smem_optin) cudaDeviceGetAttribute(max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  return AA_OK;
}
