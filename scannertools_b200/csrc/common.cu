// Error reporting, device queries and library-level entry points of the C ABI (include/stb.h).
#include "stb_rt.h"

#include <cstring>

namespace stb {

static thread_local char g_err[512] = "";
#ifndef STB_CPU_EMU
std::atomic<long long> g_launches{0};
#endif

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
  set_error("CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
  // cudaErrorNoDevice = 100, cudaErrorInsufficientDriver = 35
  if ((int)e == 100 || (int)e == 35) return STB_ERR_NO_DEVICE;
  return (int)e > 0 ? (int)e : STB_ERR_INVALID;
}

int current_device() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;
  return dev;
}

int num_sms() {
#ifdef STB_CPU_EMU
  return 2;
#else
  static int cached[64] = {};
  const int dev = current_device();
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0) cached[dev] = n;
    else return 148;
  }
  return cached[dev];
#endif
}

}  // namespace stb

extern "C" {

int stb_version(void) { return 100; }

const char* stb_last_error(void) { return stb::g_err; }

long long stb_launch_count(void) {
#ifndef STB_CPU_EMU
  return stb::g_launches.load(std::memory_order_relaxed);
#else
  return 0;
#endif
}

int stb_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    (void)cudaGetLastError();
    return 0;
  }
  return n;
}

}  // extern "C"

// The CPU emulator library (tests/cuda_emu) is built from a fixed list of translation units; sources added after
// that list join this one there.  The nvcc build compiles them on their own (build.py SOURCES).
#ifdef STB_CPU_EMU_BUILD
#include "blur.cu"
#endif
