// Host-side runtime bits shared by every translation unit: thread-local error text, launch counter.
#include "dfd_common.cuh"

#include <atomic>
#include <cstdarg>
#include <cstdio>

namespace dfd {

std::atomic<int64_t> g_launches{0};

static thread_local char t_err[1024] = "";

void set_last_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(t_err, sizeof(t_err), fmt, ap);
  va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what, const char* file, int line) {
  set_last_error("CUDA error %d (%s) in %s at %s:%d", (int)e, cudaGetErrorString(e), what, file, line);
  if (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) return DFD_ERR_NO_DEVICE;
  return DFD_ERR_CUDA;
}

}  // namespace dfd

extern "C" DFD_API const char* dfd_last_error(void) { return dfd::t_err; }
extern "C" DFD_API int dfd_version(void) { return 102; }
extern "C" DFD_API int64_t dfd_launch_count(void) {
  return dfd::g_launches.load(std::memory_order_relaxed);
}
