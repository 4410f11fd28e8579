// lib.cu -- library plumbing: error text, launch counter, device properties.
#include <stdarg.h>

#include <atomic>
#include <mutex>
#include <unordered_map>

#include "common.cuh"

namespace colo {

static thread_local char g_err[512] = "";
static std::atomic<unsigned long long> g_launches{0};
// launches per Bellman-solver path (colo_solver_path_launches), counted on the host where the path is chosen
static std::atomic<unsigned long long> g_path_launches[COLO_PATH_KINDS];

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

void count_launch(unsigned long long n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
void count_solver_path(int kind) { g_path_launches[kind].fetch_add(1, std::memory_order_relaxed); }

int check_launch(const char* what) {
  count_launch(1);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("launch of %s failed: %s", what, cudaGetErrorString(e));
    return COLO_ERR_CUDA;
  }
  return COLO_OK;
}

// cudaFuncAttributeMaxDynamicSharedMemorySize is per-kernel STATE: a host thread that lowers it between another
// thread's set and launch makes that launch fail ("invalid argument").  The library's entry points are called from
// several host threads (one stream each), so the attribute only ever GROWS, under a lock.
int ensure_dynamic_smem(const void* kernel, size_t bytes) {
  static std::mutex mu;
  static std::unordered_map<const void*, size_t> current;
  std::lock_guard<std::mutex> lock(mu);
  size_t& cur = current[kernel];
  if (bytes > cur) {
    const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) {
      cudaGetLastError();
      set_error("cudaFuncSetAttribute(MaxDynamicSharedMemorySize = %zu) failed: %s", bytes, cudaGetErrorString(e));
      return COLO_ERR_CUDA;
    }
    cur = bytes;
  }
  return COLO_OK;
}

int sm_count() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

}  // namespace colo

extern "C" {
const char* colo_last_error(void) { return colo::g_err; }
int colo_version(void) { return 100; }
unsigned long long colo_launch_count(void) { return colo::g_launches.load(); }
void colo_reset_launch_count(void) { colo::g_launches.store(0); }
unsigned long long colo_solver_path_launches(int kind) {
  return kind >= 0 && kind < COLO_PATH_KINDS ? colo::g_path_launches[kind].load(std::memory_order_relaxed) : 0ULL;
}
int colo_stream_synchronize(void* stream) {
  COLO_CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
  return COLO_OK;
}
}
