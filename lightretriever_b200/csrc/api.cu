// api.cu — error reporting and device queries of the C ABI (include/lr_b200.h).
#include "umma_gemm.cuh"

#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <map>
#include <utility>

namespace lr {

static thread_local char g_err[1024] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int sm_count() {
  static int cached[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) {
    cudaGetLastError();
    return 148;  // B200; only reached on a box without a CUDA device (workspace sizing in CPU tests)
  }
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) {
      cudaGetLastError();
      return 148;
    }
    cached[dev] = n;
  }
  return cached[dev];
}

int ensure_dyn_smem(const void* func, int bytes) {
  static std::mutex mu;
  static std::map<std::pair<int, const void*>, int> have;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) {
    set_error("no CUDA device: %s", cudaGetErrorString(cudaGetLastError()));
    return LR_ECUDA;
  }
  std::lock_guard<std::mutex> lock(mu);
  int& cur = have[std::make_pair(dev, func)];
  if (bytes <= cur) return LR_OK;
  cudaError_t e = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess) {
    set_error("cudaFuncSetAttribute(MaxDynamicSharedMemorySize=%d) failed: %s", bytes, cudaGetErrorString(e));
    return LR_ECUDA;
  }
  cur = bytes;
  return LR_OK;
}

static std::atomic<unsigned long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

static std::atomic<unsigned> g_env_epoch{1};
unsigned env_epoch() { return g_env_epoch.load(std::memory_order_acquire); }

// an unset or empty variable means the default
static int env_int(const char* name, int dflt) {
  const char* s = getenv(name);
  return (s && *s) ? atoi(s) : dflt;
}

// Every knob the library reads, with its default (DESIGN.md appendix mirrors this list).
const Knobs& knobs() {
  static thread_local Knobs k;
  static thread_local unsigned epoch = 0;
  const unsigned ep = env_epoch();
  if (epoch != ep) {
    k.flatip_prefix_docs = env_int("LR_FLATIP_PREFIX_DOCS", -1);
    k.flatip_cluster = env_int("LR_FLATIP_CLUSTER", 0);
    k.flatip_refresh = env_int("LR_FLATIP_REFRESH", -1);
    k.head_tiles_per_split = env_int("LR_SPARSE_HEAD_TILES_PER_SPLIT", KNOB_UNSET);
    k.head_docs_per_unit = env_int("LR_SPARSE_HEAD_DOCS_PER_UNIT", KNOB_UNSET);
    k.head_sched = env_int("LR_SPARSE_HEAD_SCHED", 1);
    k.head_team_band = env_int("LR_SPARSE_HEAD_TEAM_BAND", KNOB_UNSET);
    k.head_team_window = env_int("LR_SPARSE_HEAD_TEAM_WINDOW", 1);
    k.head_cluster = env_int("LR_SPARSE_HEAD_CLUSTER", 0);
    const int kern = env_int("LR_SPARSE_KERNEL", 0);
    k.sparse_kernel = (kern == 1 || kern == 3) ? kern : 0;
    k.sparse_acc32 = env_int("LR_SPARSE_ACC", 0) == 32;
    k.sparse_debug = env_int("LR_SPARSE_DEBUG", 0) != 0;
    epoch = ep;
  }
  return k;
}

ProfileEvents& profile_events() {
  static thread_local ProfileEvents pe;
  return pe;
}

}  // namespace lr

extern "C" int lr_set_profile_events(void* ev_begin, void* ev_end) {
  lr::ProfileEvents& pe = lr::profile_events();
  pe.begin = static_cast<cudaEvent_t>(ev_begin);
  pe.end = static_cast<cudaEvent_t>(ev_end);
  return LR_OK;
}

extern "C" int lr_reload_env(void) {
  lr::g_env_epoch.fetch_add(1, std::memory_order_acq_rel);
  return LR_OK;
}

extern "C" unsigned long long lr_kernel_launches(void) { return lr::g_launches.load(std::memory_order_relaxed); }

extern "C" const char* lr_last_error(void) { return lr::g_err; }
extern "C" int lr_version(void) { return 100; }
extern "C" int lr_device_sm_count(void) {
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess ||
      cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) {
    lr::set_error("no CUDA device: %s", cudaGetErrorString(cudaGetLastError()));
    return LR_ECUDA;
  }
  return n;
}
