// Library-level entry points: error text, device info, tunables.
#include <stdarg.h>
#include <string.h>

#include <map>
#include <mutex>
#include <set>
#include <string>
#include <utility>

#include "common.cuh"

namespace unreal {

static thread_local char t_error[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(t_error, sizeof(t_error), fmt, ap);
  va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
  set_error("CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
  return UNREAL_ECUDA;
}

// Lazy set-up is per device: a process may drive several devices, and function attributes and device properties belong to
// the device that was current when they were set or queried.
static std::mutex g_dev_mu;

int sm_count() {
  static std::map<int, int> cached;   // device -> SM count
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) == cudaSuccess) {
    std::lock_guard<std::mutex> lk(g_dev_mu);
    auto it = cached.find(dev);
    if (it != cached.end()) return it->second;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess) return cached[dev] = n;
  }
  set_error("cannot query the SM count (no CUDA device?)");
  return 0;
}

int allow_dynamic_smem(const void* kernel, int bytes) {
  static std::set<std::pair<const void*, int>> done;
  int dev = 0;
  UNREAL_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lk(g_dev_mu);
  if (done.count({kernel, dev})) return UNREAL_OK;
  UNREAL_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  done.insert({kernel, dev});
  return UNREAL_OK;
}

static std::mutex g_tun_mu;
static std::map<std::string, int> g_tunables;

int get_tunable(const char* name, int dflt) {
  std::lock_guard<std::mutex> lk(g_tun_mu);
  auto it = g_tunables.find(name);
  return it == g_tunables.end() ? dflt : it->second;
}

}  // namespace unreal

extern "C" const char* unreal_last_error(void) { return unreal::t_error; }

extern "C" int unreal_abi_version(void) { return 1; }

extern "C" int unreal_device_info(int* sm_count, int* cc_major, int* cc_minor) {
  int dev = 0, n = 0, maj = 0, min = 0;
  UNREAL_CUDA(cudaGetDevice(&dev));
  UNREAL_CUDA(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
  UNREAL_CUDA(cudaDeviceGetAttribute(&maj, cudaDevAttrComputeCapabilityMajor, dev));
  UNREAL_CUDA(cudaDeviceGetAttribute(&min, cudaDevAttrComputeCapabilityMinor, dev));
  if (sm_count) *sm_count = n;
  if (cc_major) *cc_major = maj;
  if (cc_minor) *cc_minor = min;
  if (maj != 10) {
    unreal::set_error("libunreal_b200 is built for sm_100a only; device is sm_%d%d", maj, min);
    return UNREAL_ESTATE;
  }
  return UNREAL_OK;
}

extern "C" int unreal_set_tunable(const char* name, int value) {
  UNREAL_REQUIRE(name != nullptr, "unreal_set_tunable: name is null");
  std::lock_guard<std::mutex> lk(unreal::g_tun_mu);
  unreal::g_tunables[name] = value;
  return UNREAL_OK;
}

extern "C" int unreal_get_tunable(const char* name, int* value) {
  UNREAL_REQUIRE(name != nullptr && value != nullptr, "unreal_get_tunable: null argument");
  std::lock_guard<std::mutex> lk(unreal::g_tun_mu);
  auto it = unreal::g_tunables.find(name);
  UNREAL_REQUIRE(it != unreal::g_tunables.end(), "unreal_get_tunable: '%s' is not set", name);
  *value = it->second;
  return UNREAL_OK;
}
