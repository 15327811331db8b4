// Library-level plumbing: error string, ABI version, launch counter, per-device launch settings.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"

namespace hqq {

static thread_local char g_err[512] = "";
std::atomic<long long> g_launches{0};
std::atomic<int> g_env_epoch{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int cur_device() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) dev = 0;
  return dev;
}

int sm_count() {
  static int n[kMaxDevices] = {};
  const int dev = cur_device();
  if (!n[dev]) {
    if (cudaDeviceGetAttribute(&n[dev], cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n[dev] <= 0) n[dev] = kNumSMs;
  }
  return n[dev];
}

bool pdl_enabled() {
  HQQ_ENV_KNOB(on, ([] { const char* e = getenv("HQQ_B200_PDL"); return (e && e[0] == '0') ? 0 : 1; })());
  return on == 1;
}

}  // namespace hqq

extern "C" int hqq_b200_abi_version(void) { return HQQ_B200_ABI_VERSION; }
extern "C" const char* hqq_b200_last_error(void) { return hqq::g_err; }
extern "C" int64_t hqq_b200_launch_count(void) { return (int64_t)hqq::g_launches.load(); }
extern "C" void hqq_b200_launch_count_reset(void) { hqq::g_launches.store(0); }
extern "C" void hqq_b200_reload_env(void) { hqq::g_env_epoch.fetch_add(1); }
