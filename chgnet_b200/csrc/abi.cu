// Library-level pieces of the C ABI: error string, version, launch counter, the one run-time option.
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>

#include "common.cuh"

namespace chg {
namespace {
thread_local char g_err[512] = "";
std::atomic<int64_t> g_launches{0};
std::atomic<int> g_ws_min_rows{4096};  // gated_common.cuh
}  // namespace

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

int sm_count() {  // of the CURRENT device (cached per device ordinal)
  static std::atomic<int> cache[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;  // B200
  int n = cache[dev].load(std::memory_order_relaxed);
  if (n == 0) {
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cache[dev].store(n, std::memory_order_relaxed);
  }
  return n;
}
int ws_min_rows() { return g_ws_min_rows.load(); }
}  // namespace chg

extern "C" int chg_set_option(const char* name, int32_t value) {
  if (name == nullptr) return CHG_ERR_ARG;
  if (strcmp(name, "ws_min_rows") == 0) { chg::g_ws_min_rows.store(value < 0 ? 0 : value); return CHG_OK; }
  chg::set_error("chg_set_option: unknown option %s", name);
  return CHG_ERR_ARG;
}

extern "C" const char* chg_last_error(void) { return chg::g_err; }
extern "C" int chg_abi_version(void) { return 3; }
extern "C" int64_t chg_launch_count(void) { return chg::g_launches.load(std::memory_order_relaxed); }
