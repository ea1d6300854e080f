// Error reporting / bookkeeping of the C ABI.
#include <stdarg.h>

#include <atomic>

#include "common.cuh"

namespace ava {

static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

TensorMapEncodeFn get_tensor_map_encode_fn() {
  static TensorMapEncodeFn fn = nullptr;
  if (fn == nullptr) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<TensorMapEncodeFn>(p);
  }
  return fn;
}

}  // namespace ava

extern "C" const char* ava_b200_last_error(void) { return ava::g_err; }
extern "C" int ava_b200_abi_version(void) { return AVA_B200_ABI_VERSION; }
extern "C" long long ava_b200_launch_count(void) { return ava::g_launches.load(); }
