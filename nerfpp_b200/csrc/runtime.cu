// Error text, launch counter and ABI version for libnerfpp_b200.so.
#include "common.cuh"
#include <atomic>
#include <cstdarg>

namespace nrf {

static thread_local char g_err[512] = "";
static std::atomic<int64_t> g_launches{0};

void set_error(const char* fmt, ...)
{
	va_list ap;
	va_start(ap, fmt);
	vsnprintf(g_err, sizeof(g_err), fmt, ap);
	va_end(ap);
}

void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

}  // namespace nrf

extern "C" {

int nrf_abi_version(void) { return NRF_ABI_VERSION; }
const char* nrf_last_error(void) { return nrf::g_err; }
int64_t nrf_launch_count(void) { return nrf::g_launches.load(std::memory_order_relaxed); }

}
