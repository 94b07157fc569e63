// Library info, error state and the diagnostic launch counters of libdmv3d.
#include <atomic>
#include <mutex>
#include <stdarg.h>
#include <unordered_map>

#include "common.cuh"

namespace dmv {
static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};
static std::atomic<long long> g_tc_launches{0};
// per-label counts, keyed by the label literal's address (the same text from two translation units may be two keys;
// dmv_launch_count_named sums them by content)
static std::mutex g_named_mu;
static std::unordered_map<const char*, long long> g_named;

void count_launch_named(const char* what) {
    std::lock_guard<std::mutex> lk(g_named_mu);
    ++g_named[what];
}

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
void count_tc_launch() { g_tc_launches.fetch_add(1, std::memory_order_relaxed); }
long long tc_launches() { return g_tc_launches.load(std::memory_order_relaxed); }
}  // namespace dmv

extern "C" {
int dmv_version(void) { return 100; /* 0.1.0 */ }
const char* dmv_arch(void) { return "sm_100a"; }
int dmv_last_error(char* buf, size_t n) {
    if (!buf || n == 0) return DMV_E_INVALID_ARG;
    strncpy(buf, dmv::g_err, n - 1);
    buf[n - 1] = 0;
    return DMV_OK;
}
long long dmv_launch_count(void) { return dmv::g_launches.load(std::memory_order_relaxed); }
long long dmv_tc_launch_count(void) { return dmv::tc_launches(); }
long long dmv_launch_count_named(const char* what) {
    if (!what) return 0;
    std::lock_guard<std::mutex> lk(dmv::g_named_mu);
    long long n = 0;
    for (const auto& kv : dmv::g_named)
        if (strcmp(kv.first, what) == 0) n += kv.second;
    return n;
}
}
