// Error plumbing and launch accounting for libnpf_b200.
#include <stdarg.h>
#include <string.h>

#include <atomic>

#include "common.cuh"

namespace npf {

static thread_local char g_err[512] = "";
static std::atomic<unsigned long long> g_launches{0};

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

void count_launch(int n) { g_launches.fetch_add((unsigned long long)n, std::memory_order_relaxed); }

static unsigned long long* g_trace = nullptr;
unsigned long long* trace_buffer() { return g_trace; }

int check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s: %s", what, cudaGetErrorString(e));
        return NPF_ECUDA;
    }
    return NPF_OK;
}

}  // namespace npf

// diagnostics: a device buffer of >= 4096 u64 into which CTA 0 of the warp-specialised kernels that support it writes
// (role, event, clock64) records -- profiles/microbench/trace_timeline.py; NULL (the default) disables it
extern "C" int npf_debug_set_trace(unsigned long long* device_buffer) { npf::g_trace = device_buffer; return NPF_OK; }
extern "C" int npf_abi_version(void) { return NPF_ABI_VERSION; }
extern "C" const char* npf_last_error(void) { return npf::g_err; }
extern "C" unsigned long long npf_launch_count(void) { return npf::g_launches.load(std::memory_order_relaxed); }
