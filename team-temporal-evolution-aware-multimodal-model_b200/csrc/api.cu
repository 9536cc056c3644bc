// Error plumbing + device check for the C ABI (include/team_b200.h).
#include <stdarg.h>
#include <atomic>
#include "common.cuh"

namespace team {
static std::atomic<long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
int cuda_fail(cudaError_t e, const char* what) {
    set_error("CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
    return TEAM_ECUDA;
}
}  // namespace team

extern "C" const char* team_last_error(void) { return team::g_err; }
extern "C" int team_version(void) { return 100; }
extern "C" int team_device_check(void) {
    int dev = 0;
    TEAM_CUDA_CHECK(cudaGetDevice(&dev));
    cudaDeviceProp p;
    TEAM_CUDA_CHECK(cudaGetDeviceProperties(&p, dev));
    if (p.major != 10) {
        team::set_error("libteam_b200 is built for sm_100a only; device %d is sm_%d%d", dev, p.major, p.minor);
        return TEAM_EUNSUPPORTED;
    }
    return TEAM_OK;
}

extern "C" long long team_launch_count(void) { return team::g_launches.load(); }
