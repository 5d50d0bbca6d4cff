// libhgr.so: error reporting, version and launch accounting of the C ABI (include/hgr.h).
#include "hgr_internal.cuh"

namespace hgr {

static thread_local char t_error[512] = "";
std::atomic<uint64_t> g_launches{0};

int set_error(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(t_error, sizeof(t_error), fmt, ap);
    va_end(ap);
    return code;
}

}  // namespace hgr

extern "C" {

const char *hgr_last_error(void) { return hgr::t_error; }

int hgr_version(void) { return 102; }  // 0.1.2

uint64_t hgr_launch_count(void) { return hgr::g_launches.load(std::memory_order_relaxed); }

}  // extern "C"
