// api.cu -- error plumbing and ABI bookkeeping of libb200ssm.so (see include/b200_ssm.h).
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <mutex>

#include "common.cuh"

namespace b200 {

static thread_local char g_err[512] = "";
static std::atomic<int> g_launches{0};

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

int check_launch(const char* what) {
    count_launch(1);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
        return (int)e;
    }
    return 0;
}

cudaError_t func_attr_per_device(const void* kernel, cudaFuncAttribute attr, int value) {
    struct Entry { const void* k; int attr; unsigned long long devs; };
    static Entry table[512];
    static int n = 0;
    static std::mutex mu;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) dev = 0;
    const unsigned long long bit = 1ull << (dev & 63);
    std::lock_guard<std::mutex> lock(mu);
    Entry* e = nullptr;
    for (int i = 0; i < n; ++i)
        if (table[i].k == kernel && table[i].attr == (int)attr) { e = &table[i]; break; }
    if (e && (e->devs & bit)) return cudaSuccess;
    const cudaError_t rc = cudaFuncSetAttribute(kernel, attr, value);
    if (rc != cudaSuccess) return rc;
    if (!e && n < 512) { table[n] = Entry{kernel, (int)attr, 0ull}; e = &table[n++]; }
    if (e) e->devs |= bit;      // table full: the attribute is simply set again next time (cheap, never wrong)
    return cudaSuccess;
}

}  // namespace b200

extern "C" const char* b200_last_error(void) { return b200::g_err; }
extern "C" int b200_version(void) { return 4; }
extern "C" int b200_kernel_launches(void) { return b200::g_launches.load(std::memory_order_relaxed); }
extern "C" size_t b200_sizeof_params(int32_t which) {
    switch (which) {
        case 0: return sizeof(b200_sscan_fwd_params);
        case 1: return sizeof(b200_sscan_bwd_params);
        case 2: return sizeof(b200_ssd_fwd_params);
        case 3: return sizeof(b200_ssd_bwd_params);
        case 4: return sizeof(b200_ssu_params);
        default: return 0;
    }
}
