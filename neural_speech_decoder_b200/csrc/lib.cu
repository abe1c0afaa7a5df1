// Library-level entry points: version, error string, device info.
#include <stdarg.h>

#include "common.cuh"

namespace nsd {

static thread_local char g_err[512] = "";

unsigned long long launches();

void set_seed_offset_ptr(const unsigned long long* p);

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

static unsigned long long g_launches = 0;
void count_launch(int n) { __atomic_fetch_add(&g_launches, (unsigned long long)n, __ATOMIC_RELAXED); }
unsigned long long launches() { return __atomic_load_n(&g_launches, __ATOMIC_RELAXED); }

int sm_count() {
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (cached[dev] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached[dev] = n;
    }
    return cached[dev];
}

static const unsigned long long* g_seed_off = nullptr;
const unsigned long long* seed_offset_ptr() { return g_seed_off; }
void set_seed_offset_ptr(const unsigned long long* p) { g_seed_off = p; }

}  // namespace nsd

extern "C" {

int nsd_version(void) { return 100; }   // 0.1.0

int nsd_set_seed_offset_ptr(const void* dev_u64) {
    nsd::set_seed_offset_ptr(reinterpret_cast<const unsigned long long*>(dev_u64));
    return NSD_OK;
}

unsigned long long nsd_launch_count(void) { return nsd::launches(); }

const char* nsd_last_error(void) { return nsd::g_err; }

int nsd_device_info(int* sm_count, int* cc_major, int* cc_minor) {
    int dev = 0;
    NSD_CUDA(cudaGetDevice(&dev));
    cudaDeviceProp p;
    NSD_CUDA(cudaGetDeviceProperties(&p, dev));
    if (sm_count) *sm_count = p.multiProcessorCount;
    if (cc_major) *cc_major = p.major;
    if (cc_minor) *cc_minor = p.minor;
    return NSD_OK;
}

}  // extern "C"
