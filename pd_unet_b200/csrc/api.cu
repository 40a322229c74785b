// Library-wide entry points: errors, version, device info, variant switches, launch counter.
#include <stdarg.h>
#include <string.h>

#include <stdlib.h>

#include <atomic>
#include <mutex>

#include "common.cuh"

namespace pdu {

static thread_local char g_err[512] = "";
static std::atomic<long> g_launches{0};
static std::atomic<int> g_opts[OPT_COUNT] = {{-1}, {-1}, {-1}, {-1}, {-1}, {-1}, {-1}};
// room for the longest record (the sorted-gather adjoint, the generic CG: about 270 characters) up to its shape
static thread_local char g_kernel[OP_COUNT][512];

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

// -1 (unset) falls back to the environment: PDU_RADON_FWD_VARIANT, PDU_RADON_ADJ_VARIANT, ...
int option(int which) {
    const int v = g_opts[which].load(std::memory_order_relaxed);
    if (v >= 0) return v;
    static const char* names[OPT_COUNT] = {"PDU_RADON_FWD_VARIANT", "PDU_RADON_ADJ_VARIANT", "PDU_FILTER_VARIANT",
                                           "PDU_NUFFT_ADJ_VARIANT", "PDU_NUFFT_FWD_VARIANT", "PDU_DEBUG_FAULT",
                                           "PDU_TEX_WEIGHTS"};
    static int env[OPT_COUNT];
    static std::once_flag once;
    std::call_once(once, [] {
        for (int i = 0; i < OPT_COUNT; ++i) {
            const char* e = getenv(names[i]);
            env[i] = e && *e ? atoi(e) : -1;
        }
    });
    return env[which];
}
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

void note_kernel(int op, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_kernel[op], sizeof(g_kernel[op]), fmt, ap);
    va_end(ap);
}

int* device_error_word() {
    static int* word = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        if (cudaHostAlloc(&p, 64, cudaHostAllocMapped | cudaHostAllocPortable) == cudaSuccess) {
            memset(p, 0, 64);
            word = (int*)p;
        } else {
            (void)cudaGetLastError();
        }
    });
    return word;
}

int check_device_error(const char* who) {
    int* w = device_error_word();
    const int code = w ? *(volatile int*)w : 0;
    if (code == DEV_ERR_NONE) return PDU_OK;
    static const char* what[] = {"", "forward projector (TMA / mbarrier wait timed out)",
                                 "tensor-core sinogram filter (TMA / MMA pipeline wait timed out)",
                                 "NUFFT (TMA / mbarrier wait timed out)"};
    set_error("%s: an earlier kernel reported a device-side failure: %s; its output is invalid "
              "(pdu_device_error(1) clears the flag)", who, what[code >= 0 && code <= 3 ? code : 0]);
    return PDU_ECUDA;
}

int sm_count() {
    static thread_local int cached_dev = -1, cached = 0;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (dev != cached_dev) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached = n;
        cached_dev = dev;
    }
    return cached;
}

static int opt_index(const char* key) {
    if (!key) return -1;
    if (!strcmp(key, "radon_fwd_variant")) return OPT_RADON_FWD;
    if (!strcmp(key, "radon_adj_variant")) return OPT_RADON_ADJ;
    if (!strcmp(key, "filter_variant")) return OPT_FILTER;
    if (!strcmp(key, "nufft_adj_variant")) return OPT_NUFFT_ADJ;
    if (!strcmp(key, "nufft_fwd_variant")) return OPT_NUFFT_FWD;
    if (!strcmp(key, "debug_fault")) return OPT_DEBUG_FAULT;
    if (!strcmp(key, "tex_weights")) return OPT_TEX_WEIGHTS;
    return -1;
}

}  // namespace pdu

extern "C" {

const char* pdu_last_error(void) { return pdu::g_err; }

int pdu_version(void) { return 100; }

int pdu_device_info(int* sm_count, int* cc_major, int* cc_minor) {
    int dev = 0;
    PDU_CUDA(cudaGetDevice(&dev));
    int v = 0;
    if (sm_count) {
        PDU_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev));
        *sm_count = v;
    }
    if (cc_major) {
        PDU_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrComputeCapabilityMajor, dev));
        *cc_major = v;
    }
    if (cc_minor) {
        PDU_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrComputeCapabilityMinor, dev));
        *cc_minor = v;
    }
    return PDU_OK;
}

int pdu_set_option(const char* key, int value) {
    int i = pdu::opt_index(key);
    PDU_REQUIRE(i >= 0, "pdu_set_option: unknown key '%s'", key ? key : "(null)");
    pdu::g_opts[i].store(value, std::memory_order_relaxed);
    return PDU_OK;
}

int pdu_get_option(const char* key, int* value) {
    int i = pdu::opt_index(key);
    PDU_REQUIRE(i >= 0 && value, "pdu_get_option: unknown key '%s'", key ? key : "(null)");
    *value = pdu::g_opts[i].load(std::memory_order_relaxed);
    return PDU_OK;
}

int pdu_device_error(int reset) {
    int* w = pdu::device_error_word();
    if (!w) return 0;
    const int code = *(volatile int*)w;
    if (reset) *(volatile int*)w = 0;
    return code;
}

const char* pdu_last_kernel(const char* op) {
    static const char* names[pdu::OP_COUNT] = {"radon_fwd", "radon_adj", "filter", "nufft_fwd", "nufft_adj",
                                               "toep", "cg", "smaps_grad"};
    if (!op) return "";
    for (int i = 0; i < pdu::OP_COUNT; ++i)
        if (!strcmp(op, names[i])) return pdu::g_kernel[i];
    return "";
}

long pdu_launch_count(int reset) {
    if (reset) return pdu::g_launches.exchange(0, std::memory_order_relaxed);
    return pdu::g_launches.load(std::memory_order_relaxed);
}

}  // extern "C"
