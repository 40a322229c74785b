// Shared plumbing of libpdu_b200: error reporting, launch accounting, option switches.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "pdu.h"

namespace pdu {

void set_error(const char* fmt, ...);
int option(int which);                 // see enum Opt; -1 == default
void count_launch(int n = 1);
int sm_count();                        // cached multiProcessorCount of the current device

enum Opt { OPT_RADON_FWD = 0, OPT_RADON_ADJ = 1, OPT_FILTER = 2, OPT_NUFFT_ADJ = 3, OPT_NUFFT_FWD = 4, OPT_DEBUG_FAULT = 5,
           OPT_TEX_WEIGHTS = 6, OPT_COUNT };

// Device error word: one int in mapped pinned host memory (same address on host and device, every context).
// A kernel whose mbarrier wait times out (TMA fault, pipeline bug, ...) stores a DEV_ERR_* code there and gives up
// instead of reading an unfilled tile; every entry point looks at the word first (a host read, no synchronisation)
// and returns PDU_ECUDA while it is set.  pdu_device_error(1) reads and clears it.
enum DevErr { DEV_ERR_NONE = 0, DEV_ERR_RADON_FWD = 1, DEV_ERR_FILTER_TC = 2, DEV_ERR_NUFFT = 3 };
int* device_error_word();              // nullptr only if the allocation failed (then kernels skip the report)
int check_device_error(const char* who);

// the kernel the dispatcher of an operator chose most recently (this thread): pdu_last_kernel()
enum Op { OP_RADON_FWD = 0, OP_RADON_ADJ = 1, OP_FILTER = 2, OP_NUFFT_FWD = 3, OP_NUFFT_ADJ = 4, OP_TOEP = 5, OP_CG = 6,
          OP_SMAPS_GRAD = 7, OP_COUNT };
void note_kernel(int op, const char* fmt, ...);

#define PDU_CHECK_DEVICE(who)                          \
    do {                                               \
        int rc__ = pdu::check_device_error(who);       \
        if (rc__) return rc__;                         \
    } while (0)

#define PDU_REQUIRE(cond, ...)                         \
    do {                                               \
        if (!(cond)) {                                 \
            pdu::set_error(__VA_ARGS__);               \
            return PDU_EINVAL;                         \
        }                                              \
    } while (0)

#define PDU_CUDA(call)                                                                      \
    do {                                                                                    \
        cudaError_t e__ = (call);                                                           \
        if (e__ != cudaSuccess) {                                                           \
            pdu::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            return PDU_ECUDA;                                                               \
        }                                                                                   \
    } while (0)

// after a <<<>>> launch
#define PDU_LAUNCHED()                                                                      \
    do {                                                                                    \
        pdu::count_launch();                                                                \
        cudaError_t e__ = cudaPeekAtLastError();                                            \
        if (e__ != cudaSuccess) {                                                           \
            (void)cudaGetLastError();                                                       \
            pdu::set_error("%s:%d launch -> %s", __FILE__, __LINE__, cudaGetErrorString(e__)); \
            return PDU_ECUDA;                                                               \
        }                                                                                   \
    } while (0)

static inline long cdiv(long a, long b) { return (a + b - 1) / b; }

#ifdef __CUDACC__
// cudaFuncAttributeMaxDynamicSharedMemorySize once per (kernel, device, size): the attribute belongs to the device's
// context, so a process that drives several GPUs must set it on each of them (a plain `static bool` did it once).
// Kern is the kernel itself (non-type template parameter): one record per kernel instantiation.
template <auto Kern>
inline cudaError_t ensure_dyn_smem(int bytes) {
    static int set_bytes[64] = {};             // per device ordinal; racing first calls repeat an idempotent call
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    int& rec = set_bytes[dev & 63];
    if (rec >= bytes) return cudaSuccess;
    e = cudaFuncSetAttribute(Kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess) rec = bytes;
    return e;
}
#endif

#ifdef __CUDACC__
// ------------------------------------------------------------------ bounded mbarrier wait + error report
__device__ __forceinline__ unsigned long long global_timer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
// One try with a suspend-time hint (the warp sleeps in hardware instead of spinning).
__device__ __forceinline__ bool mbar_try_wait_hint(uint32_t bar_smem, uint32_t parity, uint32_t hint_ns) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar_smem), "r"(parity), "r"(hint_ns)
        : "memory");
    return ok != 0;
}
// Waits until the barrier phase completes or `timeout_ns` of wall time have passed (a barrier that never completes
// must not hang the GPU box).  Returns false on time-out: the caller reports through report_device_error() and
// abandons its work -- it must NOT go on to read the tile the barrier guards.
__device__ __forceinline__ bool mbar_wait_bounded(uint32_t bar_smem, uint32_t parity, unsigned long long timeout_ns) {
    if (mbar_try_wait_hint(bar_smem, parity, 20000u)) return true;
    const unsigned long long t0 = global_timer_ns();
    do {                                       // the clock is read once per 16 polls: a poll is 4 instructions, the
#pragma unroll 1                               // 64-bit time comparison 7, and waiting warps share the issue slots
        for (int i = 0; i < 16; ++i)           // with the warps that are sampling
            if (mbar_try_wait_hint(bar_smem, parity, 20000u)) return true;
    } while (global_timer_ns() - t0 < timeout_ns);
    return false;
}
__device__ __forceinline__ void report_device_error(int* err_word, int code) {
    if (err_word) {
        *(volatile int*)err_word = code;
        __threadfence_system();
    }
}
constexpr unsigned long long MBAR_TIMEOUT_NS = 2000000000ull;        // 2 s: far beyond any legitimate wait
constexpr unsigned long long MBAR_TIMEOUT_FAULT_NS = 20000000ull;    // 20 ms under debug_fault (tests)

// packed-FP32 helpers (sm_100 FFMA2 / FADD2): a 64-bit register holds (lo, hi) floats
typedef unsigned long long ull;
__device__ __forceinline__ ull pk2(float lo, float hi) { ull r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void upk2(ull v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ ull fma2(ull a, ull b, ull c) { ull d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ ull add2(ull a, ull b) { ull d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ ull add2_rm(ull a, ull b) { ull d; asm("add.rm.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ ull sub2(ull a, ull b) { ull d; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ ull mul2(ull a, ull b) { ull d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
#endif

}  // namespace pdu
