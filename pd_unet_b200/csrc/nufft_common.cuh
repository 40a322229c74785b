// Shared by nufft.cu (generic path: pad / cuFFT or generic pruned FFT, table gather, atomic scatter, CSR gather) and
// nufft_fused.cu (row-binned separable interpolation fused into the register-resident FFT passes).
#pragma once
#include <cufft.h>

#include <map>
#include <mutex>

#include "common.cuh"
#include "pfft.cuh"
#include "pfft_fast.cuh"

struct pdu_nufft_plan {
    int n0 = 0, n1 = 0, k0 = 0, k1 = 0, J = 0, L = 0, shift0 = 0, shift1 = 0;
    int device;
    float2* d_t0 = nullptr;
    float2* d_t1 = nullptr;
    float* d_s0 = nullptr;
    float* d_s1 = nullptr;
    std::map<int, cufftHandle> fft;   // batched 2-D C2C plans keyed by number of planes
    std::mutex mu;
    // own pruned FFT (pfft.cuh): per-axis radix plans and float64-computed twiddle tables; pfft_ok == false
    // (a grid size with a prime factor above 5) keeps the cuFFT path
    bool pfft_ok = false;
    pdu::PfftPlan pf0, pf1;
    float2* d_w0 = nullptr;
    float2* d_w1 = nullptr;
    // a plan of the Toeplitz-embedded normal operator (pdu_toep_plan_create): grid 2 n, no interpolation tables, unit
    // apodisation tables of k0 / k1 entries; accepted only by the pdu_toep_* entry points
    bool toep = false;
};

namespace pdu {

constexpr int MAXJ = 8;

struct NufftDims {
    int n0, n1, k0, k1, J, L;
    float gam0, gam1;       // float32(2 pi / K)
    double shift0, shift1;
};

__device__ __forceinline__ float2 cmul(float2 a, float2 b) {
    return make_float2(fmaf(a.x, b.x, -a.y * b.y), fmaf(a.x, b.y, a.y * b.x));
}
__device__ __forceinline__ float2 cmul_conj(float2 a, float2 b) {   // a * conj(b)
    return make_float2(fmaf(a.x, b.x, a.y * b.y), fmaf(a.y, b.x, -a.x * b.y));
}

// per-axis taps of one sample: wrapped grid index and table coefficient.  JT > 0: compile-time tap count (the
// default J = 6 gets straight-line code, 6-entry register arrays and no per-tap branches); JT == 0: run-time J <= MAXJ
template <int JT = 0>
__device__ __forceinline__ void axis_taps(float om, float gam, int K, int Jrt, int L, const float2* __restrict__ table,
                                          int* gi, float2* co) {
    const int J = JT > 0 ? JT : Jrt;
    constexpr int N = JT > 0 ? JT : MAXJ;
    const float tm = __fdiv_rn(om, gam);
    const int koff = (int)floorf(__fsub_rn(tm, 0.5f * (float)J));
    const int half = (J * L) / 2;
#pragma unroll
    for (int j = 0; j < N; ++j) {
        if (j < J) {
            const int g = koff + 1 + j;
            const float dist = __fmul_rn(__fsub_rn(tm, (float)g), (float)L);
            int q = (int)rintf(dist) + half;
            q = min(max(q, 0), J * L);
            co[j] = __ldg(table + q);
            int gw = g % K;
            if (gw < 0) gw += K;
            gi[j] = gw;
        }
    }
}

__device__ __forceinline__ float2 shift_phase(float om0, float om1, double s0, double s1) {
    double sn, cs;
    sincos((double)om0 * s0 + (double)om1 * s1, &sn, &cs);
    return make_float2((float)cs, (float)sn);
}

static inline NufftDims dims_of(const pdu_nufft_plan* p) {
    NufftDims d;
    d.n0 = p->n0; d.n1 = p->n1; d.k0 = p->k0; d.k1 = p->k1; d.J = p->J; d.L = p->L;
    d.gam0 = (float)(2.0 * 3.14159265358979323846 / p->k0);
    d.gam1 = (float)(2.0 * 3.14159265358979323846 / p->k1);
    d.shift0 = (double)p->shift0;
    d.shift1 = (double)p->shift1;
    return d;
}

// the cropped planes U [planes][n0][n1] of an adjoint as a dense "grid" (k = n), for crop_apod_kernel / smaps_grad_kernel
static inline NufftDims cropped_dims(const pdu_nufft_plan* p) {
    NufftDims d = dims_of(p);
    d.k0 = d.n0;
    d.k1 = d.n1;
    return d;
}

static inline size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

// The coil-map gradient ending of an adjoint (pdu_nufft_adj_smaps_grad_c64, pdu_toep_smaps_grad_c64): instead of
// combining the coils of the cropped planes U [batch][coils], gs[s][c] (+)= scale' * sum_{b : s(b) = s} U[b][c] conj(q[b]),
// s(b) = 0 with one shared map, b with one map per batch element; b runs in increasing order, in registers.
struct SmapsGrad {
    float2* gs;           // [per_batch ? batch : 1][coils][n0][n1] of this chunk
    const float* q;       // [batch][n0][n1] complex64, or [batch][2][n0][n1] float32 (q_split)
    int batch;            // batch elements of this chunk
    int per_batch;        // 0: every b sums into gs[0]; 1: b writes gs[b]
    int q_split;
    int accumulate;       // add to gs instead of overwriting it
    float scale;          // multiplies the transform's own scale (-1 for the conjugate-gradient solve)
};
// The two endings of an adjoint, from planes U [batch][coils] of geometry d (k0 x k1 planes, the n0 x n1 corner kept):
// the image (x apodisation x scale, x conj(smaps) summed over coils), or the coil-map gradient into sg.gs
int launch_crop_apod(pdu_nufft_plan* p, const float2* U, NufftDims d, const float2* smaps, float2* image, int out_planes,
                     int coils, int smaps_batch, float scale, int split, cudaStream_t st);
int launch_smaps_grad(pdu_nufft_plan* p, const float2* U, NufftDims d, int coils, float scale, const SmapsGrad& sg,
                      cudaStream_t st);

// nufft_fused.cu
bool fused_supported(const pdu_nufft_plan* p);
size_t fused_workspace_bytes(const pdu_nufft_plan* p, int planes, long m);
int fused_forward(pdu_nufft_plan* p, const float* image, float* kdata, const float* smaps, int batch, int coils, int smaps_batch,
                  long m, float scale, const void* bins, int flags, void* ws, cudaStream_t st);
// sg: end in smaps_grad_kernel (smaps null) instead of writing the image
int fused_adjoint(pdu_nufft_plan* p, const float* kdata, float* image, const float* smaps, const float* kweight, int batch,
                  int coils, int smaps_batch, long m, float scale, const void* bins, int flags, void* ws, cudaStream_t st,
                  const SmapsGrad* sg = nullptr);

}  // namespace pdu
