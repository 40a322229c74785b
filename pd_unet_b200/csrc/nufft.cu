// Radial-MRI non-uniform FFT: Kaiser-Bessel table interpolation around an oversampled FFT.
// Replaces [RECALL] torchkbnufft KbNufft / KbNufftAdjoint / KbInterp / KbInterpAdjoint, which are
// compositions of ATen ops (complex multiply, pad, torch.fft, index arithmetic, index_add_).
//
//   forward :  grids 512 / 640 (the BASELINE shapes): ff_rows_fwd_kernel (apodise, * smaps, pruned row FFT of the
//                N non-zero rows) ; ff_cols_fwd_kernel (pruned column FFT)        -- pfft_fast.cuh, 2 passes
//              other grids: apod_pad_kernel + cuFFT, or the generic pruned FFT of pfft.cuh (variant 1)
//              interp_fwd_kernel J x J table-weighted gather per k-space sample, * phase
//   normal operator (Toeplitz embedding, pdu_toep_*; no interpolation):
//              square 2 N a FastFft size: ff_rows_fwd_kernel (unit apodisation) ; tz_cols_kernel (pruned column FFT,
//                x kernel column, pruned inverse column FFT, in place) ; tz_rows_out_kernel (pruned inverse row FFT,
//                x conj(smaps) summed over coils)                                  -- 3 launches, no K x K grid
//              other 2, 3, 5 sizes: pfft rows / cols forward, tz_mul_kernel, pfft rows / cols adjoint, crop_apod_kernel
//   adjoint :  trajectory used more than once: sorted (CSR) gather interp_adj_csrT_kernel on plane-interleaved
//                kdata -- no atomics, no memset, reproducible; else memset + interp_adj_kernel (float2 atomics)
//              inverse FFT: ff_rows_adj_kernel / ff_cols_adj_kernel (only the N kept outputs per axis), or cuFFT
//              crop_apod_kernel  crop * scaling_coef (* conj(smaps), summed over coils)
//
// Grid offsets and table indices are computed with explicitly rounded float32 operations, the same
// sequence oracle/nufft.py::_tap_indices_f32 performs, so both read the same table entries.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <math.h>

#include <algorithm>
#include <climits>
#include <initializer_list>
#include <map>
#include <mutex>
#include <vector>

#include "nufft_common.cuh"

namespace pdu {

// ------------------------------------------------------------------ apodise + zero pad
// one thread = two neighbouring grid cells (one 16-byte store); three quarters of the stores are zeros
__global__ void __launch_bounds__(256)
    apod_pad_kernel(const float2* __restrict__ image, const float2* __restrict__ smaps, float4* __restrict__ grid,
                    const float* __restrict__ s0, const float* __restrict__ s1, NufftDims d, int coils, int smaps_batch,
                    long total2) {
    const int k1h = d.k1 >> 1;
    const long plane = (long)d.n0 * d.n1;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total2; i += (long)gridDim.x * blockDim.x) {
        const int c1 = (int)(i % k1h) * 2;
        const long t = i / k1h;
        const int c0 = (int)(t % d.k0);
        const long p = t / d.k0;
        float4 out = make_float4(0.f, 0.f, 0.f, 0.f);
        if (c0 < d.n0 && c1 < d.n1) {
            const long b = p / coils, c = p - b * coils;
            const float w0 = __ldg(s0 + c0);
            float2 v[2];
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                v[e] = make_float2(0.f, 0.f);
                if (c1 + e < d.n1) {
                    const long pix = (long)c0 * d.n1 + c1 + e;
                    if (smaps) {
                        const long sb = smaps_batch == 1 ? 0 : b;
                        v[e] = cmul(__ldg(image + b * plane + pix), __ldg(smaps + (sb * coils + c) * plane + pix));
                    } else {
                        v[e] = __ldg(image + p * plane + pix);
                    }
                    const float w = w0 * __ldg(s1 + c1 + e);
                    v[e].x *= w;
                    v[e].y *= w;
                }
            }
            out = make_float4(v[0].x, v[0].y, v[1].x, v[1].y);
        }
        grid[i] = out;
    }
}

// ------------------------------------------------------------------ crop + apodise (+ coil combine)
__global__ void __launch_bounds__(256)
    crop_apod_kernel(const float2* __restrict__ grid, const float2* __restrict__ smaps, float2* __restrict__ image,
                     const float* __restrict__ s0, const float* __restrict__ s1, NufftDims d, int coils, int smaps_batch,
                     float scale, long total, int split = 0) {
    const long plane = (long)d.n0 * d.n1;
    const long gplane = (long)d.k0 * d.k1;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        const int c1 = (int)(i % d.n1);
        const long t = i / d.n1;
        const int c0 = (int)(t % d.n0);
        const long q = t / d.n0;          // output plane: b (with smaps) or b * coils + c
        const float w = __ldg(s0 + c0) * __ldg(s1 + c1) * scale;
        const long gp = (long)c0 * d.k1 + c1;
        float2 v;
        if (smaps) {
            const long sb = smaps_batch == 1 ? 0 : q;
            // coils in groups of four: eight independent loads in flight per thread (the serial loop was
            // latency bound: ncu long-scoreboard 19 cycles per issue)
            float2 acc = make_float2(0.f, 0.f);
            const float2* gq = grid + q * coils * gplane + gp;
            const float2* sq = smaps + sb * coils * plane + (long)c0 * d.n1 + c1;
            int c = 0;
            for (; c + 4 <= coils; c += 4) {
                float2 gv[4], sv[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    gv[u] = __ldg(gq + (c + u) * gplane);
                    sv[u] = __ldg(sq + (c + u) * plane);
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const float2 z = cmul_conj(gv[u], sv[u]);
                    acc.x += z.x;
                    acc.y += z.y;
                }
            }
            for (; c < coils; ++c) {
                const float2 z = cmul_conj(__ldg(gq + c * gplane), __ldg(sq + c * plane));
                acc.x += z.x;
                acc.y += z.y;
            }
            v = acc;
        } else {
            v = __ldg(grid + q * gplane + gp);
        }
        if (split) {              // [planes][2][n0][n1] float32: real plane, imaginary plane
            float* o = reinterpret_cast<float*>(image) + 2 * q * plane + (long)c0 * d.n1 + c1;
            o[0] = v.x * w;
            o[plane] = v.y * w;
        } else {
            image[i] = make_float2(v.x * w, v.y * w);
        }
    }
}

// ------------------------------------------------------------------ crop + apodise, coil-map gradient (SmapsGrad)
// the sibling of crop_apod_kernel for the gradient of the coil maps: the same per-plane grid (or cropped planes U), but
// summed over the batch elements sharing a map instead of over the coils, each times conj(q[b]); b in increasing order
__device__ __forceinline__ float2 sg_q(const float* q, int q_split, long b, long plane, long pix) {
    if (q_split) return make_float2(__ldg(q + 2 * b * plane + pix), __ldg(q + (2 * b + 1) * plane + pix));
    return __ldg(reinterpret_cast<const float2*>(q) + b * plane + pix);
}

__global__ void __launch_bounds__(256)
    smaps_grad_kernel(const float2* __restrict__ grid, const float* __restrict__ q, float2* __restrict__ gs,
                      const float* __restrict__ s0, const float* __restrict__ s1, NufftDims d, int coils, int batch,
                      int per_batch, int q_split, int accumulate, float scale, long total) {
    const long plane = (long)d.n0 * d.n1;
    const long gplane = (long)d.k0 * d.k1;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        const int c1 = (int)(i % d.n1);
        const long t = i / d.n1;
        const int c0 = (int)(t % d.n0);
        const long o = t / d.n0;          // gs plane: s * coils + c
        const long s = o / coils, c = o - s * coils;
        const long b_lo = per_batch ? s : 0, b_hi = per_batch ? s + 1 : batch;
        const float w = __ldg(s0 + c0) * __ldg(s1 + c1) * scale;
        const long pix = (long)c0 * d.n1 + c1;
        const float2* gc = grid + c * gplane + (long)c0 * d.k1 + c1;     // plane b * coils + c
        float2 acc = make_float2(0.f, 0.f);
        long b = b_lo;
        for (; b + 4 <= b_hi; b += 4) {   // four batch elements' loads in flight, added in order
            float2 gv[4], qv[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                gv[u] = __ldg(gc + (b + u) * coils * gplane);
                qv[u] = sg_q(q, q_split, b + u, plane, pix);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const float2 z = cmul_conj(gv[u], qv[u]);
                acc.x += z.x;
                acc.y += z.y;
            }
        }
        for (; b < b_hi; ++b) {
            const float2 z = cmul_conj(__ldg(gc + b * coils * gplane), sg_q(q, q_split, b, plane, pix));
            acc.x += z.x;
            acc.y += z.y;
        }
        float2 v = make_float2(acc.x * w, acc.y * w);
        if (accumulate) {
            const float2 old = gs[i];
            v.x += old.x;
            v.y += old.y;
        }
        gs[i] = v;
    }
}

// ------------------------------------------------------------------ interpolation (gather)
// thread = one sample m; loops over the PC planes of its plane chunk (blockIdx.y)
template <int JT>
__global__ void __launch_bounds__(128)    // (r02: capping at 64 registers for 32 warps / SM spills and is not faster)
    interp_fwd_kernel(const float2* __restrict__ grid, float2* __restrict__ kdata, const float* __restrict__ omega,
                      const float2* __restrict__ t0, const float2* __restrict__ t1, NufftDims d, int planes, int pc,
                      long M, float scale) {
    const long m = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= M) return;
    const int J = JT > 0 ? JT : d.J;
    constexpr int N = JT > 0 ? JT : MAXJ;
    const float om0 = __ldg(omega + m), om1 = __ldg(omega + M + m);
    int g0[N], g1[N];
    float2 c0[N], c1[N];
    axis_taps<JT>(om0, d.gam0, d.k0, d.J, d.L, t0, g0, c0);
    axis_taps<JT>(om1, d.gam1, d.k1, d.J, d.L, t1, g1, c1);
    float2 ph = shift_phase(om0, om1, d.shift0, d.shift1);
    ph.x *= scale;
    ph.y *= scale;
    const long gplane = (long)d.k0 * d.k1;
    const int p_end = min(planes, ((int)blockIdx.y + 1) * pc);
    for (int p = blockIdx.y * pc; p < p_end; ++p) {
        const float2* gp = grid + p * gplane;
        float2 acc = make_float2(0.f, 0.f);
#pragma unroll
        for (int a = 0; a < N; ++a) {
            if (a < J) {
                const float2* row = gp + (long)g0[a] * d.k1;
                float2 racc = make_float2(0.f, 0.f);
#pragma unroll
                for (int b = 0; b < N; ++b) {
                    if (b < J) {
                        const float2 z = cmul(__ldg(row + g1[b]), c1[b]);
                        racc.x += z.x;
                        racc.y += z.y;
                    }
                }
                const float2 z = cmul(racc, c0[a]);
                acc.x += z.x;
                acc.y += z.y;
            }
        }
        kdata[(long)p * M + m] = cmul(acc, ph);
    }
}

// ------------------------------------------------------------------ interpolation adjoint (scatter)
template <int JT>
__global__ void __launch_bounds__(128)
    interp_adj_kernel(const float2* __restrict__ kdata, float2* __restrict__ grid, const float* __restrict__ omega,
                      const float2* __restrict__ t0, const float2* __restrict__ t1, NufftDims d, int planes, int pc,
                      long M) {
    const long m = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= M) return;
    const int J = JT > 0 ? JT : d.J;
    constexpr int N = JT > 0 ? JT : MAXJ;
    const float om0 = __ldg(omega + m), om1 = __ldg(omega + M + m);
    int g0[N], g1[N];
    float2 c0[N], c1[N];
    axis_taps<JT>(om0, d.gam0, d.k0, d.J, d.L, t0, g0, c0);
    axis_taps<JT>(om1, d.gam1, d.k1, d.J, d.L, t1, g1, c1);
    const float2 ph = shift_phase(om0, om1, d.shift0, d.shift1);
    const long gplane = (long)d.k0 * d.k1;
    const int p_end = min(planes, ((int)blockIdx.y + 1) * pc);
    for (int p = blockIdx.y * pc; p < p_end; ++p) {
        const float2 y = cmul_conj(__ldg(kdata + (long)p * M + m), ph);
        float2* gp = grid + p * gplane;
#pragma unroll
        for (int a = 0; a < N; ++a) {
            if (a < J) {
                const float2 ya = cmul_conj(y, c0[a]);
                float2* row = gp + (long)g0[a] * d.k1;
#pragma unroll
                for (int b = 0; b < N; ++b) {
                    if (b < J) atomicAdd(row + g1[b], cmul_conj(ya, c1[b]));
                }
            }
        }
    }
}

static unsigned stream_grid(long items) {
    const long want = cdiv(items, 256);
    const long cap = (long)sm_count() * 16;
    return (unsigned)(want < 1 ? 1 : (want < cap ? want : cap));
}

static int plane_chunk(int planes, long M) {
    // enough CTAs for two waves when the problem allows it, otherwise reuse the taps across planes
    // one plane per thread until there are more than ~16 CTAs per SM slot (measured: the gather is latency
    // bound, 2.7 us / plane at 4 planes per thread against 1.9 us at 1)
    const long ctas_m = cdiv(M, 128);
    int pc = 1;
    while (pc < planes && ctas_m * cdiv(planes, pc) > 16L * 16 * sm_count()) pc *= 2;
    return pc;
}

// The cuFFT handle of a plan is shared state (stream binding, work area): the plan's mutex is held from the
// cufftSetStream to the end of the exec call, so two host threads that share a plan cannot retarget each other's
// transform.  (Kernels of one handle still run in the order they were enqueued; use one plan per stream for overlap.)
static int run_fft(pdu_nufft_plan* p, float2* grid, int planes, int dir, cudaStream_t st) {
    std::lock_guard<std::mutex> lock(p->mu);
    auto it = p->fft.find(planes);
    if (it == p->fft.end()) {
        cufftHandle h;
        int n[2] = {p->k0, p->k1};
        cufftResult r = cufftPlanMany(&h, 2, n, nullptr, 1, 0, nullptr, 1, 0, CUFFT_C2C, planes);
        if (r != CUFFT_SUCCESS) {
            set_error("cufftPlanMany(%d x %d, batch %d) failed with %d", p->k0, p->k1, planes, (int)r);
            return PDU_EFFT;
        }
        it = p->fft.emplace(planes, h).first;
    }
    cufftResult r = cufftSetStream(it->second, st);
    if (r != CUFFT_SUCCESS) {
        set_error("cufftSetStream failed with %d", (int)r);
        return PDU_EFFT;
    }
    r = cufftExecC2C(it->second, (cufftComplex*)grid, (cufftComplex*)grid, dir);
    if (r != CUFFT_SUCCESS) {
        set_error("cufftExecC2C failed with %d", (int)r);
        return PDU_EFFT;
    }
    count_launch(2);   // a 2-D C2C transform is at least two library kernels
    return PDU_OK;
}

static int launch_interp_fwd(pdu_nufft_plan* p, const float2* grid, float2* kdata, const float* omega, int planes,
                             long M, float scale, cudaStream_t st) {
    const int pc = plane_chunk(planes, M);
    dim3 g((unsigned)cdiv(M, 128), (unsigned)cdiv(planes, pc));
    if (p->J == 6) interp_fwd_kernel<6><<<g, 128, 0, st>>>(grid, kdata, omega, p->d_t0, p->d_t1, dims_of(p), planes, pc, M, scale);
    else interp_fwd_kernel<0><<<g, 128, 0, st>>>(grid, kdata, omega, p->d_t0, p->d_t1, dims_of(p), planes, pc, M, scale);
    PDU_LAUNCHED();
    return PDU_OK;
}

static int launch_interp_adj(pdu_nufft_plan* p, const float2* kdata, float2* grid, const float* omega, int planes,
                             long M, cudaStream_t st) {
    const int pc = plane_chunk(planes, M);
    dim3 g((unsigned)cdiv(M, 128), (unsigned)cdiv(planes, pc));
    if (p->J == 6) interp_adj_kernel<6><<<g, 128, 0, st>>>(kdata, grid, omega, p->d_t0, p->d_t1, dims_of(p), planes, pc, M);
    else interp_adj_kernel<0><<<g, 128, 0, st>>>(kdata, grid, omega, p->d_t0, p->d_t1, dims_of(p), planes, pc, M);
    PDU_LAUNCHED();
    return PDU_OK;
}

// ------------------------------------------------------------------ pruned FFT passes (pfft.cuh)
template <typename T>
__device__ __forceinline__ T* pf_smem() {
    extern __shared__ __align__(16) unsigned char pf_dyn[];
    return reinterpret_cast<T*>(pf_dyn);
}

// forward, along the last axis: SEQ image rows of one plane -> T [planes][n0][k1]
template <int SEQ>
__global__ void __launch_bounds__(256)
    pfft_rows_fwd_kernel(const float2* __restrict__ image, const float2* __restrict__ smaps, float2* __restrict__ T,
                         const float* __restrict__ s0, const float* __restrict__ s1, const float2* __restrict__ tw_g,
                         PfftPlan pl, NufftDims d, int coils, int smaps_batch, int pitch) {
    float2* buf0 = pf_smem<float2>();
    float2* buf1 = buf0 + SEQ * pitch;
    float2* tw = buf1 + SEQ * pitch;
    const int tid = threadIdx.x, K = pl.K;
    const long p = blockIdx.y;
    const int r0 = blockIdx.x * SEQ;
    for (int i = tid; i < K; i += blockDim.x) tw[i] = __ldg(tw_g + i);
    const long plane = (long)d.n0 * d.n1;
    const long b = p / coils, c = p - b * coils;
    const int tps = blockDim.x / SEQ, s = tid / tps, row = r0 + s;      // a fixed row per thread: no run-time division below
    for (int col = tid - s * tps; col < K; col += tps) {
        float2 v = make_float2(0.f, 0.f);
        if (row < d.n0 && col < d.n1) {
            const long pix = (long)row * d.n1 + col;
            if (smaps) {
                const long sb = smaps_batch == 1 ? 0 : b;
                v = cmul(__ldg(image + b * plane + pix), __ldg(smaps + (sb * coils + c) * plane + pix));
            } else {
                v = __ldg(image + p * plane + pix);
            }
            const float w = __ldg(s0 + row) * __ldg(s1 + col);
            v.x *= w;
            v.y *= w;
        }
        buf0[s * pitch + pf_pos(col)] = v;
    }
    __syncthreads();
    const float2* res = pf_transform<false>(buf0, buf1, tw, pl, SEQ, pitch, tid, blockDim.x);
    if (row < d.n0)
        for (int col = tid - s * tps; col < K; col += tps) T[(p * d.n0 + row) * K + col] = res[s * pitch + pf_pos(col)];
}

// forward, along the first axis: SEQ neighbouring columns of T [planes][n0][k1] -> grid [planes][k0][k1]
template <int SEQ>
__global__ void __launch_bounds__(256)
    pfft_cols_fwd_kernel(const float2* __restrict__ T, float2* __restrict__ grid, const float2* __restrict__ tw_g, PfftPlan pl,
                         NufftDims d, int pitch) {
    float2* buf0 = pf_smem<float2>();
    float2* buf1 = buf0 + SEQ * pitch;
    float2* tw = buf1 + SEQ * pitch;
    const int tid = threadIdx.x, K = pl.K;           // K == k0
    const long p = blockIdx.y;
    const int c0 = blockIdx.x * SEQ;
    for (int i = tid; i < K; i += blockDim.x) tw[i] = __ldg(tw_g + i);
    for (int i = tid; i < SEQ * K; i += blockDim.x) {
        const int row = i / SEQ, s = i - row * SEQ, col = c0 + s;
        float2 v = make_float2(0.f, 0.f);
        if (row < d.n0 && col < d.k1) v = __ldg(T + (p * d.n0 + row) * d.k1 + col);
        buf0[s * pitch + pf_pos(row)] = v;
    }
    __syncthreads();
    const float2* res = pf_transform<false>(buf0, buf1, tw, pl, SEQ, pitch, tid, blockDim.x);
    for (int i = tid; i < SEQ * K; i += blockDim.x) {
        const int row = i / SEQ, s = i - row * SEQ, col = c0 + s;
        if (col < d.k1) grid[(p * K + row) * d.k1 + col] = res[s * pitch + pf_pos(row)];
    }
}

// adjoint (unnormalised inverse), along the last axis: SEQ grid rows -> T [planes][k0][n1] (first n1 outputs kept)
template <int SEQ>
__global__ void __launch_bounds__(256)
    pfft_rows_adj_kernel(const float2* __restrict__ grid, float2* __restrict__ T, const float2* __restrict__ tw_g, PfftPlan pl,
                         NufftDims d, int pitch) {
    float2* buf0 = pf_smem<float2>();
    float2* buf1 = buf0 + SEQ * pitch;
    float2* tw = buf1 + SEQ * pitch;
    const int tid = threadIdx.x, K = pl.K;           // K == k1
    const long p = blockIdx.y;
    const int r0 = blockIdx.x * SEQ;
    for (int i = tid; i < K; i += blockDim.x) tw[i] = __ldg(tw_g + i);
    const int tps = blockDim.x / SEQ, s = tid / tps, row = r0 + s;
    for (int col = tid - s * tps; col < K; col += tps)
        buf0[s * pitch + pf_pos(col)] = row < d.k0 ? __ldg(grid + (p * d.k0 + row) * K + col) : make_float2(0.f, 0.f);
    __syncthreads();
    const float2* res = pf_transform<true>(buf0, buf1, tw, pl, SEQ, pitch, tid, blockDim.x);
    if (row < d.k0)
        for (int col = tid - s * tps; col < d.n1; col += tps) T[(p * d.k0 + row) * d.n1 + col] = res[s * pitch + pf_pos(col)];
}

// adjoint, along the first axis: SEQ neighbouring columns of T [planes][k0][n1] -> U [planes][n0][n1]
template <int SEQ>
__global__ void __launch_bounds__(256)
    pfft_cols_adj_kernel(const float2* __restrict__ T, float2* __restrict__ U, const float2* __restrict__ tw_g, PfftPlan pl,
                         NufftDims d, int pitch) {
    float2* buf0 = pf_smem<float2>();
    float2* buf1 = buf0 + SEQ * pitch;
    float2* tw = buf1 + SEQ * pitch;
    const int tid = threadIdx.x, K = pl.K;           // K == k0
    const long p = blockIdx.y;
    const int c0 = blockIdx.x * SEQ;
    for (int i = tid; i < K; i += blockDim.x) tw[i] = __ldg(tw_g + i);
    for (int i = tid; i < SEQ * K; i += blockDim.x) {
        const int row = i / SEQ, s = i - row * SEQ, col = c0 + s;
        buf0[s * pitch + pf_pos(row)] = col < d.n1 ? __ldg(T + (p * K + row) * d.n1 + col) : make_float2(0.f, 0.f);
    }
    __syncthreads();
    const float2* res = pf_transform<true>(buf0, buf1, tw, pl, SEQ, pitch, tid, blockDim.x);
    for (int i = tid; i < SEQ * d.n0; i += blockDim.x) {
        const int row = i / SEQ, s = i - row * SEQ, col = c0 + s;
        if (col < d.n1) U[(p * d.n0 + row) * d.n1 + col] = res[s * pitch + pf_pos(row)];
    }
}

// ------------------------------------------------------------------ register-resident pruned FFT (pfft_fast.cuh)
// Same four passes as above for K = 512 / 640 (grid = 2 x image).  Row kernels: thread = (row s, butterfly t),
// consecutive threads along the row; column kernels: consecutive threads across the SEQ neighbouring columns so
// that a warp touches whole 64-byte runs of every grid row.
// These kernels run only for grid == 2 x image (ff_supported): N = K / 2 is a compile-time constant, every element
// address is base(thread) + r * constant.
template <int K, int SEQ>
__global__ void __launch_bounds__(SEQ* FastFft<K>::TPS)
    ff_rows_fwd_kernel(const float2* __restrict__ image, const float2* __restrict__ smaps, float2* __restrict__ T,
                       const float* __restrict__ s0, const float* __restrict__ s1, const float2* __restrict__ tw_g, NufftDims d,
                       int coils, int smaps_batch) {
    using F = FastFft<K>;
    constexpr int N = K / 2, TPS = F::TPS, NS3 = F::NS3;
    float2* buf = pf_smem<float2>();
    float2* tw = buf + SEQ * F::template pitch<4>();
    const int tid = threadIdx.x, s = tid / TPS, t = tid - s * TPS;
    const int p = blockIdx.y;
    const int row = blockIdx.x * SEQ + s;
    for (int i = tid; i < K; i += SEQ * TPS) tw[i] = __ldg(tw_g + i);
    const int b = p / coils, c = p - b * coils;
    const bool live = row < N;
    const float w0 = live ? __ldg(s0 + row) : 0.f;
    const float2* src = image + ((long)(smaps ? b : p) * N + row) * N + t;
    const float2* sm = smaps ? smaps + ((long)((smaps_batch == 1 ? 0 : b) * coils + c) * N + row) * N + t : nullptr;
    const float* s1t = s1 + t;
    auto ld = [&](int r) {                     // element t + r TPS < N
        if (!live) return make_float2(0.f, 0.f);
        float2 v = __ldg(src + r * TPS);
        if (sm) v = cmul(v, __ldg(sm + r * TPS));
        const float w = w0 * __ldg(s1t + r * TPS);
        return make_float2(v.x * w, v.y * w);
    };
    float2* dst = T + ((long)p * N + row) * K;
    auto st = [&](int j, int r, float2 v) {
        if (live) dst[j + r * NS3] = v;
    };
    ff_transform<K, 4, false, true, false, false, false, true>(buf + s * F::template pitch<4>(), tw, t, ld, st);
}

template <int K, int SEQ>
__global__ void __launch_bounds__(SEQ* FastFft<K>::TPS, K <= 640 ? 3 : 1)
    ff_cols_fwd_kernel(const float2* __restrict__ T, float2* __restrict__ grid, const float2* __restrict__ tw_g, NufftDims d) {
    using F = FastFft<K>;
    constexpr int N = K / 2, TPS = F::TPS, NS3 = F::NS3;
    float2* buf = pf_smem<float2>();
    float2* tw = buf + SEQ * F::template pitch<3>();
    const int tid = threadIdx.x, t = tid / SEQ, s = tid - t * SEQ;
    const int p = blockIdx.y;
    const int col = blockIdx.x * SEQ + s;
    for (int i = tid; i < K; i += SEQ * TPS) tw[i] = __ldg(tw_g + i);
    const bool live = col < K;
    const float2* src = T + ((long)p * N + t) * K + col;
    float2* dst = grid + (long)p * K * K + col;
    auto ld = [&](int r) { return live ? __ldcs(src + r * (TPS * K)) : make_float2(0.f, 0.f); };
    auto st = [&](int j, int r, float2 v) {
        if (live) __stcs(dst + j * K + r * (NS3 * K), v);
    };
    ff_transform<K, 3, false, true, false>(buf + s * F::template pitch<3>(), tw, t, ld, st);
}

template <int K, int SEQ>
__global__ void __launch_bounds__(SEQ* FastFft<K>::TPS)
    ff_rows_adj_kernel(const float2* __restrict__ grid, float2* __restrict__ T, const float2* __restrict__ tw_g, NufftDims d) {
    using F = FastFft<K>;
    constexpr int N = K / 2, TPS = F::TPS, NS3 = F::NS3;
    float2* buf = pf_smem<float2>();
    float2* tw = buf + SEQ * F::template pitch<4>();
    const int tid = threadIdx.x, s = tid / TPS, t = tid - s * TPS;
    const int p = blockIdx.y;
    const int row = blockIdx.x * SEQ + s;
    for (int i = tid; i < K; i += SEQ * TPS) tw[i] = __ldg(tw_g + i);
    const bool live = row < K;
    const float2* src = grid + ((long)p * K + row) * K + t;
    float2* dst = T + ((long)p * K + row) * N;
    auto ld = [&](int r) { return live ? __ldcs(src + r * TPS) : make_float2(0.f, 0.f); };
    auto st = [&](int j, int r, float2 v) {
        if (live) __stcs(dst + j + r * NS3, v);
    };
    ff_transform<K, 4, true, false, true, false, false, true>(buf + s * F::template pitch<4>(), tw, t, ld, st);
}

// The row pass on the COMPACT gridded samples (interp_adj_csrT_kernel<.., true>): a thread looks up the compact index of
// each of its eight inputs (nz_idx, 4 bytes per cell, coalesced and L2 resident) and loads the value only where the cell
// is non-empty.  Against the dense form the gather writes and this pass reads one value per non-empty cell instead of K
// per row.  Branch-free: an empty cell reads the plane's first value (one shared sector) and discards it, so that the
// eight indices and then the eight values are in flight together -- with a branch per input the loads went out one at
// a time (95 us for this pass at 64 planes of 640^2).  Other forms measured there: the non-empty cells spread over a
// zeroed shared-memory row and the transform started from it (three more CTA barriers: 86 us against 72 for the dense
// pass in spite of 94 instead of 210 MB); occupancy words + population count instead of the index array (two loads and
// ~6 more instructions per input: 4 us more for the call; as two separate arrays 12 us more); six CTAs per SM (32
// registers, maximum shared-memory carve-out) instead of four: 4 us more.
template <int K, int SEQ>
__global__ void __launch_bounds__(SEQ* FastFft<K>::TPS)
    ff_rows_adj_compact_kernel(const float2* __restrict__ gridc, float2* __restrict__ T, const float2* __restrict__ tw_g,
                               const int* __restrict__ nz_idx, NufftDims d) {
    using F = FastFft<K>;
    constexpr int N = K / 2, TPS = F::TPS, NS3 = F::NS3;
    float2* buf = pf_smem<float2>();
    float2* tw = buf + SEQ * F::template pitch<4>();
    const int tid = threadIdx.x, s = tid / TPS, t = tid - s * TPS;
    const int p = blockIdx.y;
    const int row = blockIdx.x * SEQ + s;
    for (int i = tid; i < K; i += SEQ * TPS) tw[i] = __ldg(tw_g + i);
    const bool live = row < K;
    const float2* src = gridc + (long)p * K * K;
    float2* dst = T + ((long)p * K + row) * N;
    float2 val[8];
    {
        const int* irow = nz_idx + (long)row * K + t;
        int ix[8];
#pragma unroll
        for (int r = 0; r < 8; ++r) ix[r] = live ? __ldg(irow + r * TPS) : -1;
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            const float2 x = __ldcs(src + (ix[r] >= 0 ? ix[r] : 0));
            val[r] = ix[r] >= 0 ? x : make_float2(0.f, 0.f);
        }
    }
    auto ld = [&](int r) { return val[r]; };
    auto st = [&](int j, int r, float2 v) {
        if (live) __stcs(dst + j + r * NS3, v);
    };
    ff_transform<K, 4, true, false, true, false, false, true>(buf + s * F::template pitch<4>(), tw, t, ld, st);
}

template <int K, int SEQ>
__global__ void __launch_bounds__(SEQ* FastFft<K>::TPS, K <= 640 ? 3 : 1)
    ff_cols_adj_kernel(const float2* __restrict__ T, float2* __restrict__ U, const float2* __restrict__ tw_g, NufftDims d) {
    using F = FastFft<K>;
    constexpr int N = K / 2, TPS = F::TPS, NS3 = F::NS3;
    float2* buf = pf_smem<float2>();
    float2* tw = buf + SEQ * F::template pitch<3>();
    const int tid = threadIdx.x, t = tid / SEQ, s = tid - t * SEQ;
    const int p = blockIdx.y;
    const int col = blockIdx.x * SEQ + s;
    for (int i = tid; i < K; i += SEQ * TPS) tw[i] = __ldg(tw_g + i);
    const bool live = col < N;
    const float2* src = T + ((long)p * K + t) * N + col;
    float2* dst = U + (long)p * N * N + col;
    auto ld = [&](int r) { return live ? __ldcs(src + r * (TPS * N)) : make_float2(0.f, 0.f); };
    auto st = [&](int j, int r, float2 v) {
        if (live) __stcs(dst + j * N + r * (NS3 * N), v);
    };
    ff_transform<K, 3, true, false, true>(buf + s * F::template pitch<3>(), tw, t, ld, st);
}

constexpr int FF_SEQ_ROWS = 4;
template <int K>
static constexpr int ff_seq_cols() { return K <= 1024 ? 8 : 4; }     // SEQ * K / 8 threads <= 1024
template <int K>
static constexpr size_t ff_smem_bytes(int seq) { return ((size_t)seq * FastFft<K>::template pitch<3>() + K) * sizeof(float2); }   // PS = 3 is the larger pitch

static bool ff_supported(const pdu_nufft_plan* p) {
    return p->k0 == p->k1 && p->k0 == 2 * p->n0 && p->k1 == 2 * p->n1 && fast_fft_size(p->k0) && p->d_w0 && p->d_w1;
}

template <int K>
static int ff_forward(pdu_nufft_plan* p, const float2* image, const float2* smaps, float2* T, float2* grid, int planes,
                      int coils, int smaps_batch, cudaStream_t st) {
    const NufftDims d = dims_of(p);
    constexpr int FF_SEQ_COLS = ff_seq_cols<K>();
    auto rows = ff_rows_fwd_kernel<K, FF_SEQ_ROWS>;
    auto cols = ff_cols_fwd_kernel<K, FF_SEQ_COLS>;
    PDU_CUDA((ensure_dyn_smem<ff_rows_fwd_kernel<K, FF_SEQ_ROWS>>((int)ff_smem_bytes<K>(FF_SEQ_ROWS))));
    PDU_CUDA((ensure_dyn_smem<ff_cols_fwd_kernel<K, FF_SEQ_COLS>>((int)ff_smem_bytes<K>(FF_SEQ_COLS))));
    rows<<<dim3((unsigned)cdiv(p->n0, FF_SEQ_ROWS), (unsigned)planes), FF_SEQ_ROWS * FastFft<K>::TPS, ff_smem_bytes<K>(FF_SEQ_ROWS), st>>>(
        image, smaps, T, p->d_s0, p->d_s1, p->d_w1, d, coils, smaps_batch);
    PDU_LAUNCHED();
    cols<<<dim3((unsigned)cdiv(p->k1, FF_SEQ_COLS), (unsigned)planes), FF_SEQ_COLS * FastFft<K>::TPS, ff_smem_bytes<K>(FF_SEQ_COLS), st>>>(
        T, grid, p->d_w0, d);
    PDU_LAUNCHED();
    return PDU_OK;
}

// nz_idx: the compact form of the gridded samples (CsrView), nullptr for dense K x K planes
template <int K>
static int ff_adjoint(pdu_nufft_plan* p, const float2* grid, float2* T, float2* U, int planes, cudaStream_t st,
                      const int* nz_idx = nullptr) {
    const NufftDims d = dims_of(p);
    constexpr int FF_SEQ_COLS = ff_seq_cols<K>();
    auto rows = ff_rows_adj_kernel<K, FF_SEQ_ROWS>;
    auto rows_c = ff_rows_adj_compact_kernel<K, FF_SEQ_ROWS>;
    auto cols = ff_cols_adj_kernel<K, FF_SEQ_COLS>;
    PDU_CUDA((ensure_dyn_smem<ff_rows_adj_kernel<K, FF_SEQ_ROWS>>((int)ff_smem_bytes<K>(FF_SEQ_ROWS))));
    PDU_CUDA((ensure_dyn_smem<ff_rows_adj_compact_kernel<K, FF_SEQ_ROWS>>((int)ff_smem_bytes<K>(FF_SEQ_ROWS))));
    PDU_CUDA((ensure_dyn_smem<ff_cols_adj_kernel<K, FF_SEQ_COLS>>((int)ff_smem_bytes<K>(FF_SEQ_COLS))));
    const dim3 gr((unsigned)cdiv(p->k0, FF_SEQ_ROWS), (unsigned)planes);
    if (nz_idx) rows_c<<<gr, FF_SEQ_ROWS * FastFft<K>::TPS, ff_smem_bytes<K>(FF_SEQ_ROWS), st>>>(grid, T, p->d_w1, nz_idx, d);
    else rows<<<gr, FF_SEQ_ROWS * FastFft<K>::TPS, ff_smem_bytes<K>(FF_SEQ_ROWS), st>>>(grid, T, p->d_w1, d);
    PDU_LAUNCHED();
    cols<<<dim3((unsigned)cdiv(p->n1, FF_SEQ_COLS), (unsigned)planes), FF_SEQ_COLS * FastFft<K>::TPS, ff_smem_bytes<K>(FF_SEQ_COLS), st>>>(
        T, U, p->d_w0, d);
    PDU_LAUNCHED();
    return PDU_OK;
}

constexpr int PF_SEQ_ROWS = 4, PF_SEQ_COLS = 8;

static size_t pf_smem_bytes(int seq, int K) { return ((size_t)2 * seq * pfft_pitch(K) + K) * sizeof(float2); }

template <typename Kern>
static int pf_set_smem(Kern kern, size_t bytes) {
    PDU_REQUIRE(bytes <= 200 * 1024, "pruned FFT: %zu bytes of shared memory needed (grid too large)", bytes);
    PDU_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    return PDU_OK;
}

// ------------------------------------------------------------------ adjoint interpolation as a sorted gather
// The atomic scatter above sits on the L2 atomic unit's rate (measured 0.23 T float2 atomics/s on B200
// whatever the occupancy), and its summation order changes from run to run.  For a trajectory that is
// used more than once -- every unrolled iteration, every DCF iteration, every training step -- the
// adjoint interpolator is built once as a sparse matrix in CSR form (one row per grid cell: the samples
// that touch it and their conjugated Kaiser-Bessel weights, phase included), sorted by cell with a
// stable radix sort, and applied as a gather: no atomics, no memset, bit-reproducible.
//   csr buffer:  row_ptr int32[cells + 1] | samp int32[n] | w float2[n] | build scratch      (n = M J^2)
// Rows with more entries than this are summed by a whole warp (lanes stride the entries: coalesced index and weight
// loads).  A bound that follows the trajectory's average, 4 x entries per cell, so that dense trajectories keep their
// cells on the lane-group loop, was measured and lost (128^2 x 256 spokes, 8 planes: 218 against 159 us): the warp form
// is the better one for every row of 32 entries or more; what dense trajectories need is enough warp-per-row CTAs.
static int csr_long_threshold(const pdu_nufft_plan*, long) { return 32; }

struct CsrView {
    int* row_ptr;
    int* n_long;       // [1] number of long rows
    int* long_rows;    // [cells] their indices in nz_cell (first n_long valid)
    int* nz_cell;      // [cells] the non-empty cells in increasing order (first nz_ptr[k0] valid)
    int* nz_ptr;       // [k0 + 1] grid row r owns nz_cell[nz_ptr[r] .. nz_ptr[r + 1])
    int* nz_idx;       // [cells] compact index of a non-empty cell, -1 for an empty one
    int* nz_rptr;      // [cells + 1] row_ptr of the non-empty cells: entries of compact cell i are [nz_rptr[i], nz_rptr[i + 1])
    int* samp;
    float2* w;
    // build scratch
    unsigned* key_in;
    unsigned* id_in;
    unsigned* key_out;
    unsigned* id_out;
    float2* w_unsorted;
    int* rank;         // [cells + 1] number of non-empty cells before cell c
    void* cub_tmp;
    size_t cub_bytes;
    size_t total;
};

static CsrView csr_layout(const pdu_nufft_plan* p, long M, void* base, bool with_scratch = true) {
    const size_t n = (size_t)M * p->J * p->J, cells = (size_t)p->k0 * p->k1;
    CsrView v;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += align256(bytes); return (char*)base + o; };
    v.row_ptr = (int*)take((cells + 1) * 4);
    v.n_long = (int*)take(4);
    v.long_rows = (int*)take(cells * 4);
    v.nz_cell = (int*)take(cells * 4);
    v.nz_ptr = (int*)take(((size_t)p->k0 + 1) * 4);
    v.nz_idx = (int*)take(cells * 4);
    v.nz_rptr = (int*)take((cells + 1) * 4);
    v.samp = (int*)take(n * 4);
    v.w = (float2*)take(n * 8);
    v.key_in = (unsigned*)take(n * 4);
    v.id_in = (unsigned*)take(n * 4);
    v.key_out = (unsigned*)take(n * 4);
    v.id_out = (unsigned*)take(n * 4);
    v.w_unsorted = (float2*)take(n * 8);
    v.rank = (int*)take((cells + 1) * 4);
    v.cub_bytes = 0;
    v.cub_tmp = nullptr;
    v.total = off;
    if (!with_scratch) return v;      // applying the matrix only needs the arrays before key_in
    cub::DeviceRadixSort::SortPairs(nullptr, v.cub_bytes, (const unsigned*)nullptr, (unsigned*)nullptr, (const unsigned*)nullptr,
                                    (unsigned*)nullptr, (int)n);
    size_t scan_bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, (const int*)nullptr, (int*)nullptr, (int)(cells + 1));
    if (scan_bytes > v.cub_bytes) v.cub_bytes = scan_bytes;
    v.cub_tmp = take(v.cub_bytes);
    v.total = off;
    return v;
}

// one thread per sample: its J^2 (cell, weight) entries, weight = conj(phase * c0 * c1)
__global__ void __launch_bounds__(128)
    csr_entries_kernel(const float* __restrict__ omega, const float2* __restrict__ t0, const float2* __restrict__ t1,
                       NufftDims d, long M, unsigned* __restrict__ key, unsigned* __restrict__ id, float2* __restrict__ w) {
    const long m = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= M) return;
    const float om0 = __ldg(omega + m), om1 = __ldg(omega + M + m);
    int g0[MAXJ], g1[MAXJ];
    float2 c0[MAXJ], c1[MAXJ];
    axis_taps(om0, d.gam0, d.k0, d.J, d.L, t0, g0, c0);
    axis_taps(om1, d.gam1, d.k1, d.J, d.L, t1, g1, c1);
    const float2 ph = shift_phase(om0, om1, d.shift0, d.shift1);
    const float2 one = make_float2(1.f, 0.f);
    const float2 cph = cmul_conj(one, ph);                       // conj(phase)
    long e = m * d.J * d.J;
#pragma unroll
    for (int a = 0; a < MAXJ; ++a) {
        if (a < d.J) {
            const float2 wa = cmul_conj(cph, c0[a]);            // the same association as the scatter: ((y conj ph) conj c0) conj c1
#pragma unroll
            for (int b = 0; b < MAXJ; ++b) {
                if (b < d.J) {
                    key[e] = (unsigned)(g0[a] * d.k1 + g1[b]);
                    id[e] = (unsigned)e;
                    w[e] = cmul_conj(wa, c1[b]);
                    ++e;
                }
            }
        }
    }
}

__global__ void __launch_bounds__(256)
    csr_finish_kernel(const unsigned* __restrict__ key_sorted, const unsigned* __restrict__ id_sorted,
                      const float2* __restrict__ w_unsorted, int* __restrict__ row_ptr, int* __restrict__ samp,
                      float2* __restrict__ w, long n, long cells, int taps) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const unsigned e = id_sorted[i];
        samp[i] = (int)(e / (unsigned)taps);
        w[i] = w_unsorted[e];
    }
    if (i <= cells) {          // row_ptr[c] = first sorted position whose key is >= c
        long lo = 0, hi = n;
        while (lo < hi) {
            const long mid = (lo + hi) >> 1;
            if ((long)key_sorted[mid] < i) lo = mid + 1; else hi = mid;
        }
        row_ptr[i] = (int)lo;
    }
}

// A sparse trajectory leaves most of the oversampled grid empty (48 radial spokes on 640^2: 61 % of the cells), so the
// NUFFT adjoint keeps the gridded samples COMPACT between the gather and the row pass: one value per non-empty cell, in
// cell order.  flag[c] = 1 for a non-empty cell (c < cells), 0 for c == cells; its exclusive sum is the compact index.
__global__ void __launch_bounds__(256) csr_flag_kernel(const int* __restrict__ row_ptr, int* __restrict__ flag, long cells) {
    const long c = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c <= cells) flag[c] = (c < cells && row_ptr[c + 1] > row_ptr[c]) ? 1 : 0;
}
// the compact list itself, the first compact index of every grid row, and the rows too long for one thread (the k-space
// centre of a radial trajectory collects every spoke) by their compact index
__global__ void __launch_bounds__(256)
    csr_compact_kernel(const int* __restrict__ row_ptr, const int* __restrict__ rank, int* __restrict__ nz_cell,
                       int* __restrict__ nz_ptr, int* __restrict__ nz_idx, int* __restrict__ nz_rptr, int* __restrict__ n_long,
                       int* __restrict__ long_rows, long cells, int k0, int k1, int long_thresh) {
    const long c = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c > cells) return;
    if (c % k1 == 0) nz_ptr[c / k1] = rank[c];          // c == cells: nz_ptr[k0] = the number of non-empty cells
    if (c == cells) {
        nz_rptr[rank[c]] = row_ptr[c];                  // closes the last non-empty cell
        return;
    }
    const int len = row_ptr[c + 1] - row_ptr[c];
    if (len > 0) {
        nz_cell[rank[c]] = (int)c;
        nz_rptr[rank[c]] = row_ptr[c];
    }
    nz_idx[c] = len > 0 ? rank[c] : -1;
    if (len > long_thresh) long_rows[atomicAdd(n_long, 1)] = rank[c];
}

// one thread per grid cell, PG planes per thread (an entry is loaded once for all of them)
template <int PG>
__global__ void __launch_bounds__(256)
    interp_adj_csr_kernel(const float2* __restrict__ kdata, float2* __restrict__ grid, const int* __restrict__ row_ptr,
                          const int* __restrict__ samp, const float2* __restrict__ w, long cells, long M, int planes,
                          int long_thresh) {
    const long c = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cells) return;
    const int p0 = blockIdx.y * PG;
    float2 acc[PG];
#pragma unroll
    for (int q = 0; q < PG; ++q) acc[q] = make_float2(0.f, 0.f);
    const int beg = __ldg(row_ptr + c), end = __ldg(row_ptr + c + 1);
    if (end - beg > long_thresh) return;                  // interp_adj_csr_long_kernel owns this cell
    for (int i = beg; i < end; ++i) {
        const long m = __ldg(samp + i);
        const float2 wi = __ldg(w + i);
#pragma unroll
        for (int q = 0; q < PG; ++q) {
            if (p0 + q < planes) {
                const float2 z = cmul(__ldg(kdata + (long)(p0 + q) * M + m), wi);
                acc[q].x += z.x;
                acc[q].y += z.y;
            }
        }
    }
#pragma unroll
    for (int q = 0; q < PG; ++q)
        if (p0 + q < planes) grid[(long)(p0 + q) * cells + c] = acc[q];
}

// kdata [planes][M] -> kT [M][planes4] (planes4 = planes rounded up to 4, padding zeroed): an entry of the sparse
// matrix then finds the samples of PG neighbouring planes in PG * 8 contiguous bytes (one or two 16-byte loads
// from one sector) instead of PG sectors M * 8 bytes apart
__global__ void __launch_bounds__(256)
    transpose_kdata_kernel(const float2* __restrict__ kdata, float2* __restrict__ kT, long M, int planes, int planes4) {
    __shared__ float2 t[32][33];
    const long m0 = (long)blockIdx.x * 32;
    const int p0 = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += 8) {
        const int pl = p0 + r;
        const long m = m0 + threadIdx.x;
        t[r][threadIdx.x] = (pl < planes && m < M) ? __ldg(kdata + (long)pl * M + m) : make_float2(0.f, 0.f);
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += 8) {
        const long m = m0 + r;
        const int pl = p0 + threadIdx.x;
        if (m < M && pl < planes4) kT[m * planes4 + pl] = t[threadIdx.x][r];
    }
}

// Sorted gather on the plane-interleaved samples.  LPC neighbouring lanes share a cell; a lane owns two planes in each of
// G plane groups 2 LPC apart, i.e. one 16-byte load per entry and group, and the LPC lanes of a cell read LPC * 16
// contiguous bytes: a warp instruction touches 32 / LPC cache lines, only 32 / LPC cells share a warp's trip count, per
// plane a warp writes 32 / LPC neighbouring cells, and an entry's index and weight are loaded once for 2 LPC G planes
// with G independent sample loads in flight.  r01's form -- one thread = one cell x 8 planes = four 16-byte loads, every
// one of them from 32 different lines (ncu: L1 74 % busy at 18 % of the DRAM rate, 40 % warps active) -- against
// (LPC, G), whole adjoint at 64 planes of 640^2, one box: (4, 1) 280, (4, 2) 253, (4, 4) 259, (4, 8) 290, (8, 1) 284,
// (8, 2) 259, (8, 4) 263, (2, 4) 266, (2, 8) 296 us, r01's form with the long rows as a kernel of their own ~ 300;
// two or four neighbouring cells per thread with 16-byte stores lost to the merged loop's divergence (310 / 361 us).
// Entries are summed in the same order per (cell, plane) whatever the shape: bit-identical results.
// The first long_blocks CTAs of every plane group take the long rows (the k-space centre: more than csr_long_threshold entries),
// one warp per row, lanes striding the entries and a fixed-order shuffle tree adding them up, exactly as
// interp_adj_csr_long_kernel does from the planar samples -- inside this launch, and scheduled first, the serial walk
// over a centre cell's ~1700 entries (18 us as a kernel of its own) is hidden behind the short cells.
// COMPACT: one value per NON-EMPTY cell (nz_cell, csr_compact_kernel) at grid[plane * cells + compact index] -- the row
// pass (ff_rows_adj_compact_kernel) spreads them over its shared-memory row; otherwise the dense K x K planes.
template <int LPC, int G, bool COMPACT>
__global__ void __launch_bounds__(256)
    interp_adj_csrT_kernel(const float2* __restrict__ kT, float2* __restrict__ grid, const int* __restrict__ row_ptr,
                           const int* __restrict__ samp, const float2* __restrict__ w, const int* __restrict__ n_long,
                           const int* __restrict__ long_rows, const int* __restrict__ nz_cell, const int* __restrict__ nz_rptr,
                           const int* __restrict__ n_nz, long cells, int planes, int planes4, int long_blocks, int long_thresh) {
    constexpr int CPB = 256 / LPC;
    if ((int)blockIdx.x < long_blocks) {
        constexpr int PG = 2 * LPC * G;                   // planes of this plane group
        const int lane = threadIdx.x & 31, p0 = blockIdx.y * PG;
        const int nl = __ldg(n_long);
        for (int r = blockIdx.x * 8 + (threadIdx.x >> 5); r < nl; r += long_blocks * 8) {
            const int ci = __ldg(long_rows + r);
            const long slot = COMPACT ? (long)ci : (long)__ldg(nz_cell + ci);     // where the cell's value goes inside a plane
            const int beg = __ldg(nz_rptr + ci), end = __ldg(nz_rptr + ci + 1);
            // four planes at a time: eight accumulators, so that this rare path does not set the kernel's register count
#pragma unroll 1
            for (int h = 0; h < PG && p0 + h < planes4; h += 4) {
                float2 acc[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) acc[q] = make_float2(0.f, 0.f);
                for (int i = beg + lane; i < end; i += 32) {
                    const long m = __ldg(samp + i);
                    const float2 wi = __ldg(w + i);
                    const float4* src = reinterpret_cast<const float4*>(kT + m * planes4 + p0 + h);
#pragma unroll
                    for (int q = 0; q < 4; q += 2) {
                        const float4 v = __ldg(src + q / 2);
                        const float2 z0 = cmul(make_float2(v.x, v.y), wi), z1 = cmul(make_float2(v.z, v.w), wi);
                        acc[q].x += z0.x;
                        acc[q].y += z0.y;
                        acc[q + 1].x += z1.x;
                        acc[q + 1].y += z1.y;
                    }
                }
#pragma unroll
                for (int q = 0; q < 4; ++q) {
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) {
                        acc[q].x += __shfl_xor_sync(0xffffffffu, acc[q].x, o);
                        acc[q].y += __shfl_xor_sync(0xffffffffu, acc[q].y, o);
                    }
                    if (lane == 0 && p0 + h + q < planes) grid[(long)(p0 + h + q) * cells + slot] = acc[q];
                }
            }
        }
        return;
    }
    const int sub = threadIdx.x % LPC;
    const long o = (long)(blockIdx.x - long_blocks) * CPB + threadIdx.x / LPC;
    const int p = blockIdx.y * (2 * LPC * G) + 2 * sub;   // first of this lane's planes; the others follow 2 LPC apart
    if (o >= (COMPACT ? (long)__ldg(n_nz) : cells) || p >= planes4) return;
    // compact: the row pointer of the non-empty cells (one load level less than nz_cell -> row_ptr)
    const int* rp = COMPACT ? nz_rptr + o : row_ptr + o;
    const int beg = __ldg(rp), end = __ldg(rp + 1);
    if (end - beg > long_thresh) return;                  // the long-row CTAs own this cell
    float2 a0[G], a1[G];
#pragma unroll
    for (int g = 0; g < G; ++g) a0[g] = a1[g] = make_float2(0.f, 0.f);
    const float2* src = kT + p;
    for (int i = beg; i < end; ++i) {
        const long m = __ldg(samp + i);
        const float2 wi = __ldg(w + i);
        const float4* sp = reinterpret_cast<const float4*>(src + m * planes4);
        float4 v[G];
#pragma unroll
        for (int g = 0; g < G; ++g)
            v[g] = p + g * 2 * LPC < planes4 ? __ldg(sp + g * LPC) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int g = 0; g < G; ++g) {
            const float2 z0 = cmul(make_float2(v[g].x, v[g].y), wi), z1 = cmul(make_float2(v[g].z, v[g].w), wi);
            a0[g].x += z0.x;
            a0[g].y += z0.y;
            a1[g].x += z1.x;
            a1[g].y += z1.y;
        }
    }
#pragma unroll
    for (int g = 0; g < G; ++g) {
        const int pg = p + g * 2 * LPC;
        if (pg < planes) grid[(long)pg * cells + o] = a0[g];
        if (pg + 1 < planes) grid[(long)(pg + 1) * cells + o] = a1[g];
    }
}

// one warp per long row; lanes stride the entries, a fixed-order shuffle tree adds them up (reproducible)
template <int PG>
__global__ void __launch_bounds__(256)
    interp_adj_csr_long_kernel(const float2* __restrict__ kdata, float2* __restrict__ grid, const int* __restrict__ row_ptr,
                               const int* __restrict__ n_long, const int* __restrict__ long_rows, const int* __restrict__ nz_cell,
                               const int* __restrict__ samp, const float2* __restrict__ w, long cells, long M, int planes) {
    const int lane = threadIdx.x & 31;
    const int warps = (gridDim.x * blockDim.x) >> 5;
    const int p0 = blockIdx.y * PG;
    const int nl = __ldg(n_long);
    for (int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < nl; r += warps) {
        const long c = __ldg(nz_cell + __ldg(long_rows + r));
        const int beg = __ldg(row_ptr + c), end = __ldg(row_ptr + c + 1);
        float2 acc[PG];
#pragma unroll
        for (int q = 0; q < PG; ++q) acc[q] = make_float2(0.f, 0.f);
        for (int i = beg + lane; i < end; i += 32) {
            const long m = __ldg(samp + i);
            const float2 wi = __ldg(w + i);
#pragma unroll
            for (int q = 0; q < PG; ++q) {
                if (p0 + q < planes) {
                    const float2 z = cmul(__ldg(kdata + (long)(p0 + q) * M + m), wi);
                    acc[q].x += z.x;
                    acc[q].y += z.y;
                }
            }
        }
#pragma unroll
        for (int q = 0; q < PG; ++q) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                acc[q].x += __shfl_xor_sync(0xffffffffu, acc[q].x, o);
                acc[q].y += __shfl_xor_sync(0xffffffffu, acc[q].y, o);
            }
            if (lane == 0 && p0 + q < planes) grid[(long)(p0 + q) * cells + c] = acc[q];
        }
    }
}

static int csr_build(pdu_nufft_plan* p, const float* omega, long M, void* buf, size_t bytes, cudaStream_t st) {
    const long n = M * p->J * p->J, cells = (long)p->k0 * p->k1;
    PDU_REQUIRE(n < 2147483647L && cells < 2147483647L, "pdu_nufft_csr_build: %ld entries exceed 32-bit indexing", n);
    CsrView v = csr_layout(p, M, buf);
    if (!buf || bytes < v.total || ((uintptr_t)buf & 255)) {
        set_error("pdu_nufft_csr_build: buffer of %zu bytes (256-byte aligned) required, got %zu", v.total, buf ? bytes : (size_t)0);
        return PDU_ENOMEM;
    }
    csr_entries_kernel<<<(unsigned)cdiv(M, 128), 128, 0, st>>>(omega, p->d_t0, p->d_t1, dims_of(p), M, v.key_in, v.id_in,
                                                              v.w_unsorted);
    PDU_LAUNCHED();
    int bits = 1;
    while ((1L << bits) < cells) ++bits;
    PDU_CUDA(cub::DeviceRadixSort::SortPairs(v.cub_tmp, v.cub_bytes, v.key_in, v.key_out, v.id_in, v.id_out, (int)n, 0, bits, st));
    count_launch(4);
    const long work = n > cells + 1 ? n : cells + 1;
    csr_finish_kernel<<<(unsigned)cdiv(work, 256), 256, 0, st>>>(v.key_out, v.id_out, v.w_unsorted, v.row_ptr, v.samp, v.w, n,
                                                                 cells, p->J * p->J);
    PDU_LAUNCHED();
    PDU_CUDA(cudaMemsetAsync(v.n_long, 0, 4, st));
    int* flag = (int*)v.key_out;                        // the sorted keys have been consumed by csr_finish_kernel
    int* flag_buf = n >= cells + 1 ? flag : v.rank;     // (a trajectory with fewer entries than cells: scan in place)
    csr_flag_kernel<<<(unsigned)cdiv(cells + 1, 256), 256, 0, st>>>(v.row_ptr, flag_buf, cells);
    PDU_LAUNCHED();
    PDU_CUDA(cub::DeviceScan::ExclusiveSum(v.cub_tmp, v.cub_bytes, flag_buf, v.rank, (int)(cells + 1), st));
    count_launch(2);
    csr_compact_kernel<<<(unsigned)cdiv(cells + 1, 256), 256, 0, st>>>(v.row_ptr, v.rank, v.nz_cell, v.nz_ptr, v.nz_idx, v.nz_rptr, v.n_long, v.long_rows,
                                                                      cells, p->k0, p->k1, csr_long_threshold(p, M));
    PDU_LAUNCHED();
    return PDU_OK;
}

// kT_scratch (optional): room for M * round_up(planes, 4) float2 -- the plane-interleaved copy of kdata
// compact (with kT_scratch only): see interp_adj_csrT_kernel; *compact is cleared when the dense form was written
static int launch_interp_adj_csr(pdu_nufft_plan* p, const float2* kdata, float2* grid, const void* csr, int planes, long M,
                                 cudaStream_t st, float2* kT_scratch = nullptr, bool* compact = nullptr) {
    const CsrView v = csr_layout(p, M, const_cast<void*>(csr), false);
    const long cells = (long)p->k0 * p->k1;
    constexpr int PG = 4;
    dim3 g((unsigned)cdiv(cells, 256), (unsigned)cdiv(planes, PG));
    if (kT_scratch && planes >= 4) {
        const int planes4 = (planes + 3) & ~3;
        transpose_kdata_kernel<<<dim3((unsigned)cdiv(M, 32), (unsigned)cdiv(planes4, 32)), dim3(32, 8), 0, st>>>(
            kdata, kT_scratch, M, planes, planes4);
        PDU_LAUNCHED();
        const int long_blocks = sm_count();               // 8 warps each, grid-stride over the long rows
        const bool cpt = compact && *compact;
        // compact: the grid is sized for the non-empty cells the trajectory can have at most (min(cells, entries)); threads
        // past the actual count (nz_ptr[k0], on the device) leave at once
        const long slots = cpt ? std::min(cells, M * p->J * p->J) : cells;
#define PDU_CSRT(L, G_)                                                                                                     \
    do {                                                                                                                    \
        const int lt_ = csr_long_threshold(p, M);                                                                           \
        dim3 gt_((unsigned)(long_blocks + cdiv(slots, 256 / L)), (unsigned)cdiv(planes4, 2 * L * G_));                       \
        if (cpt)                                                                                                            \
            interp_adj_csrT_kernel<L, G_, true><<<gt_, 256, 0, st>>>(kT_scratch, grid, v.row_ptr, v.samp, v.w, v.n_long,      \
                                                                    v.long_rows, v.nz_cell, v.nz_rptr, v.nz_ptr + p->k0, cells, \
                                                                    planes, planes4, long_blocks, lt_);                     \
        else                                                                                                                \
            interp_adj_csrT_kernel<L, G_, false><<<gt_, 256, 0, st>>>(kT_scratch, grid, v.row_ptr, v.samp, v.w, v.n_long,     \
                                                                     v.long_rows, v.nz_cell, v.nz_rptr, v.nz_ptr + p->k0, cells,\
                                                                     planes, planes4, long_blocks, lt_);                    \
    } while (0)
        // 16 planes per plane group for sparse trajectories (few entries per cell: the index loads are a large part of the
        // loop) and from 64 planes on; 8 otherwise (measured, 16 / 32 planes: 320^2 x 48 spokes 91 / 151 against 97 / 165 us,
        // 512^2 x 96 226 / 425 against 253 / 485; but 320^2 x 160 spokes 228 / 325 against 184 / 312)
        const double per_cell = (double)M * p->J * p->J / (double)cells;
        // (re-measured in the compact form at 64 planes: (4, 1) 251, (4, 2) 228, (4, 4) 226, (8, 1) 249, (8, 2) 234 us)
        if (planes4 >= 16 && (per_cell <= 5.0 || planes4 >= 64)) PDU_CSRT(4, 2);
        else if (planes4 >= 8) PDU_CSRT(4, 1);
        else PDU_CSRT(2, 1);
#undef PDU_CSRT
        PDU_LAUNCHED();
        return PDU_OK;
    }
    if (compact) *compact = false;
    interp_adj_csr_kernel<PG><<<g, 256, 0, st>>>(kdata, grid, v.row_ptr, v.samp, v.w, cells, M, planes, csr_long_threshold(p, M));
    PDU_LAUNCHED();
    dim3 gl((unsigned)(2 * sm_count()), (unsigned)cdiv(planes, PG));      // 8 warps per CTA, grid-stride over the long rows
    interp_adj_csr_long_kernel<PG><<<gl, 256, 0, st>>>(kdata, grid, v.row_ptr, v.n_long, v.long_rows, v.nz_cell, v.samp, v.w,
                                                       cells, M, planes);
    PDU_LAUNCHED();
    return PDU_OK;
}

// [planes][2][n] float32 (real plane, imaginary plane) <-> [planes][n] complex64: the layout change between the CNN
// side of PD-UNet and the generic (complex64) operator path, one pass, optionally times a real weight per element index
// (density compensation).  The fused path reads and writes the split layout directly and does not need these.
__global__ void __launch_bounds__(256)
    layout_to_complex_kernel(const float* __restrict__ split, float2* __restrict__ out, const float* __restrict__ weight, long n,
                             long total) {
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        const long p = i / n, e = i - p * n;
        const float w = weight ? __ldg(weight + e) : 1.f;
        out[i] = make_float2(w * __ldg(split + (2 * p) * n + e), w * __ldg(split + (2 * p + 1) * n + e));
    }
}
__global__ void __launch_bounds__(256)
    layout_to_split_kernel(const float2* __restrict__ in, float* __restrict__ split, long n, long total) {
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        const long p = i / n, e = i - p * n;
        const float2 v = __ldg(in + i);
        split[(2 * p) * n + e] = v.x;
        split[(2 * p + 1) * n + e] = v.y;
    }
}

int launch_crop_apod(pdu_nufft_plan* p, const float2* U, NufftDims d, const float2* smaps, float2* image, int out_planes,
                     int coils, int smaps_batch, float scale, int split, cudaStream_t st) {
    const long total = (long)out_planes * p->n0 * p->n1;
    crop_apod_kernel<<<stream_grid(total), 256, 0, st>>>(U, smaps, image, p->d_s0, p->d_s1, d, coils, smaps_batch, scale, total,
                                                         split);
    PDU_LAUNCHED();
    return PDU_OK;
}

int launch_smaps_grad(pdu_nufft_plan* p, const float2* U, NufftDims d, int coils, float scale, const SmapsGrad& sg,
                      cudaStream_t st) {
    const long total = (long)(sg.per_batch ? sg.batch : 1) * coils * p->n0 * p->n1;
    smaps_grad_kernel<<<stream_grid(total), 256, 0, st>>>(U, sg.q, sg.gs, p->d_s0, p->d_s1, d, coils, sg.batch, sg.per_batch,
                                                          sg.q_split, sg.accumulate, scale * sg.scale, total);
    PDU_LAUNCHED();
    return PDU_OK;
}

static int check_plan_device(const pdu_nufft_plan* p, const char* who) {
    int dev = -1;
    PDU_CUDA(cudaGetDevice(&dev));
    PDU_REQUIRE(dev == p->device, "%s: plan was created on device %d, current device is %d", who, p->device, dev);
    return PDU_OK;
}

// the argument checks of the NUFFT entry points
static int check_call(const pdu_nufft_plan* p, const void* a, const void* b, const void* omega, int batch, int coils,
                      int smaps_batch, const void* smaps, long m, const char* who) {
    PDU_REQUIRE(p != nullptr, "%s: plan is null", who);
    PDU_REQUIRE(!p->toep, "%s: a Toeplitz plan (pdu_toep_plan_create) has no interpolation tables", who);
    PDU_REQUIRE(a && b && omega, "%s: null pointer", who);
    PDU_REQUIRE(batch > 0 && coils > 0 && m > 0, "%s: batch, coils and m must be > 0", who);
    PDU_REQUIRE((long)batch * coils <= 65535L * 64, "%s: too many planes", who);
    if (smaps) PDU_REQUIRE(smaps_batch == 1 || smaps_batch == batch, "%s: smaps batch must be 1 or batch", who);
    return check_plan_device(p, who);
}

// the argument checks of the pdu_toep_* entry points; ptrs: every pointer the entry point requires is set
static int check_toep_call(const pdu_nufft_plan* p, bool ptrs, int batch, int coils, int kernel_batch, const void* smaps,
                           int smaps_batch, const char* who) {
    PDU_REQUIRE(p != nullptr, "%s: plan is null", who);
    PDU_REQUIRE(p->toep, "%s: not a Toeplitz plan (use pdu_toep_plan_create)", who);
    PDU_REQUIRE(ptrs, "%s: null pointer", who);
    PDU_REQUIRE(batch > 0 && coils > 0 && coils <= 65535, "%s: batch must be > 0 and coils in 1..65535", who);
    PDU_REQUIRE(kernel_batch == 1 || kernel_batch == batch, "%s: kernel batch must be 1 or batch", who);
    if (smaps) PDU_REQUIRE(smaps_batch == 1 || smaps_batch == batch, "%s: smaps batch must be 1 or batch", who);
    return check_plan_device(p, who);
}

// the caller's workspace: at least `need` bytes, 256-byte aligned if `aligned`; `code` when it is not
static int check_workspace(const char* who, const void* ws, size_t bytes, size_t need, bool aligned, int code) {
    if (ws && bytes >= need && !(aligned && ((uintptr_t)ws & 255))) return PDU_OK;
    set_error("%s: workspace of %zu bytes%s required, got %zu", who, need, aligned ? " (256-byte aligned)" : "",
              ws ? bytes : (size_t)0);
    return code;
}

// A call is cut into batch chunks so that the scratch (plane_bytes per plane) stays under 512 MB and a chunk has at most
// plane_cap planes.  Measured on B200: chunking the NUFFT down to L2-resident grids (56 MB) does NOT pay -- cuFFT runs at
// ~3 TB/s either way and the gather / scatter lose parallelism -- so the budget only caps the workspace.  Both callers
// cap a chunk at 65535 planes: their FFT passes launch one grid row per plane (gridDim.y = planes), and on small grids
// (a 16 x 16 image has 8 KB of oversampled grid, an 8 x 8 Toeplitz plane 3.5 KB) the budget alone allows more.
static int batch_chunk(size_t plane_bytes, long plane_cap, int batch, int coils) {
    long planes = (long)(((size_t)512 << 20) / plane_bytes);
    if (planes > plane_cap) planes = plane_cap;
    long cb = planes / coils;
    if (cb < 1) cb = 1;
    return (int)(cb < batch ? cb : batch);
}

// f(b0, nb) for the chunks [b0, b0 + nb) of cb batch elements (the last one shorter), stopping at the first error
template <typename Fn>
static int for_each_chunk(int batch, int cb, Fn&& f) {
    for (int b0 = 0; b0 < batch; b0 += cb) {
        const int rc = f(b0, b0 + cb <= batch ? cb : batch - b0);
        if (rc) return rc;
    }
    return PDU_OK;
}

// ------------------------------------------------------------------ Toeplitz-embedded normal operator (pdu_toep_*)
// T x = crop(ifft2(kernel . fft2(zero_pad_2N(x))))  -- A^H W A of the NUFFT without any interpolation ([RECALL]
// torchkbnufft ToepNufft / calc_toeplitz_kernel).  The kernel is the 2-D DFT of the point-spread function p in
// circulant layout (DESIGN.md section 3.4).

// p_circ [kernels][2 n0][2 n1] from q1 = A^H w (omega) and q2 = A^H w (omega0 negated), both with n_shift 0:
//   q1[a, b] = p[a, b], q2[a, b] = p[-a, b], p[-a, -b] = conj p[a, b] (real weights); the row i0 = n0 and the column
//   i1 = n1 are zero
__global__ void __launch_bounds__(256)
    tz_assemble_kernel(const float2* __restrict__ q1, const float2* __restrict__ q2, float2* __restrict__ out, int n0, int n1,
                       float scale, long total) {
    const int l0 = 2 * n0, l1 = 2 * n1;
    const long plane = (long)n0 * n1;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        const int i1 = (int)(i % l1);
        const long t = i / l1;
        const int i0 = (int)(t % l0);
        const long b = t / l0;
        float2 v = make_float2(0.f, 0.f);
        if (i0 != n0 && i1 != n1) {
            const bool lo0 = i0 < n0, lo1 = i1 < n1;
            const int a0 = lo0 ? i0 : l0 - i0, a1 = lo1 ? i1 : l1 - i1;
            v = __ldg((lo0 == lo1 ? q1 : q2) + b * plane + (long)a0 * n1 + a1);
            if (!lo1) v.y = -v.y;
        }
        out[i] = make_float2(v.x * scale, v.y * scale);
    }
}

// generic path: grid [planes][k0][k1] *= kernel (or its conjugate); plane p uses kernel p / coils (batch element) when
// there is one kernel per batch element
__global__ void __launch_bounds__(256)
    tz_mul_kernel(float2* __restrict__ grid, const float2* __restrict__ kern, long cells, int coils, int kernel_batch, int conj,
                  long total) {
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        const long p = i / cells, c = i - p * cells;
        float2 k = __ldg(kern + (kernel_batch == 1 ? 0 : p / coils) * cells + c);
        if (conj) k.y = -k.y;
        grid[i] = cmul(grid[i], k);
    }
}

// fast path, pass 2: SEQ neighbouring columns of T [planes][N][K] (the row pass's output) per CTA, the layout of
// ff_cols_fwd_kernel.  Per column: forward FFT of the N stored rows (HALF_IN), x kernel column on the way into shared
// memory (ST_BUF), inverse FFT from there (LD_BUF) keeping the first N outputs (HALF_OUT), written back in place -- the
// CTA owns its columns across every row, so no other CTA reads them.
template <int K, int SEQ>
__global__ void __launch_bounds__(SEQ* FastFft<K>::TPS)
    tz_cols_kernel(float2* __restrict__ T, const float2* __restrict__ kern, const float2* __restrict__ tw_g, int coils,
                   int kernel_batch, int conj) {
    using F = FastFft<K>;
    constexpr int N = K / 2, TPS = F::TPS, NS3 = F::NS3, PITCH = F::template pitch<3>();
    float2* buf = pf_smem<float2>();
    float2* tw = buf + SEQ * PITCH;
    const int tid = threadIdx.x, t = tid / SEQ, s = tid - t * SEQ;
    const int p = blockIdx.y;
    const int col = blockIdx.x * SEQ + s;          // K is a multiple of SEQ: every column exists
    for (int i = tid; i < K; i += SEQ * TPS) tw[i] = __ldg(tw_g + i);
    float2* colp = T + (long)p * N * K + col;
    const float2* kc = kern + (long)(kernel_batch == 1 ? 0 : p / coils) * K * K + col;
    float2* seq = buf + s * PITCH;
    {
        const float2* src = colp + (long)t * K;
        auto ld = [&](int r) { return __ldcs(src + r * (TPS * K)); };
        // output element e = j + r NS3 (row frequency) at its padded position pos(j) + r (NS3 + NS3 / 8)
        auto st = [&](int j, int r, float2 v) {
            float2 k = __ldg(kc + (long)(j + r * NS3) * K);
            if (conj) k.y = -k.y;
            seq[(j + (j >> 3)) + r * (NS3 + NS3 / 8)] = cmul(v, k);
        };
        ff_transform<K, 3, false, true, false, false, true>(seq, tw, t, ld, st);
    }
    __syncthreads();                               // every product is in shared memory
    {
        const float2* in = seq + (t + (t >> 3));   // input element t + r TPS at pos(t) + r (TPS + TPS / 8)
        auto ld = [&](int r) { return in[r * (TPS + TPS / 8)]; };
        auto st = [&](int j, int r, float2 v) { __stcs(colp + (long)(j + r * NS3) * K, v); };
        ff_transform<K, 3, true, false, true, true>(seq, tw, t, ld, st);
    }
}

// The conjugate-gradient epilogue of an apply (pdu_toep_cg_c64): q = T p + lam p and, per CTA, the float64 partial of
// Re<p, q> in the slot part[system * gridDim.x + blockIdx.x].  A system is a plane, or a batch element with coil maps;
// its lam is lam[system / lam_div] (lam_div 0: lam[0]; lam null: 0).
struct TzCg {
    const float2* p;          // the apply's input, laid out as its output
    const float* lam;
    int lam_div;
    double* part;
};

__device__ __forceinline__ float cg_lam(const float* lam, int lam_div, int sys) {
    return lam ? __ldg(lam + (lam_div ? sys / lam_div : 0)) : 0.f;
}

// sum of one double per thread over the CTA in a fixed order: a shuffle tree in each warp, then the warps in index
// order; the result is valid in thread 0 (blockDim.x a multiple of 32, `red` 32 doubles of shared memory)
__device__ __forceinline__ double cg_block_sum(double v, double* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
    if (threadIdx.x == 0)
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[w];
    return s;
}

// fast path, pass 3: SEQ rows of one output plane per CTA: pruned inverse row FFT of T's N rows (first N outputs),
// x scale; with coil maps the CTA walks the batch element's coils in a fixed order and sums conj(S_c) T_c in registers
// (bit-reproducible; no cropped intermediate, no crop_apod_kernel pass).  CG: the TzCg epilogue at the output store.
// GS (the coil-map gradient, SmapsGrad): the CTA owns rows of coil c of gs plane blockIdx.y = s * coils + c and walks the
// other axis instead -- the batch elements b sharing that map, in increasing order -- summing T_{b, c} conj(q_b); out
// is gs.
template <int K, int SEQ, bool CG = false, bool GS = false>
__global__ void __launch_bounds__(SEQ* FastFft<K>::TPS)
    tz_rows_out_kernel(const float2* __restrict__ T, const float2* __restrict__ smaps, float2* __restrict__ out,
                       const float2* __restrict__ tw_g, int coils, int smaps_batch, float scale, TzCg cg, SmapsGrad sg) {
    using F = FastFft<K>;
    constexpr int N = K / 2, TPS = F::TPS, NS3 = F::NS3, R3 = F::R3;
    constexpr int PER = TPS >= NS3 ? 1 : NS3 / TPS;     // last-pass butterflies per thread (ff_transform)
    static_assert(PER <= 2, "outputs j = t or t + TPS");
    float2* buf = pf_smem<float2>();
    float2* tw = buf + SEQ * F::template pitch<4>();
    const int tid = threadIdx.x, s = tid / TPS, t = tid - s * TPS;
    const int q = blockIdx.y;                            // batch element (coil maps) or plane
    const int row = blockIdx.x * SEQ + s;
    for (int i = tid; i < K; i += SEQ * TPS) tw[i] = __ldg(tw_g + i);
    const bool live = row < N;
    float2 acc[PER][R3];
#pragma unroll
    for (int i = 0; i < PER; ++i)
#pragma unroll
        for (int r = 0; r < R3; ++r) acc[i][r] = make_float2(0.f, 0.f);
    // GS: the walk runs over b in [b_lo, b_hi) for coil gc, reading q_b's row where the apply reads S_c's
    const int gc = GS ? q % coils : 0;
    const int b_lo = GS ? (sg.per_batch ? q / coils : 0) : 0;
    const int nc = GS ? (sg.per_batch ? b_lo + 1 : sg.batch) : (smaps ? coils : 1);
    const float2* sm = GS ? reinterpret_cast<const float2*>(sg.q) + (long)row * N
                          : (smaps ? smaps + ((long)(smaps_batch == 1 ? 0 : q) * coils * N + row) * N : nullptr);
    for (int c = b_lo; c < nc; ++c) {
        const long p = GS ? (long)c * coils + gc : (smaps ? (long)q * coils + c : q);
        const float2* src = T + (p * N + row) * K + t;
        const float2* smc = sm ? sm + (long)c * N * N : nullptr;
        auto ld = [&](int r) { return live ? __ldcs(src + r * TPS) : make_float2(0.f, 0.f); };
        auto st = [&](int j, int r, float2 v) {
            if (!live) return;
            if (smc) v = cmul_conj(v, __ldg(smc + j + r * NS3));
            if (PER == 1 || j < TPS) {
                acc[0][r].x += v.x;
                acc[0][r].y += v.y;
            } else {
                acc[PER - 1][r].x += v.x;
                acc[PER - 1][r].y += v.y;
            }
        };
        ff_transform<K, 4, true, false, true, false, false, true>(buf + s * F::template pitch<4>(), tw, t, ld, st);
        __syncthreads();                                 // the next coil's pass-1 stores reuse the buffer
    }
    if constexpr (!CG) {
        if (!live) return;
        float2* dst = out + ((long)q * N + row) * N;
#pragma unroll
        for (int i = 0; i < PER; ++i) {
            const int j = t + i * TPS;
            if (j < NS3) {
#pragma unroll
                for (int r = 0; r < R3 / 2; ++r) {
                    float2 v = make_float2(acc[i][r].x * scale, acc[i][r].y * scale);
                    if constexpr (GS) {
                        if (sg.accumulate) {
                            const float2 old = dst[j + r * NS3];
                            v.x += old.x;
                            v.y += old.y;
                        }
                    }
                    dst[j + r * NS3] = v;
                }
            }
        }
    } else {
        __shared__ double red[32];
        const float lam = cg_lam(cg.lam, cg.lam_div, q);
        double dot = 0.0;
        if (live) {
            float2* dst = out + ((long)q * N + row) * N;
            const float2* src = cg.p + ((long)q * N + row) * N;
#pragma unroll
            for (int i = 0; i < PER; ++i) {
                const int j = t + i * TPS;
                if (j < NS3) {
#pragma unroll
                    for (int r = 0; r < R3 / 2; ++r) {
                        const float2 pv = __ldg(src + j + r * NS3);
                        const float2 v = make_float2(fmaf(lam, pv.x, acc[i][r].x * scale), fmaf(lam, pv.y, acc[i][r].y * scale));
                        dst[j + r * NS3] = v;
                        dot = fma((double)pv.x, (double)v.x, dot);
                        dot = fma((double)pv.y, (double)v.y, dot);
                    }
                }
            }
        }
        dot = cg_block_sum(dot, red);
        if (tid == 0) cg.part[(long)q * gridDim.x + blockIdx.x] = dot;
    }
}

// ------------------------------------------------------------------ conjugate gradient on T + lam I (pdu_toep_cg_c64)
// Per system (a plane, or a batch element with coil maps), every launch does the same work whatever the data: the
// scalars live on the device, a frozen system's kernels return early, and nothing is read back to the host.  Each CTA
// of the vector kernels first sums its system's partial slots in a fixed order, derives the same alpha / beta / freeze
// decision as every other CTA of the system, does its share of the vector work and writes its own partial of the next
// reduction.  No atomics: a system's result is bit-identical whatever else is in the batch.
constexpr int CG_THREADS = 256;

// CTAs per system of the vector kernels, and slots of their partial sums: a function of the system size alone, so that
// a system's sums add in the same order however the batch is made up or chunked
static int cg_ctas(long n) { return (int)std::min(std::max(cdiv(cdiv(n, 2), 2 * CG_THREADS), 1L), 256L); }

// 16-byte accesses when n is even and every vector of the call is 16-byte aligned; the element pairs, and so the
// order of every sum, are the same either way
static int cg_v4(long n, std::initializer_list<const void*> ptrs) {
    if (n & 1) return 0;
    for (const void* q : ptrs)
        if (q && ((uintptr_t)q & 15)) return 0;
    return 1;
}

// element pair k of a system's vector: elements 2 k and 2 k + 1 (zero past the end of an odd n)
__device__ __forceinline__ void cg_ld(const float2* v, long k, long n, int v4, float2& a, float2& b) {
    if (v4) {
        const float4 t = reinterpret_cast<const float4*>(v)[k];
        a = make_float2(t.x, t.y);
        b = make_float2(t.z, t.w);
    } else {
        a = v[2 * k];
        b = 2 * k + 1 < n ? v[2 * k + 1] : make_float2(0.f, 0.f);
    }
}
__device__ __forceinline__ void cg_st(float2* v, long k, long n, int v4, float2 a, float2 b) {
    if (v4) {
        reinterpret_cast<float4*>(v)[k] = make_float4(a.x, a.y, b.x, b.y);
    } else {
        v[2 * k] = a;
        if (2 * k + 1 < n) v[2 * k + 1] = b;
    }
}
// acc + Re(conj(a) b), in float64
__device__ __forceinline__ double cg_dot(double acc, float2 a, float2 b) {
    return fma((double)a.y, (double)b.y, fma((double)a.x, (double)b.x, acc));
}
__device__ __forceinline__ float2 cg_axpy(float a, float2 x, float2 y) { return make_float2(fmaf(a, x.x, y.x), fmaf(a, x.y, y.y)); }

// a system's `count` partial slots (written by an earlier kernel) summed in a fixed order by one warp: lane l adds
// slots l, l + 32, ..., then a shuffle tree; every lane gets the result
__device__ __forceinline__ double cg_slots(const double* s, int count) {
    double v = 0.0;
    for (int i = threadIdx.x & 31; i < count; i += 32) v += __ldcg(s + i);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    return __shfl_sync(0xffffffffu, v, 0);
}

// the iteration runs for a system that is not frozen, has rho != 0 and a positive curvature pi = Re<p, (T + lam) p>
__device__ __forceinline__ bool cg_runs(int frozen, double rho, double pi) { return !frozen && rho != 0.0 && pi > 0.0; }

// generic path: q += lam p on the apply's cropped output, and per-CTA partials of Re<p, q> (the fast path does this in
// tz_rows_out_kernel's epilogue).  Grid (cg_ctas(n), systems).
__global__ void __launch_bounds__(CG_THREADS)
    cg_lam_dot_kernel(float2* __restrict__ q, const float2* __restrict__ p, const float* __restrict__ lam, int lam_div,
                      double* __restrict__ part, long n, int v4) {
    __shared__ double red[32];
    const int sys = blockIdx.y;
    const long base = (long)sys * n, pairs = (n + 1) / 2;
    const float l = cg_lam(lam, lam_div, sys);
    double dot = 0.0;
    for (long k = (long)blockIdx.x * CG_THREADS + threadIdx.x; k < pairs; k += (long)gridDim.x * CG_THREADS) {
        float2 p0, p1, q0, q1;
        cg_ld(p + base, k, n, v4, p0, p1);
        cg_ld(q + base, k, n, v4, q0, q1);
        q0 = cg_axpy(l, p0, q0);
        q1 = cg_axpy(l, p1, q1);
        cg_st(q + base, k, n, v4, q0, q1);
        dot = cg_dot(cg_dot(dot, p0, q0), p1, q1);
    }
    dot = cg_block_sum(dot, red);
    if (threadIdx.x == 0) part[(long)sys * gridDim.x + blockIdx.x] = dot;
}

// set-up: x = x0 (zero when x0 is null; untouched when x0 == x), r = b - q (q = (T + lam) x0; r = b when q is null),
// p = r, and per-CTA partials of ||r||^2 and ||b||^2.  Grid (cg_ctas(n), systems).
__global__ void __launch_bounds__(CG_THREADS)
    cg_init_kernel(const float2* __restrict__ b, const float2* x0, float2* x, const float2* __restrict__ q, float2* __restrict__ r,
                   float2* __restrict__ p, double* __restrict__ rr_part, double* __restrict__ bb_part, long n, int v4) {
    __shared__ double red[2][32];
    const int sys = blockIdx.y;
    const long base = (long)sys * n, pairs = (n + 1) / 2;
    double rr = 0.0, bb = 0.0;
    for (long k = (long)blockIdx.x * CG_THREADS + threadIdx.x; k < pairs; k += (long)gridDim.x * CG_THREADS) {
        float2 b0, b1, r0, r1;
        cg_ld(b + base, k, n, v4, b0, b1);
        if (x0 != x) {
            float2 x00 = make_float2(0.f, 0.f), x01 = x00;
            if (x0) cg_ld(x0 + base, k, n, v4, x00, x01);
            cg_st(x + base, k, n, v4, x00, x01);
        }
        r0 = b0;
        r1 = b1;
        if (q) {
            float2 q0, q1;
            cg_ld(q + base, k, n, v4, q0, q1);
            r0 = make_float2(b0.x - q0.x, b0.y - q0.y);
            r1 = make_float2(b1.x - q1.x, b1.y - q1.y);
        }
        cg_st(r + base, k, n, v4, r0, r1);
        cg_st(p + base, k, n, v4, r0, r1);
        rr = cg_dot(cg_dot(rr, r0, r0), r1, r1);
        bb = cg_dot(cg_dot(bb, b0, b0), b1, b1);
    }
    rr = cg_block_sum(rr, red[0]);
    bb = cg_block_sum(bb, red[1]);
    if (threadIdx.x == 0) {
        rr_part[(long)sys * gridDim.x + blockIdx.x] = rr;
        bb_part[(long)sys * gridDim.x + blockIdx.x] = bb;
    }
}

// the scalars of one iteration, by warp 0 of every CTA of a system: pi from the apply's slots; rho and the frozen flag
// from the previous iteration's direction kernel, or on the first iteration (rr_first non-null) rho from the set-up's
// slots with the flag clear
__device__ __forceinline__ void cg_scalars(int sys, const double* pi_part, int pi_slots, const double* rr_first,
                                           const double* rho_in, const int* frz_in, double& pi, double& rho, int& frozen) {
    pi = cg_slots(pi_part + (long)sys * pi_slots, pi_slots);
    rho = rr_first ? cg_slots(rr_first + (long)sys * gridDim.x, gridDim.x) : __ldcg(rho_in + sys);
    frozen = rr_first ? 0 : __ldcg(frz_in + sys);
}

// x += alpha p, r -= alpha q with alpha = rho / pi, and per-CTA partials of the new ||r||^2 (rr_out); a system whose
// iteration does not run (cg_runs) is left as it is.  Grid (cg_ctas(n), systems).
__global__ void __launch_bounds__(CG_THREADS)
    cg_update_kernel(float2* __restrict__ x, float2* __restrict__ r, const float2* __restrict__ p, const float2* __restrict__ q,
                     const double* __restrict__ pi_part, int pi_slots, const double* __restrict__ rr_first,
                     const double* __restrict__ rho_in, const int* __restrict__ frz_in, double* __restrict__ rr_out, long n,
                     int v4) {
    __shared__ double red[32];
    __shared__ double s_alpha;
    __shared__ int s_run;
    const int sys = blockIdx.y;
    if (threadIdx.x < 32) {
        double pi, rho;
        int frozen;
        cg_scalars(sys, pi_part, pi_slots, rr_first, rho_in, frz_in, pi, rho, frozen);
        if (threadIdx.x == 0) {
            s_run = cg_runs(frozen, rho, pi);
            s_alpha = s_run ? rho / pi : 0.0;
        }
    }
    __syncthreads();
    if (!s_run) return;                                  // uniform over the CTA
    const float a = (float)s_alpha;
    const long base = (long)sys * n, pairs = (n + 1) / 2;
    double rr = 0.0;
    for (long k = (long)blockIdx.x * CG_THREADS + threadIdx.x; k < pairs; k += (long)gridDim.x * CG_THREADS) {
        float2 x0, x1, r0, r1, p0, p1, q0, q1;
        cg_ld(p + base, k, n, v4, p0, p1);
        cg_ld(q + base, k, n, v4, q0, q1);
        cg_ld(x + base, k, n, v4, x0, x1);
        cg_ld(r + base, k, n, v4, r0, r1);
        cg_st(x + base, k, n, v4, cg_axpy(a, p0, x0), cg_axpy(a, p1, x1));
        r0 = cg_axpy(-a, q0, r0);
        r1 = cg_axpy(-a, q1, r1);
        cg_st(r + base, k, n, v4, r0, r1);
        rr = cg_dot(cg_dot(rr, r0, r0), r1, r1);
    }
    rr = cg_block_sum(rr, red);
    if (threadIdx.x == 0) rr_out[(long)sys * gridDim.x + blockIdx.x] = rr;
}

// p = r + beta p with beta = rho' / rho, rho' the sum of cg_update_kernel's partials (rr_new).  The system freezes
// instead when this iteration's update did not run (the same decision from the same slots) or rho' <= tol^2 ||b||^2.
// CTA 0 writes rho and the flag of the next iteration (rho_out / frz_out: the other parity's buffers, which no CTA of
// this launch reads) and, on the first iteration, ||b||^2 (bb_io, read on the later ones).  Grid (cg_ctas(n), systems).
__global__ void __launch_bounds__(CG_THREADS)
    cg_direction_kernel(float2* __restrict__ p, const float2* __restrict__ r, const double* __restrict__ pi_part, int pi_slots,
                        const double* __restrict__ rr_first, const double* __restrict__ bb_first, const double* __restrict__ rho_in,
                        const int* __restrict__ frz_in, double* bb_io, const double* __restrict__ rr_new,
                        double* __restrict__ rho_out, int* __restrict__ frz_out, double tol2, long n, int v4) {
    __shared__ double s_beta;
    __shared__ int s_frozen;
    const int sys = blockIdx.y;
    if (threadIdx.x < 32) {
        double pi, rho;
        int frozen;
        cg_scalars(sys, pi_part, pi_slots, rr_first, rho_in, frz_in, pi, rho, frozen);
        const double bb = rr_first ? cg_slots(bb_first + (long)sys * gridDim.x, gridDim.x) : __ldcg(bb_io + sys);
        double rho_next = rho, beta = 0.0;
        int frozen_next = 1;
        if (cg_runs(frozen, rho, pi)) {
            rho_next = cg_slots(rr_new + (long)sys * gridDim.x, gridDim.x);
            if (!(rho_next <= tol2 * bb)) {
                frozen_next = 0;
                beta = rho_next / rho;
            }
        }
        if (threadIdx.x == 0) {
            s_beta = beta;
            s_frozen = frozen_next;
            if (blockIdx.x == 0) {
                rho_out[sys] = rho_next;
                frz_out[sys] = frozen_next;
                if (rr_first) bb_io[sys] = bb;
            }
        }
    }
    __syncthreads();
    if (s_frozen) return;                                // uniform over the CTA
    const float be = (float)s_beta;
    const long base = (long)sys * n, pairs = (n + 1) / 2;
    for (long k = (long)blockIdx.x * CG_THREADS + threadIdx.x; k < pairs; k += (long)gridDim.x * CG_THREADS) {
        float2 r0, r1, p0, p1;
        cg_ld(r + base, k, n, v4, r0, r1);
        cg_ld(p + base, k, n, v4, p0, p1);
        cg_st(p + base, k, n, v4, cg_axpy(be, p0, r0), cg_axpy(be, p1, r1));
    }
}

static bool tz_fast(const pdu_nufft_plan* p) { return p->n0 == p->n1 && p->k0 == p->k1 && fast_fft_size(p->k0); }

// scratch per plane: T [N][K] on the fast path; grid + intermediate + cropped planes on the generic one
static size_t tz_plane_bytes(const pdu_nufft_plan* p) {
    if (tz_fast(p)) return (size_t)p->n0 * p->k1 * sizeof(float2);
    const size_t mid = (size_t)std::max((long)p->n0 * p->k1, (long)p->k0 * p->n1);
    return ((size_t)p->k0 * p->k1 + mid + (size_t)p->n0 * p->n1) * sizeof(float2);
}

// batch elements per chunk: a chunk's planes also fit gridDim.y; pd_unet_b200/nufft.py::_ToepPlan.workspace_bytes
// repeats this arithmetic to size the workspace
static int tz_batch_chunk(const pdu_nufft_plan* p, int batch, int coils) {
    return batch_chunk(tz_plane_bytes(p), 65535, batch, coils);
}

constexpr int TZ_SEQ_ROWS = 4;
template <int K>
static constexpr int tz_seq_rows_out() { return K == 2048 ? 2 : TZ_SEQ_ROWS; }

// cg: the conjugate-gradient epilogue (tz_rows_out_kernel<K, SO, true>), or null for the plain apply; sg: the coil-map
// gradient walk (tz_rows_out_kernel<K, SO, false, true>) into sg->gs instead of out
template <int K>
static int tz_apply_fast(pdu_nufft_plan* p, const float2* image, float2* out, const float2* kern, int kernel_batch,
                         const float2* smaps, int batch, int coils, int smaps_batch, int conj, float2* T, const TzCg* cg,
                         cudaStream_t st, const SmapsGrad* sg) {
    constexpr int N = K / 2, SC = ff_seq_cols<K>(), SO = tz_seq_rows_out<K>();
    const int planes = batch * coils;
    PDU_CUDA((ensure_dyn_smem<ff_rows_fwd_kernel<K, FF_SEQ_ROWS>>((int)ff_smem_bytes<K>(FF_SEQ_ROWS))));
    PDU_CUDA((ensure_dyn_smem<tz_cols_kernel<K, SC>>((int)ff_smem_bytes<K>(SC))));
    if (cg) PDU_CUDA((ensure_dyn_smem<tz_rows_out_kernel<K, SO, true>>((int)ff_smem_bytes<K>(SO))));
    else if (sg) PDU_CUDA((ensure_dyn_smem<tz_rows_out_kernel<K, SO, false, true>>((int)ff_smem_bytes<K>(SO))));
    else PDU_CUDA((ensure_dyn_smem<tz_rows_out_kernel<K, SO>>((int)ff_smem_bytes<K>(SO))));
    ff_rows_fwd_kernel<K, FF_SEQ_ROWS><<<dim3((unsigned)cdiv(N, FF_SEQ_ROWS), (unsigned)planes), FF_SEQ_ROWS * FastFft<K>::TPS,
                                         ff_smem_bytes<K>(FF_SEQ_ROWS), st>>>(image, smaps, T, p->d_s0, p->d_s1, p->d_w1,
                                                                              dims_of(p), coils, smaps_batch);
    PDU_LAUNCHED();
    tz_cols_kernel<K, SC><<<dim3((unsigned)(K / SC), (unsigned)planes), SC * FastFft<K>::TPS, ff_smem_bytes<K>(SC), st>>>(
        T, kern, p->d_w0, coils, kernel_batch, conj);
    PDU_LAUNCHED();
    const int out_planes = smaps ? batch : planes;
    const dim3 grid_out((unsigned)cdiv(N, SO), (unsigned)out_planes);
    const float scale = 1.f / ((float)K * (float)K);
    if (cg) {
        tz_rows_out_kernel<K, SO, true><<<grid_out, SO * FastFft<K>::TPS, ff_smem_bytes<K>(SO), st>>>(
            T, smaps, out, p->d_w1, coils, smaps_batch, scale, *cg, SmapsGrad{});
        PDU_LAUNCHED();
        note_kernel(OP_CG, "ff_rows_fwd_kernel<%d,%d> + tz_cols_kernel<%d,%d> + tz_rows_out_kernel<%d,%d,cg> + cg_update_kernel + "
                    "cg_direction_kernel (fast path, %d systems of %dx%d)", K, FF_SEQ_ROWS, K, SC, K, SO, out_planes, N, N);
        return PDU_OK;
    }
    if (sg) {
        const dim3 grid_gs((unsigned)cdiv(N, SO), (unsigned)((sg->per_batch ? batch : 1) * coils));
        tz_rows_out_kernel<K, SO, false, true><<<grid_gs, SO * FastFft<K>::TPS, ff_smem_bytes<K>(SO), st>>>(
            T, nullptr, sg->gs, p->d_w1, coils, 1, scale * sg->scale, TzCg{}, *sg);
        PDU_LAUNCHED();
        note_kernel(OP_SMAPS_GRAD, "ff_rows_fwd_kernel<%d,%d> + tz_cols_kernel<%d,%d> + tz_rows_out_kernel<%d,%d,smaps_grad> per "
                    "term (fast path, %d planes of %dx%d)", K, FF_SEQ_ROWS, K, SC, K, SO, planes, N, N);
        return PDU_OK;
    }
    tz_rows_out_kernel<K, SO><<<grid_out, SO * FastFft<K>::TPS, ff_smem_bytes<K>(SO), st>>>(T, smaps, out, p->d_w1, coils,
                                                                                            smaps_batch, scale, TzCg{},
                                                                                            SmapsGrad{});
    PDU_LAUNCHED();
    note_kernel(OP_TOEP, "ff_rows_fwd_kernel<%d,%d> + tz_cols_kernel<%d,%d> + tz_rows_out_kernel<%d,%d> (fast path, %d planes of %dx%d)",
                K, FF_SEQ_ROWS, K, SC, K, SO, planes, N, N);
    return PDU_OK;
}

// the generic passes' column SEQ: 8 where it fits shared memory, 2 otherwise (2048-point columns)
static bool tz_cols_seq8(const pdu_nufft_plan* p) { return pf_smem_bytes(PF_SEQ_COLS, p->k0) <= 200 * 1024; }

template <int SC>
static int tz_apply_generic(pdu_nufft_plan* p, const float2* image, float2* out, const float2* kern, int kernel_batch,
                            const float2* smaps, int batch, int coils, int smaps_batch, int conj, float2* ws, const TzCg* cg,
                            cudaStream_t st, const SmapsGrad* sg) {
    const int planes = batch * coils;
    const long cells = (long)p->k0 * p->k1;
    float2* grid = ws;
    float2* T = grid + planes * cells;
    float2* U = T + (long)planes * std::max((long)p->n0 * p->k1, (long)p->k0 * p->n1);
    const NufftDims d = dims_of(p);
    const int pitch1 = pfft_pitch(p->k1), pitch0 = pfft_pitch(p->k0);
    int rc = pf_set_smem(pfft_rows_fwd_kernel<PF_SEQ_ROWS>, pf_smem_bytes(PF_SEQ_ROWS, p->k1));
    if (!rc) rc = pf_set_smem(pfft_cols_fwd_kernel<SC>, pf_smem_bytes(SC, p->k0));
    if (!rc) rc = pf_set_smem(pfft_rows_adj_kernel<PF_SEQ_ROWS>, pf_smem_bytes(PF_SEQ_ROWS, p->k1));
    if (!rc) rc = pf_set_smem(pfft_cols_adj_kernel<SC>, pf_smem_bytes(SC, p->k0));
    if (rc) return rc;
    pfft_rows_fwd_kernel<PF_SEQ_ROWS><<<dim3((unsigned)cdiv(p->n0, PF_SEQ_ROWS), (unsigned)planes), 256,
                                        pf_smem_bytes(PF_SEQ_ROWS, p->k1), st>>>(image, smaps, T, p->d_s0, p->d_s1, p->d_w1, p->pf1,
                                                                                 d, coils, smaps_batch, pitch1);
    PDU_LAUNCHED();
    pfft_cols_fwd_kernel<SC><<<dim3((unsigned)cdiv(p->k1, SC), (unsigned)planes), 256, pf_smem_bytes(SC, p->k0), st>>>(
        T, grid, p->d_w0, p->pf0, d, pitch0);
    PDU_LAUNCHED();
    tz_mul_kernel<<<stream_grid(planes * cells), 256, 0, st>>>(grid, kern, cells, coils, kernel_batch, conj, planes * cells);
    PDU_LAUNCHED();
    pfft_rows_adj_kernel<PF_SEQ_ROWS><<<dim3((unsigned)cdiv(p->k0, PF_SEQ_ROWS), (unsigned)planes), 256,
                                        pf_smem_bytes(PF_SEQ_ROWS, p->k1), st>>>(grid, T, p->d_w1, p->pf1, d, pitch1);
    PDU_LAUNCHED();
    pfft_cols_adj_kernel<SC><<<dim3((unsigned)cdiv(p->n1, SC), (unsigned)planes), 256, pf_smem_bytes(SC, p->k0), st>>>(
        T, U, p->d_w0, p->pf0, d, pitch0);
    PDU_LAUNCHED();
    if (sg) {
        rc = launch_smaps_grad(p, U, cropped_dims(p), coils, 1.f / ((float)p->k0 * (float)p->k1), *sg, st);
        if (rc) return rc;
        note_kernel(OP_SMAPS_GRAD, "pfft_rows_fwd_kernel<%d> + pfft_cols_fwd_kernel<%d> + tz_mul_kernel + pfft_rows_adj_kernel<%d> + "
                    "pfft_cols_adj_kernel<%d> + smaps_grad_kernel per term (generic path, %d planes of %dx%d)",
                    PF_SEQ_ROWS, SC, PF_SEQ_ROWS, SC, planes, p->n0, p->n1);
        return PDU_OK;
    }
    const int out_planes = smaps ? batch : planes;
    rc = launch_crop_apod(p, U, cropped_dims(p), smaps, out, out_planes, coils, smaps_batch, 1.f / ((float)p->k0 * (float)p->k1),
                          0, st);
    if (rc) return rc;
    if (cg) {
        const long n = (long)p->n0 * p->n1;
        cg_lam_dot_kernel<<<dim3((unsigned)cg_ctas(n), (unsigned)out_planes), CG_THREADS, 0, st>>>(out, cg->p, cg->lam, cg->lam_div,
                                                                                                  cg->part, n, cg_v4(n, {(const void*)out, (const void*)cg->p}));
        PDU_LAUNCHED();
        note_kernel(OP_CG, "pfft_rows_fwd_kernel<%d> + pfft_cols_fwd_kernel<%d> + tz_mul_kernel + pfft_rows_adj_kernel<%d> + "
                    "pfft_cols_adj_kernel<%d> + crop_apod_kernel + cg_lam_dot_kernel + cg_update_kernel + cg_direction_kernel "
                    "(generic path, %d systems of %dx%d)", PF_SEQ_ROWS, SC, PF_SEQ_ROWS, SC, out_planes, p->n0, p->n1);
        return PDU_OK;
    }
    note_kernel(OP_TOEP, "pfft_rows_fwd_kernel<%d> + pfft_cols_fwd_kernel<%d> + tz_mul_kernel + pfft_rows_adj_kernel<%d> + "
                "pfft_cols_adj_kernel<%d> + crop_apod_kernel (generic path, %d planes of %dx%d)",
                PF_SEQ_ROWS, SC, PF_SEQ_ROWS, SC, planes, p->n0, p->n1);
    return PDU_OK;
}

static int tz_apply_chunk(pdu_nufft_plan* p, const float2* image, float2* out, const float2* kern, int kernel_batch,
                          const float2* smaps, int batch, int coils, int smaps_batch, int conj, float2* ws, cudaStream_t st,
                          const TzCg* cg = nullptr, const SmapsGrad* sg = nullptr) {
    if (tz_fast(p))
        return with_fast_fft_size(p->k0, [&](auto k) {
            return tz_apply_fast<decltype(k)::value>(p, image, out, kern, kernel_batch, smaps, batch, coils, smaps_batch, conj, ws,
                                                     cg, st, sg);
        });
    if (tz_cols_seq8(p))
        return tz_apply_generic<PF_SEQ_COLS>(p, image, out, kern, kernel_batch, smaps, batch, coils, smaps_batch, conj, ws, cg, st, sg);
    return tz_apply_generic<2>(p, image, out, kern, kernel_batch, smaps, batch, coils, smaps_batch, conj, ws, cg, st, sg);
}

// kernel build, step 4: the full (unpruned) 2-D FFT of p_circ, in place in `kern` with T as the intermediate
template <int SC>
static int tz_kernel_fft(pdu_nufft_plan* p, float2* kern, float2* T, int kernels, cudaStream_t st) {
    NufftDims d = dims_of(p);
    d.n0 = p->k0;            // pruning off: every row of the input is stored, every column is transformed
    d.n1 = p->k1;
    int rc = pf_set_smem(pfft_rows_fwd_kernel<PF_SEQ_ROWS>, pf_smem_bytes(PF_SEQ_ROWS, p->k1));
    if (!rc) rc = pf_set_smem(pfft_cols_fwd_kernel<SC>, pf_smem_bytes(SC, p->k0));
    if (rc) return rc;
    pfft_rows_fwd_kernel<PF_SEQ_ROWS><<<dim3((unsigned)cdiv(p->k0, PF_SEQ_ROWS), (unsigned)kernels), 256,
                                        pf_smem_bytes(PF_SEQ_ROWS, p->k1), st>>>(kern, nullptr, T, p->d_s0, p->d_s1, p->d_w1, p->pf1,
                                                                                 d, 1, 1, pfft_pitch(p->k1));
    PDU_LAUNCHED();
    pfft_cols_fwd_kernel<SC><<<dim3((unsigned)cdiv(p->k1, SC), (unsigned)kernels), 256, pf_smem_bytes(SC, p->k0), st>>>(
        T, kern, p->d_w0, p->pf0, d, pfft_pitch(p->k0));
    PDU_LAUNCHED();
    return PDU_OK;
}

// ------------------------------------------------------------------ pdu_toep_cg_c64: the solve's workspace and loop
// slots of the Re<p, q> partials per system: tz_rows_out_kernel's CTAs per plane on the fast path (its SEQ is
// tz_seq_rows_out), cg_lam_dot_kernel's on the generic one
static int cg_pi_slots(const pdu_nufft_plan* p) {
    if (tz_fast(p)) return (int)cdiv(p->n0, p->k0 == 2048 ? tz_seq_rows_out<2048>() : tz_seq_rows_out<256>());
    return cg_ctas((long)p->n0 * p->n1);
}

// one chunk of cb batch elements: the apply's scratch; r, p, q; the partial slots of Re<p, q>, of ||r||^2 (two sets,
// by iteration parity) and of ||b||^2; rho and the frozen flag by parity; ||b||^2
struct CgWs {
    float2 *tz, *r, *p, *q;
    double *pi, *rr[2], *bb, *rho[2], *bbv;
    int* frz[2];
    size_t bytes;
};

static CgWs cg_layout(const pdu_nufft_plan* p, int cb, int coils, bool has_smaps, void* base) {
    const size_t S = (size_t)cb * (has_smaps ? 1 : coils), n = (size_t)p->n0 * p->n1;
    const size_t G = (size_t)cg_ctas((long)n), GP = (size_t)cg_pi_slots(p);
    size_t off = 0;
    auto take = [&](size_t bytes) {
        void* q = (void*)((uintptr_t)base + off);
        off += align256(bytes);
        return q;
    };
    CgWs w;
    w.tz = (float2*)take((size_t)cb * coils * tz_plane_bytes(p));
    w.r = (float2*)take(S * n * sizeof(float2));
    w.p = (float2*)take(S * n * sizeof(float2));
    w.q = (float2*)take(S * n * sizeof(float2));
    w.pi = (double*)take(S * GP * sizeof(double));
    for (int e = 0; e < 2; ++e) w.rr[e] = (double*)take(S * G * sizeof(double));
    w.bb = (double*)take(S * G * sizeof(double));
    for (int e = 0; e < 2; ++e) w.rho[e] = (double*)take(S * sizeof(double));
    w.bbv = (double*)take(S * sizeof(double));
    for (int e = 0; e < 2; ++e) w.frz[e] = (int*)take(S * sizeof(int));
    w.bytes = off;
    return w;
}

// the whole solve of one chunk (nb batch elements): [x0: one apply] + cg_init_kernel, then per iteration the apply with
// the CG epilogue, cg_update_kernel and cg_direction_kernel -- 5 launches on the fast path, 9 on the generic one
static int tz_cg_chunk(pdu_nufft_plan* p, const float2* b, const float2* x0, float2* x, const float2* kern, int kernel_batch,
                       const float2* smaps, int nb, int coils, int smaps_batch, const float* lam, int lam_div, int max_iter,
                       double tol2, int conj, const CgWs& w, cudaStream_t st) {
    const int S = smaps ? nb : nb * coils, G = cg_ctas((long)p->n0 * p->n1), GP = cg_pi_slots(p);
    const long n = (long)p->n0 * p->n1;
    const dim3 grid((unsigned)G, (unsigned)S);
    const int v4 = cg_v4(n, {(const void*)b, (const void*)x0, (const void*)x, (const void*)w.r, (const void*)w.p, (const void*)w.q});
    TzCg cg{x0, lam, lam_div, w.pi};
    const float2* q0 = nullptr;
    if (x0 && max_iter > 0) {                            // q = (T + lam) x0 for r = b - q
        int rc = tz_apply_chunk(p, x0, w.q, kern, kernel_batch, smaps, nb, coils, smaps_batch, conj, w.tz, st, &cg);
        if (rc) return rc;
        q0 = w.q;
    }
    cg_init_kernel<<<grid, CG_THREADS, 0, st>>>(b, x0, x, q0, w.r, w.p, w.rr[0], w.bb, n, v4);
    PDU_LAUNCHED();
    cg.p = w.p;
    for (int it = 0; it < max_iter; ++it) {
        const int e = it & 1;
        const double* first = it == 0 ? w.rr[0] : nullptr;
        int rc = tz_apply_chunk(p, w.p, w.q, kern, kernel_batch, smaps, nb, coils, smaps_batch, conj, w.tz, st, &cg);
        if (rc) return rc;
        cg_update_kernel<<<grid, CG_THREADS, 0, st>>>(x, w.r, w.p, w.q, w.pi, GP, first, w.rho[e], w.frz[e], w.rr[e ^ 1], n, v4);
        PDU_LAUNCHED();
        cg_direction_kernel<<<grid, CG_THREADS, 0, st>>>(w.p, w.r, w.pi, GP, first, w.bb, w.rho[e], w.frz[e], w.bbv, w.rr[e ^ 1],
                                                         w.rho[e ^ 1], w.frz[e ^ 1], tol2, n, v4);
        PDU_LAUNCHED();
    }
    if (max_iter == 0)
        note_kernel(OP_CG, "cg_init_kernel only (max_iter 0, %d systems of %dx%d)", S, p->n0, p->n1);
    return PDU_OK;
}

// n entries of `host` to a new device array *dst
template <typename T>
static cudaError_t upload(T** dst, const T* host, size_t n) {
    cudaError_t e = cudaMalloc(dst, n * sizeof(T));
    if (e == cudaSuccess) e = cudaMemcpy(*dst, host, n * sizeof(T), cudaMemcpyHostToDevice);
    return e;
}

// the twiddle tables exp(-2 pi i j / K), j < K, of both axes (d_w0, d_w1), computed in float64
static cudaError_t upload_twiddles(pdu_nufft_plan* p) {
    cudaError_t e = cudaSuccess;
    for (int ax = 0; ax < 2 && e == cudaSuccess; ++ax) {
        const int K = ax == 0 ? p->k0 : p->k1;
        std::vector<float2> w((size_t)K);
        for (int i = 0; i < K; ++i) {
            const double a = -2.0 * 3.14159265358979323846 * (double)i / (double)K;
            w[i] = make_float2((float)cos(a), (float)sin(a));
        }
        e = upload(ax == 0 ? &p->d_w0 : &p->d_w1, w.data(), (size_t)K);
    }
    return e;
}

// a new plan of either kind for an n0 x n1 image on a k0 x k1 grid, on the current device; init(p) sets the rest and
// uploads the kind's tables.  On an error the plan is destroyed and *plan stays null.
template <typename Init>
static int plan_create(pdu_nufft_plan_t** plan, int n0, int n1, int k0, int k1, const char* who, Init&& init) {
    pdu_nufft_plan* p = new (std::nothrow) pdu_nufft_plan();
    if (!p) {
        set_error("%s: out of host memory", who);
        return PDU_ENOMEM;
    }
    p->n0 = n0; p->n1 = n1; p->k0 = k0; p->k1 = k1;
    cudaError_t e = cudaGetDevice(&p->device);
    if (e == cudaSuccess) e = init(p);
    if (e != cudaSuccess) {
        set_error("%s: %s", who, cudaGetErrorString(e));
        pdu_nufft_plan_destroy(p);
        return PDU_ECUDA;
    }
    *plan = p;
    return PDU_OK;
}

}  // namespace pdu

using namespace pdu;

extern "C" {

int pdu_nufft_plan_create(pdu_nufft_plan_t** plan, int n0, int n1, int k0, int k1, int numpoints, int table_oversamp,
                          int shift0, int shift1, const float* table0, const float* table1, const float* scal0,
                          const float* scal1) {
    PDU_REQUIRE(plan != nullptr, "pdu_nufft_plan_create: plan is null");
    *plan = nullptr;
    PDU_REQUIRE(n0 > 0 && n1 > 0 && k0 >= n0 && k1 >= n1, "pdu_nufft_plan_create: need 0 < n <= k per axis");
    PDU_REQUIRE(k1 % 2 == 0, "pdu_nufft_plan_create: the last grid dimension must be even (got %d)", k1);
    PDU_REQUIRE(numpoints >= 1 && numpoints <= MAXJ, "pdu_nufft_plan_create: numpoints must be in 1..%d", MAXJ);
    PDU_REQUIRE(table_oversamp >= 1 && (numpoints * table_oversamp) % 2 == 0,
                "pdu_nufft_plan_create: numpoints * table_oversamp must be even");
    PDU_REQUIRE(table0 && table1 && scal0 && scal1, "pdu_nufft_plan_create: null table");
    return plan_create(plan, n0, n1, k0, k1, "pdu_nufft_plan_create", [&](pdu_nufft_plan* p) {
        p->J = numpoints;
        p->L = table_oversamp;
        p->shift0 = shift0;
        p->shift1 = shift1;
        p->pfft_ok = pfft_factor(k0, &p->pf0) && pfft_factor(k1, &p->pf1) &&
                     pf_smem_bytes(PF_SEQ_ROWS, k1) <= 200 * 1024 && pf_smem_bytes(PF_SEQ_COLS, k0) <= 200 * 1024;
        const size_t tl = (size_t)numpoints * table_oversamp + 1;
        cudaError_t e = upload(&p->d_t0, (const float2*)table0, tl);
        if (e == cudaSuccess) e = upload(&p->d_t1, (const float2*)table1, tl);
        if (e == cudaSuccess) e = upload(&p->d_s0, scal0, (size_t)n0);
        if (e == cudaSuccess) e = upload(&p->d_s1, scal1, (size_t)n1);
        if (e == cudaSuccess && (p->pfft_ok || (fast_fft_size(k0) && fast_fft_size(k1)))) e = upload_twiddles(p);
        return e;
    });
}

int pdu_nufft_plan_destroy(pdu_nufft_plan_t* p) {
    if (!p) return PDU_OK;
    for (auto& kv : p->fft) cufftDestroy(kv.second);
    cudaFree(p->d_t0);
    cudaFree(p->d_t1);
    cudaFree(p->d_s0);
    cudaFree(p->d_s1);
    cudaFree(p->d_w0);
    cudaFree(p->d_w1);
    delete p;
    return PDU_OK;
}

size_t pdu_nufft_workspace_bytes(const pdu_nufft_plan_t* p, int planes) {
    if (!p || planes <= 0) return 0;
    // oversampled grid | intermediate of the pruned FFT (one axis transformed) | cropped adjoint result
    const size_t grid = (size_t)p->k0 * p->k1;
    const size_t mid = (size_t)std::max((long)p->n0 * p->k1, (long)p->k0 * p->n1);
    const size_t crop = (size_t)p->n0 * p->n1;
    return (size_t)planes * (grid + mid + crop) * sizeof(float2);
}

// batch elements per chunk of the generic path, by its oversampled grids; a chunk's planes also fit gridDim.y
static int nufft_batch_chunk(const pdu_nufft_plan* p, int batch, int coils) {
    return batch_chunk((size_t)p->k0 * p->k1 * sizeof(float2), 65535, batch, coils);
}

// variant 2 = the register-resident pruned FFT (pfft_fast.cuh), 1 = the generic pruned FFT (pfft.cuh), 0 = pad + cuFFT;
// opt: the A/B option of the direction.  Measured on B200 (64 planes of 640^2): the generic pruned passes move 2.5x fewer
// bytes but are still ~1.7x slower than cuFFT's register-resident radix kernels (row+column 407 us vs 238 us).
static int fft_variant(const pdu_nufft_plan* p, int opt) {
    int variant = option(opt);
    // default: the register-resident pruned FFT on the BASELINE grids, the generic pruned FFT on every other grid
    // that factors into 2, 3, 5 (slower than cuFFT, but the library's own); cuFFT only for other prime factors
    if (variant < 0) variant = ff_supported(p) ? 2 : (p->pfft_ok ? 1 : 0);
    if ((variant == 2 && !ff_supported(p)) || (variant == 1 && !p->pfft_ok)) variant = 0;
    return variant;
}

static int nufft_fwd_chunk(pdu_nufft_plan_t* p, const float2* image, float2* kdata, const float* omega, const float2* smaps,
                           int batch, int coils, int smaps_batch, long m, float scale, float2* grid, cudaStream_t st) {
    const int planes = batch * coils;
    const long total = (long)planes * p->k0 * p->k1;
    const int variant = fft_variant(p, OPT_NUFFT_FWD);
    float2* T = grid + total;
    int rc;
    if (variant == 2) {
        rc = with_fast_fft_size(p->k0, [&](auto k) {
            return ff_forward<decltype(k)::value>(p, image, smaps, T, grid, planes, coils, smaps_batch, st);
        });
        if (rc) return rc;
    } else if (variant == 1) {
        // pruned FFT: apodise + pad + transform the n0 non-zero rows, then every column
        const NufftDims d = dims_of(p);
        const int pitch1 = pfft_pitch(p->k1), pitch0 = pfft_pitch(p->k0);
        rc = pf_set_smem(pfft_rows_fwd_kernel<PF_SEQ_ROWS>, pf_smem_bytes(PF_SEQ_ROWS, p->k1));
        if (rc) return rc;
        rc = pf_set_smem(pfft_cols_fwd_kernel<PF_SEQ_COLS>, pf_smem_bytes(PF_SEQ_COLS, p->k0));
        if (rc) return rc;
        pfft_rows_fwd_kernel<PF_SEQ_ROWS><<<dim3((unsigned)cdiv(p->n0, PF_SEQ_ROWS), (unsigned)planes), 256,
                                            pf_smem_bytes(PF_SEQ_ROWS, p->k1), st>>>(image, smaps, T, p->d_s0, p->d_s1, p->d_w1,
                                                                                     p->pf1, d, coils, smaps_batch, pitch1);
        PDU_LAUNCHED();
        pfft_cols_fwd_kernel<PF_SEQ_COLS><<<dim3((unsigned)cdiv(p->k1, PF_SEQ_COLS), (unsigned)planes), 256,
                                            pf_smem_bytes(PF_SEQ_COLS, p->k0), st>>>(T, grid, p->d_w0, p->pf0, d, pitch0);
        PDU_LAUNCHED();
    } else {
        apod_pad_kernel<<<stream_grid(total / 2), 256, 0, st>>>(image, smaps, (float4*)grid, p->d_s0, p->d_s1, dims_of(p), coils,
                                                                smaps_batch, total / 2);
        PDU_LAUNCHED();
        rc = run_fft(p, grid, planes, CUFFT_FORWARD, st);
        if (rc) return rc;
    }
    note_kernel(OP_NUFFT_FWD, "%s + interp_fwd_kernel<%d> (%d planes of %dx%d, M=%ld)",
                variant == 2 ? "ff_rows_fwd_kernel + ff_cols_fwd_kernel (register-resident pruned FFT)"
                             : (variant == 1 ? "pfft_rows_fwd_kernel + pfft_cols_fwd_kernel (generic pruned FFT)"
                                             : "apod_pad_kernel + cuFFT C2C"),
                p->J == 6 ? 6 : 0, planes, p->k0, p->k1, m);
    return launch_interp_fwd(p, grid, kdata, omega, planes, m, scale, st);
}

static int nufft_adj_chunk(pdu_nufft_plan_t* p, const float2* kdata, float2* image, const float* omega, const float2* smaps,
                           int batch, int coils, int smaps_batch, long m, float scale, float2* grid, const void* csr,
                           cudaStream_t st, const SmapsGrad* sg = nullptr) {
    const int planes = batch * coils;
    int rc;
    const int variant = fft_variant(p, OPT_NUFFT_ADJ);
    // the gridded samples stay compact (non-empty cells only) between the sorted gather and the register FFT's row pass
    // (only for sparse trajectories, at most 8 interpolation entries per cell on average: 48 radial spokes on 640^2 have
    //  2.7 and leave 61 % of the cells empty; a dense trajectory fills the grid and would only pay for the indirection)
    bool compact = csr && variant == 2 && (double)m * p->J * p->J <= 8.0 * (double)p->k0 * p->k1;
    float2* T = grid + (long)planes * p->k0 * p->k1;
    float2* U = T + (long)planes * std::max((long)p->n0 * p->k1, (long)p->k0 * p->n1);
    if (csr) {
        // the FFT's intermediate buffer T and the cropped result U behind it are free until the transform starts: they
        // hold the plane-interleaved kdata
        const long mid_elems = (long)planes * (std::max((long)p->n0 * p->k1, (long)p->k0 * p->n1) + (long)p->n0 * p->n1);
        const bool fits = m * (long)((planes + 3) & ~3) <= mid_elems;
        rc = launch_interp_adj_csr(p, kdata, grid, csr, planes, m, st, fits ? T : nullptr, &compact);   // writes every cell: no memset
    } else {
        PDU_CUDA(cudaMemsetAsync(grid, 0, (size_t)planes * p->k0 * p->k1 * sizeof(float2), st));
        rc = launch_interp_adj(p, kdata, grid, omega, planes, m, st);
    }
    if (rc) return rc;
    note_kernel(sg ? OP_SMAPS_GRAD : OP_NUFFT_ADJ, "%s + %s + %s (%d planes of %dx%d, M=%ld)",
                csr ? (compact ? "transpose_kdata_kernel + interp_adj_csrT_kernel (sorted gather: 4 lanes per cell x 16 planes, long rows by warps, non-empty cells only)"
                               : "transpose_kdata_kernel + interp_adj_csrT_kernel (sorted gather: 4 lanes per cell x 16 planes, long rows by warps)")
                    : "interp_adj_kernel (float2 atomics)",
                variant == 2 ? (compact ? "ff_rows_adj_compact_kernel + ff_cols_adj_kernel (register-resident pruned FFT)"
                                        : "ff_rows_adj_kernel + ff_cols_adj_kernel (register-resident pruned FFT)")
                             : (variant == 1 ? "pfft_rows_adj_kernel + pfft_cols_adj_kernel (generic pruned FFT)"
                                             : "cuFFT C2C"),
                sg ? "smaps_grad_kernel" : "crop_apod_kernel", planes, p->k0, p->k1, m);
    // the planes the adjoint ends on, with their geometry: the pruned FFTs' cropped n0 x n1 planes U, or cuFFT's full grid
    const float2* Ue = U;
    NufftDims de = cropped_dims(p);
    if (variant == 2) {
        const CsrView cv = compact ? csr_layout(p, m, const_cast<void*>(csr), false) : CsrView{};
        const int* nzi = compact ? cv.nz_idx : nullptr;
        rc = with_fast_fft_size(p->k0, [&](auto k) { return ff_adjoint<decltype(k)::value>(p, grid, T, U, planes, st, nzi); });
        if (rc) return rc;
    } else if (variant == 1) {
        // pruned inverse FFT: every row but only the n1 kept outputs, then the n1 kept columns and n0 kept outputs
        const NufftDims d = dims_of(p);
        rc = pf_set_smem(pfft_rows_adj_kernel<PF_SEQ_ROWS>, pf_smem_bytes(PF_SEQ_ROWS, p->k1));
        if (rc) return rc;
        rc = pf_set_smem(pfft_cols_adj_kernel<PF_SEQ_COLS>, pf_smem_bytes(PF_SEQ_COLS, p->k0));
        if (rc) return rc;
        pfft_rows_adj_kernel<PF_SEQ_ROWS><<<dim3((unsigned)cdiv(p->k0, PF_SEQ_ROWS), (unsigned)planes), 256,
                                            pf_smem_bytes(PF_SEQ_ROWS, p->k1), st>>>(grid, T, p->d_w1, p->pf1, d,
                                                                                     pfft_pitch(p->k1));
        PDU_LAUNCHED();
        pfft_cols_adj_kernel<PF_SEQ_COLS><<<dim3((unsigned)cdiv(p->n1, PF_SEQ_COLS), (unsigned)planes), 256,
                                            pf_smem_bytes(PF_SEQ_COLS, p->k0), st>>>(T, U, p->d_w0, p->pf0, d, pfft_pitch(p->k0));
        PDU_LAUNCHED();
    } else {
        rc = run_fft(p, grid, planes, CUFFT_INVERSE, st);
        if (rc) return rc;
        Ue = grid;
        de = dims_of(p);
    }
    if (sg) return launch_smaps_grad(p, Ue, de, coils, scale, *sg, st);
    return launch_crop_apod(p, Ue, de, smaps, image, smaps ? batch : planes, coils, smaps_batch, scale, 0, st);
}

int pdu_nufft_fwd_c64(pdu_nufft_plan_t* p, const float* image, float* kdata, const float* omega, const float* smaps,
                      int batch, int coils, int smaps_batch, long m, float scale, void* workspace, size_t workspace_bytes,
                      pdu_stream_t stream) {
    int rc = check_call(p, image, kdata, omega, batch, coils, smaps_batch, smaps, m, "pdu_nufft_fwd_c64");
    if (rc) return rc;
    PDU_CHECK_DEVICE("pdu_nufft_fwd_c64");
    const int cb = nufft_batch_chunk(p, batch, coils);
    rc = check_workspace("pdu_nufft_fwd_c64", workspace, workspace_bytes, pdu_nufft_workspace_bytes(p, cb * coils), false,
                         PDU_ENOMEM);
    if (rc) return rc;
    const long plane = (long)p->n0 * p->n1;
    const long img_b = (smaps ? 1 : coils) * plane, smap_b = smaps_batch == 1 ? 0 : coils * plane;
    return for_each_chunk(batch, cb, [&](int b0, int nb) {
        return nufft_fwd_chunk(p, (const float2*)image + b0 * img_b, (float2*)kdata + (long)b0 * coils * m, omega,
                               smaps ? (const float2*)smaps + b0 * smap_b : nullptr, nb, coils, smaps_batch == 1 ? 1 : nb, m,
                               scale, (float2*)workspace, (cudaStream_t)stream);
    });
}

size_t pdu_nufft_csr_bytes(const pdu_nufft_plan_t* p, long m) {
    if (!p || m <= 0) return 0;
    return csr_layout(p, m, nullptr).total;
}

size_t pdu_nufft_csr_bytes2(const pdu_nufft_plan_t* p, long m, size_t* persist_bytes) {
    if (persist_bytes) *persist_bytes = 0;
    if (!p || m <= 0) return 0;
    const CsrView v = csr_layout(p, m, nullptr);
    // row_ptr | n_long | long_rows | samp | w are what applying the matrix reads; everything behind is sort scratch
    if (persist_bytes) *persist_bytes = (size_t)((char*)v.key_in - (char*)nullptr);
    return v.total;
}

int pdu_nufft_csr_build(pdu_nufft_plan_t* p, const float* omega, long m, void* csr, size_t csr_bytes, pdu_stream_t stream) {
    PDU_REQUIRE(p && omega && m > 0, "pdu_nufft_csr_build: null pointer or m <= 0");
    PDU_REQUIRE(!p->toep, "pdu_nufft_csr_build: a Toeplitz plan has no interpolation tables");
    return csr_build(p, omega, m, csr, csr_bytes, (cudaStream_t)stream);
}

int pdu_nufft_interp_adj_csr_c64(pdu_nufft_plan_t* p, const float* kdata, float* grid, const void* csr, int planes, long m,
                                 pdu_stream_t stream) {
    PDU_REQUIRE(p && kdata && grid && csr && planes > 0 && m > 0, "pdu_nufft_interp_adj_csr_c64: null pointer or empty problem");
    PDU_REQUIRE(!p->toep, "pdu_nufft_interp_adj_csr_c64: a Toeplitz plan has no interpolation tables");
    return launch_interp_adj_csr(p, (const float2*)kdata, (float2*)grid, csr, planes, m, (cudaStream_t)stream);
}

int pdu_nufft_adj_csr_c64(pdu_nufft_plan_t* p, const float* kdata, float* image, const float* omega, const float* smaps,
                          int batch, int coils, int smaps_batch, long m, float scale, const void* csr, void* workspace,
                          size_t workspace_bytes, pdu_stream_t stream);

int pdu_nufft_adj_c64(pdu_nufft_plan_t* p, const float* kdata, float* image, const float* omega, const float* smaps,
                      int batch, int coils, int smaps_batch, long m, float scale, void* workspace, size_t workspace_bytes,
                      pdu_stream_t stream) {
    return pdu_nufft_adj_csr_c64(p, kdata, image, omega, smaps, batch, coils, smaps_batch, m, scale, nullptr, workspace,
                                 workspace_bytes, stream);
}

int pdu_nufft_adj_csr_c64(pdu_nufft_plan_t* p, const float* kdata, float* image, const float* omega, const float* smaps,
                          int batch, int coils, int smaps_batch, long m, float scale, const void* csr, void* workspace,
                          size_t workspace_bytes, pdu_stream_t stream) {
    int rc = check_call(p, kdata, image, omega, batch, coils, smaps_batch, smaps, m, "pdu_nufft_adj_c64");
    if (rc) return rc;
    PDU_CHECK_DEVICE("pdu_nufft_adj_c64");
    const int cb = nufft_batch_chunk(p, batch, coils);
    rc = check_workspace("pdu_nufft_adj_c64", workspace, workspace_bytes, pdu_nufft_workspace_bytes(p, cb * coils), false,
                         PDU_ENOMEM);
    if (rc) return rc;
    const long plane = (long)p->n0 * p->n1;
    const long img_b = (smaps ? 1 : coils) * plane, smap_b = smaps_batch == 1 ? 0 : coils * plane;
    return for_each_chunk(batch, cb, [&](int b0, int nb) {
        return nufft_adj_chunk(p, (const float2*)kdata + (long)b0 * coils * m, (float2*)image + b0 * img_b, omega,
                               smaps ? (const float2*)smaps + b0 * smap_b : nullptr, nb, coils, smaps_batch == 1 ? 1 : nb, m,
                               scale, (float2*)workspace, csr, (cudaStream_t)stream);
    });
}

int pdu_nufft_fwd_binned_c64(pdu_nufft_plan_t* p, const float* image, float* kdata, const float* smaps, int batch, int coils,
                             int smaps_batch, long m, float scale, const void* bins, int flags, void* workspace,
                             size_t workspace_bytes, pdu_stream_t stream) {
    int rc = check_call(p, image, kdata, bins, batch, coils, smaps_batch, smaps, m, "pdu_nufft_fwd_binned_c64");
    if (rc) return rc;
    PDU_CHECK_DEVICE("pdu_nufft_fwd_binned_c64");
    if (!fused_supported(p)) {
        set_error("pdu_nufft_fwd_binned_c64: grid %d x %d (J = %d) has no fused path; use pdu_nufft_fwd_c64", p->k0, p->k1, p->J);
        return PDU_EUNSUPPORTED;
    }
    rc = check_workspace("pdu_nufft_fwd_binned_c64", workspace, workspace_bytes, fused_workspace_bytes(p, batch * coils, m), true,
                         PDU_ENOMEM);
    if (rc) return rc;
    return fused_forward(p, image, kdata, smaps, batch, coils, smaps_batch, m, scale, bins, flags, workspace, (cudaStream_t)stream);
}

int pdu_nufft_adj_binned_c64(pdu_nufft_plan_t* p, const float* kdata, float* image, const float* smaps, const float* kweight,
                             int batch, int coils, int smaps_batch, long m, float scale, const void* bins, int flags,
                             void* workspace, size_t workspace_bytes, pdu_stream_t stream) {
    int rc = check_call(p, kdata, image, bins, batch, coils, smaps_batch, smaps, m, "pdu_nufft_adj_binned_c64");
    if (rc) return rc;
    PDU_CHECK_DEVICE("pdu_nufft_adj_binned_c64");
    if (!fused_supported(p)) {
        set_error("pdu_nufft_adj_binned_c64: grid %d x %d (J = %d) has no fused path; use pdu_nufft_adj_c64", p->k0, p->k1, p->J);
        return PDU_EUNSUPPORTED;
    }
    rc = check_workspace("pdu_nufft_adj_binned_c64", workspace, workspace_bytes, fused_workspace_bytes(p, batch * coils, m), true,
                         PDU_ENOMEM);
    if (rc) return rc;
    return fused_adjoint(p, kdata, image, smaps, kweight, batch, coils, smaps_batch, m, scale, bins, flags, workspace,
                         (cudaStream_t)stream);
}

int pdu_nufft_adj_smaps_grad_c64(pdu_nufft_plan_t* p, const float* kdata, const float* q, float* gs, const float* omega,
                                 const void* csr, const void* bins, const float* kweight, int batch, int coils,
                                 int smaps_batch, long m, float scale, int flags, int accumulate, void* workspace,
                                 size_t workspace_bytes, pdu_stream_t stream) {
    const char* who = "pdu_nufft_adj_smaps_grad_c64";
    int rc = check_call(p, kdata, gs, bins ? bins : (const void*)omega, batch, coils, smaps_batch, q, m, who);
    if (rc) return rc;
    PDU_REQUIRE(q != nullptr, "%s: q is null", who);
    PDU_REQUIRE((flags & ~(PDU_NUFFT_IMAGE_SPLIT | PDU_NUFFT_KDATA_SPLIT)) == 0, "%s: unknown flags %d", who, flags);
    PDU_CHECK_DEVICE(who);
    const int q_split = (flags & PDU_NUFFT_IMAGE_SPLIT) ? 1 : 0, per_batch = smaps_batch == 1 ? 0 : 1;
    if (bins) {
        if (!fused_supported(p)) {
            set_error("%s: grid %d x %d (J = %d) has no fused path; pass bins = NULL", who, p->k0, p->k1, p->J);
            return PDU_EUNSUPPORTED;
        }
        rc = check_workspace(who, workspace, workspace_bytes, fused_workspace_bytes(p, batch * coils, m), true, PDU_ENOMEM);
        if (rc) return rc;
        const SmapsGrad sg{(float2*)gs, q, batch, per_batch, q_split, accumulate ? 1 : 0, 1.f};
        return fused_adjoint(p, kdata, nullptr, nullptr, kweight, batch, coils, 1, m, scale, bins, flags, workspace,
                             (cudaStream_t)stream, &sg);
    }
    // the plain-omega / CSR paths take complex64 kdata without weights, as pdu_nufft_adj_csr_c64 does
    PDU_REQUIRE(!kweight && !(flags & PDU_NUFFT_KDATA_SPLIT), "%s: kweight and split kdata need the row-binned path (bins)", who);
    const int cb = nufft_batch_chunk(p, batch, coils);
    rc = check_workspace(who, workspace, workspace_bytes, pdu_nufft_workspace_bytes(p, cb * coils), false, PDU_ENOMEM);
    if (rc) return rc;
    const long plane = (long)p->n0 * p->n1;
    return for_each_chunk(batch, cb, [&](int b0, int nb) {
        // a shared map's sum continues from chunk to chunk
        const SmapsGrad sg{(float2*)gs + (per_batch ? (long)b0 * coils * plane : 0), q + (long)b0 * 2 * plane, nb, per_batch,
                           q_split, (accumulate || (!per_batch && b0 > 0)) ? 1 : 0, 1.f};
        return nufft_adj_chunk(p, (const float2*)kdata + (long)b0 * coils * m, nullptr, omega, nullptr, nb, coils, 1, m, scale,
                               (float2*)workspace, csr, (cudaStream_t)stream, &sg);
    });
}

int pdu_complex_from_split_f32(const float* split, float* out, const float* weight, long planes, long n, pdu_stream_t stream) {
    PDU_REQUIRE(split && out && planes > 0 && n > 0, "pdu_complex_from_split_f32: null pointer or empty tensor");
    layout_to_complex_kernel<<<stream_grid(planes * n), 256, 0, (cudaStream_t)stream>>>(split, (float2*)out, weight, n, planes * n);
    PDU_LAUNCHED();
    return PDU_OK;
}

int pdu_split_from_complex_f32(const float* in, float* split, long planes, long n, pdu_stream_t stream) {
    PDU_REQUIRE(split && in && planes > 0 && n > 0, "pdu_split_from_complex_f32: null pointer or empty tensor");
    layout_to_split_kernel<<<stream_grid(planes * n), 256, 0, (cudaStream_t)stream>>>((const float2*)in, split, n, planes * n);
    PDU_LAUNCHED();
    return PDU_OK;
}

int pdu_nufft_interp_fwd_c64(pdu_nufft_plan_t* p, const float* grid, float* kdata, const float* omega, int planes,
                             long m, pdu_stream_t stream) {
    int rc = check_call(p, grid, kdata, omega, planes, 1, 1, nullptr, m, "pdu_nufft_interp_fwd_c64");
    if (rc) return rc;
    return launch_interp_fwd(p, (const float2*)grid, (float2*)kdata, omega, planes, m, 1.f, (cudaStream_t)stream);
}

int pdu_nufft_interp_adj_c64(pdu_nufft_plan_t* p, const float* kdata, float* grid, const float* omega, int planes,
                             long m, pdu_stream_t stream) {
    int rc = check_call(p, kdata, grid, omega, planes, 1, 1, nullptr, m, "pdu_nufft_interp_adj_c64");
    if (rc) return rc;
    return launch_interp_adj(p, (const float2*)kdata, (float2*)grid, omega, planes, m, (cudaStream_t)stream);
}

int pdu_toep_plan_create(pdu_nufft_plan_t** plan, int n0, int n1) {
    PDU_REQUIRE(plan != nullptr, "pdu_toep_plan_create: plan is null");
    *plan = nullptr;
    PDU_REQUIRE(n0 > 0 && n1 > 0 && n0 <= 2048 && n1 <= 2048, "pdu_toep_plan_create: need 0 < n <= 2048 per axis (got %d x %d)", n0, n1);
    const int k0 = 2 * n0, k1 = 2 * n1;
    PfftPlan pf0, pf1;
    // the kernel build's FFT and the generic apply run the run-time-radix passes: 2, 3, 5 sizes whose rows (4 per CTA)
    // and columns (2 per CTA) fit shared memory; the fast path's sizes are among them
    if (!pfft_factor(k0, &pf0) || !pfft_factor(k1, &pf1) || pf_smem_bytes(PF_SEQ_ROWS, k1) > 200 * 1024 ||
        pf_smem_bytes(2, k0) > 200 * 1024) {
        set_error("pdu_toep_plan_create: no Toeplitz path for %d x %d (the embedding grid %d x %d must factor into 2, 3, 5 "
                  "and fit the shared-memory FFT)", n0, n1, k0, k1);
        return PDU_EUNSUPPORTED;
    }
    return plan_create(plan, n0, n1, k0, k1, "pdu_toep_plan_create", [&](pdu_nufft_plan* p) {
        p->pfft_ok = true;
        p->pf0 = pf0;
        p->pf1 = pf1;
        p->toep = true;
        const std::vector<float> ones((size_t)std::max(k0, k1), 1.f);   // unit apodisation (every entry a row / column pass may read)
        cudaError_t e = upload(&p->d_s0, ones.data(), (size_t)k0);
        if (e == cudaSuccess) e = upload(&p->d_s1, ones.data(), (size_t)k1);
        if (e == cudaSuccess) e = upload_twiddles(p);
        return e;
    });
}

size_t pdu_toep_workspace_bytes(const pdu_nufft_plan_t* p, int planes) {
    if (!p || !p->toep || planes <= 0) return 0;
    return (size_t)planes * tz_plane_bytes(p);
}

int pdu_toep_kernel_c64(pdu_nufft_plan_t* p, const float* q1, const float* q2, float* kernel, int kernels, float scale,
                        void* ws, size_t ws_bytes, pdu_stream_t stream) {
    const char* who = "pdu_toep_kernel_c64";
    int rc = check_toep_call(p, q1 && q2 && kernel, 1, 1, 1, nullptr, 1, who);     // no batch; the kernel count is checked next
    if (rc) return rc;
    PDU_REQUIRE(kernels > 0 && kernels <= 65535, "%s: kernels must be in 1..65535", who);
    rc = check_workspace(who, ws, ws_bytes, (size_t)kernels * p->k0 * p->k1 * sizeof(float2), false, PDU_ENOMEM);
    if (rc) return rc;
    PDU_CHECK_DEVICE(who);
    cudaStream_t st = (cudaStream_t)stream;
    const long total = (long)kernels * p->k0 * p->k1;
    tz_assemble_kernel<<<stream_grid(total), 256, 0, st>>>((const float2*)q1, (const float2*)q2, (float2*)kernel, p->n0, p->n1,
                                                           scale, total);
    PDU_LAUNCHED();
    if (tz_cols_seq8(p)) return tz_kernel_fft<PF_SEQ_COLS>(p, (float2*)kernel, (float2*)ws, kernels, st);
    return tz_kernel_fft<2>(p, (float2*)kernel, (float2*)ws, kernels, st);
}

int pdu_toep_apply_c64(pdu_nufft_plan_t* p, const float* image, float* out, const float* kernel, int kernel_batch,
                       const float* smaps, int batch, int coils, int smaps_batch, int conj_kernel, void* ws, size_t ws_bytes,
                       pdu_stream_t stream) {
    const char* who = "pdu_toep_apply_c64";
    int rc = check_toep_call(p, image && out && kernel, batch, coils, kernel_batch, smaps, smaps_batch, who);
    if (rc) return rc;
    const int cb = tz_batch_chunk(p, batch, coils);
    rc = check_workspace(who, ws, ws_bytes, pdu_toep_workspace_bytes(p, cb * coils), false, PDU_ENOMEM);
    if (rc) return rc;
    PDU_CHECK_DEVICE(who);
    const long plane = (long)p->n0 * p->n1, cells = (long)p->k0 * p->k1;
    const long img_b = (smaps ? 1 : coils) * plane, out_b = img_b, smap_b = smaps_batch == 1 ? 0 : coils * plane;
    return for_each_chunk(batch, cb, [&](int b0, int nb) {
        return tz_apply_chunk(p, (const float2*)image + b0 * img_b, (float2*)out + b0 * out_b,
                              (const float2*)kernel + (kernel_batch == 1 ? 0 : b0 * cells), kernel_batch == 1 ? 1 : nb,
                              smaps ? (const float2*)smaps + b0 * smap_b : nullptr, nb, coils, smaps_batch == 1 ? 1 : nb,
                              conj_kernel ? 1 : 0, (float2*)ws, (cudaStream_t)stream);
    });
}

int pdu_toep_smaps_grad_c64(pdu_nufft_plan_t* p, const float* x, const float* g, float* gs, const float* kernel,
                            int kernel_batch, const float* smaps, int batch, int coils, int smaps_batch, int conj_kernel,
                            float out_scale, int accumulate, void* ws, size_t ws_bytes, pdu_stream_t stream) {
    const char* who = "pdu_toep_smaps_grad_c64";
    int rc = check_toep_call(p, x && g && gs && kernel && smaps, batch, coils, kernel_batch, smaps, smaps_batch, who);
    if (rc) return rc;
    const int cb = tz_batch_chunk(p, batch, coils);
    rc = check_workspace(who, ws, ws_bytes, pdu_toep_workspace_bytes(p, cb * coils), false, PDU_ENOMEM);
    if (rc) return rc;
    PDU_CHECK_DEVICE(who);
    const long plane = (long)p->n0 * p->n1, cells = (long)p->k0 * p->k1;
    const int per_batch = smaps_batch == 1 ? 0 : 1;
    const long smap_b = per_batch ? coils * plane : 0;
    return for_each_chunk(batch, cb, [&](int b0, int nb) -> int {
        // term 0: T(S_c x_b) conj(g_b); term 1: T^H(S_c g_b) conj(x_b), added on top
        for (int term = 0; term < 2; ++term) {
            const float* image = term ? g : x;
            const float* q = term ? x : g;
            const int acc = (accumulate || term == 1 || (!per_batch && b0 > 0)) ? 1 : 0;
            const SmapsGrad sg{(float2*)gs + b0 * smap_b, q + 2 * b0 * plane, nb, per_batch, 0, acc, out_scale};
            const int rc = tz_apply_chunk(p, (const float2*)image + b0 * plane, nullptr,
                                          (const float2*)kernel + (kernel_batch == 1 ? 0 : b0 * cells), kernel_batch == 1 ? 1 : nb,
                                          (const float2*)smaps + b0 * smap_b, nb, coils, per_batch ? nb : 1,
                                          (conj_kernel != 0) != (term == 1) ? 1 : 0, (float2*)ws, (cudaStream_t)stream, nullptr, &sg);
            if (rc) return rc;
        }
        return PDU_OK;
    });
}

size_t pdu_toep_cg_workspace_bytes(const pdu_nufft_plan_t* p, int batch, int coils, int has_smaps) {
    if (!p || !p->toep || batch <= 0 || coils <= 0 || coils > 65535) return 0;
    return cg_layout(p, tz_batch_chunk(p, batch, coils), coils, has_smaps != 0, nullptr).bytes;
}

int pdu_toep_cg_c64(pdu_nufft_plan_t* p, const float* b, const float* x0, float* x, const float* kernel, int kernel_batch,
                    const float* smaps, int batch, int coils, int smaps_batch, const float* lam, int lam_count, int max_iter,
                    float tol, int conj_kernel, void* ws, size_t ws_bytes, pdu_stream_t stream) {
    const char* who = "pdu_toep_cg_c64";
    int rc = check_toep_call(p, b && x && kernel, batch, coils, kernel_batch, smaps, smaps_batch, who);
    if (rc) return rc;
    PDU_REQUIRE(lam_count == 1 || lam_count == batch, "%s: lam_count must be 1 or batch (got %d)", who, lam_count);
    PDU_REQUIRE(max_iter >= 0, "%s: max_iter must be >= 0 (got %d)", who, max_iter);
    PDU_REQUIRE(tol >= 0.f, "%s: tol must be >= 0", who);
    const int cb = tz_batch_chunk(p, batch, coils);
    const CgWs w = cg_layout(p, cb, coils, smaps != nullptr, ws);
    rc = check_workspace(who, ws, ws_bytes, w.bytes, false, PDU_EINVAL);
    if (rc) return rc;
    PDU_CHECK_DEVICE(who);
    const long plane = (long)p->n0 * p->n1, cells = (long)p->k0 * p->k1;
    const long img_b = (smaps ? 1 : coils) * plane, smap_b = smaps_batch == 1 ? 0 : coils * plane;
    const int lam_div = lam_count == 1 ? 0 : (smaps ? 1 : coils);   // system -> batch element within a chunk
    const double tol2 = (double)tol * (double)tol;
    return for_each_chunk(batch, cb, [&](int b0, int nb) {
        return tz_cg_chunk(p, (const float2*)b + b0 * img_b, x0 ? (const float2*)x0 + b0 * img_b : nullptr,
                           (float2*)x + b0 * img_b, (const float2*)kernel + (kernel_batch == 1 ? 0 : b0 * cells),
                           kernel_batch == 1 ? 1 : nb, smaps ? (const float2*)smaps + b0 * smap_b : nullptr, nb, coils,
                           smaps_batch == 1 ? 1 : nb, lam ? lam + (lam_count == 1 ? 0 : b0) : nullptr, lam_div, max_iter,
                           tol2, conj_kernel ? 1 : 0, w, (cudaStream_t)stream);
    });
}

}  // extern "C"
