// Register-resident pruned FFT for the oversampled-grid sizes of the BASELINE shapes (grid = 2 x image):
//   K = 256 (128^2 images), 512 (256^2), 640 (320^2), 1024 (512^2), 2048 (1024^2)
// compile-time radices 8 x 8 x (K / 64) (2048: 8 x 16 x 16): three butterflies per thread with two shared-memory
// exchanges in between.  The first butterfly reads its inputs through a caller-supplied functor (global memory, or the
// sequence's own shared buffer when an interpolation stage has just filled it) and the last one hands its
// outputs to another functor, so a sequence crosses shared memory twice (pfft.cuh's generic run-time-radix
// passes: five times) and there is no index arithmetic that is not a shift or a compile-time constant.
//
// Stockham autosort, natural order in and out; pass with radix R, Ns = product of earlier radices:
//   butterfly j (0 <= j < K/R):  k = j mod Ns, hi = j / Ns
//     v[r] = in[j + r K/R] * W_K^(r k K/(Ns R)),  v = DFT_R(v),  out[hi Ns R + k + r Ns] = v[r]
// Pruning: HALF_IN  -- inputs K/2 .. K-1 are zero (zero padding of the image), never loaded;
//          HALF_OUT -- outputs K/2 .. K-1 are not wanted (the crop of the adjoint), never stored.
#pragma once
#include <type_traits>

#include "pfft.cuh"

namespace pdu {

template <int K>
struct FastFft {
    static constexpr bool ok = (K == 256 || K == 512 || K == 640 || K == 1024 || K == 2048);
    static constexpr int TPS = K / 8;                 // threads per sequence (one radix-8 butterfly each in the first pass)
    static constexpr int R2 = K == 2048 ? 16 : 8;     // radix of the second pass
    static constexpr int R3 = K / (8 * R2);           // radix of the last pass: 4, 8, 10, 16 (8 R2 butterflies)
    static constexpr int NS3 = 8 * R2;                // butterflies of the last pass = stride of its elements
    // Padding: one slot every 2^PS elements, chosen per thread layout (measured, ncu r01):
    //  PS = 3 (column kernels: a half-warp is 8 neighbouring sequences x 2 butterflies) -- element 8 t + r sits at
    //    9 t + r; with the pitch == 2 (mod 16) float2 every access of the three passes is conflict free;
    //  PS = 4 (row kernels: a half-warp is 16 consecutive butterflies of one sequence) -- the unit-stride loads of
    //    passes 2 and 3 then never straddle a padding slot (PS = 3 made 16 lanes span 18 slots: a 2-way conflict on
    //    every load), the stride-8 stores of pass 1 stay conflict free, only the pass-2 stores keep a 2-way conflict.
    template <int PS>
    __host__ __device__ static constexpr int pitch() {      // PS == 4: room for the second exchange's 4 slots per 64 elements
        return (K + (K >> PS) + (PS == 4 ? 4 * (K / 64) : 0) + 13) / 16 * 16 + 2;
    }
};
static inline bool fast_fft_size(int K) { return K == 256 || K == 512 || K == 640 || K == 1024 || K == 2048; }
// f(std::integral_constant<int, K>{}) for the run-time size K, one of fast_fft_size's; returns what f returns
template <typename Fn>
static int with_fast_fft_size(int K, Fn&& f) {
    switch (K) {
        case 256: return f(std::integral_constant<int, 256>{});
        case 512: return f(std::integral_constant<int, 512>{});
        case 640: return f(std::integral_constant<int, 640>{});
        case 1024: return f(std::integral_constant<int, 1024>{});
        default: return f(std::integral_constant<int, 2048>{});
    }
}
template <int PS>
__device__ __forceinline__ int ff_pos(int e) { return e + (e >> PS); }

template <bool INV>
__device__ __forceinline__ float2 ff_tw(const float2* __restrict__ tw, int i) {
    float2 w = tw[i];
    if (INV) w.y = -w.y;
    return w;
}

template <bool INV>
__device__ __forceinline__ void ff_r5(float2* x) {
    constexpr float C1 = 0.30901699437494742f, C2 = -0.80901699437494742f;
    constexpr float S1 = 0.95105651629515357f, S2 = 0.58778525229247313f;
    const float2 a1 = pf_add(x[1], x[4]), a2 = pf_add(x[2], x[3]);
    const float2 b1 = pf_sub(x[1], x[4]), b2 = pf_sub(x[2], x[3]);
    const float2 t1 = make_float2(x[0].x + C1 * a1.x + C2 * a2.x, x[0].y + C1 * a1.y + C2 * a2.y);
    const float2 t2 = make_float2(x[0].x + C2 * a1.x + C1 * a2.x, x[0].y + C2 * a1.y + C1 * a2.y);
    const float2 u1 = pf_rot<INV>(make_float2(S1 * b1.x + S2 * b2.x, S1 * b1.y + S2 * b2.y));
    const float2 u2 = pf_rot<INV>(make_float2(S2 * b1.x - S1 * b2.x, S2 * b1.y - S1 * b2.y));
    x[0] = pf_add(x[0], pf_add(a1, a2));
    x[1] = pf_add(t1, u1);
    x[4] = pf_sub(t1, u1);
    x[2] = pf_add(t2, u2);
    x[3] = pf_sub(t2, u2);
}

template <bool INV>
__device__ __forceinline__ void ff_r10(float2* v) {
    float2 e[5] = {v[0], v[2], v[4], v[6], v[8]}, o[5] = {v[1], v[3], v[5], v[7], v[9]};
    ff_r5<INV>(e);
    ff_r5<INV>(o);
    // W10^q = exp(-+ 2 pi i q / 10)
    constexpr float C[5] = {1.f, 0.80901699437494742f, 0.30901699437494742f, -0.30901699437494742f, -0.80901699437494742f};
    constexpr float S[5] = {0.f, 0.58778525229247313f, 0.95105651629515357f, 0.95105651629515357f, 0.58778525229247313f};
#pragma unroll
    for (int q = 0; q < 5; ++q) {
        const float2 w = make_float2(C[q], INV ? S[q] : -S[q]);
        const float2 t = q == 0 ? o[0] : pf_mul(o[q], w);
        v[q] = pf_add(e[q], t);
        v[q + 5] = pf_sub(e[q], t);
    }
}

// radix 16 = 4 x 4 and radix 32 = 4 x 8 inside one thread's registers (Cooley-Tukey, n = n1 + 4 n2, k = R2 k1 + k2):
// four DFT_R2 over the stride-4 subsequences, twiddles W_R^(n1 k2), then R2 DFT_4 across the subsequences.
template <bool INV, int R>
__device__ __forceinline__ void ff_r4xN(float2* v) {
    static_assert(R == 16 || R == 32, "radix 16 or 32");
    constexpr int R2 = R / 4;
    // exp(+2 pi i j / 32), j = 0 .. 31
    constexpr float C32[32] = {1.f, 0.98078528040323043f, 0.92387953251128674f, 0.83146961230254524f, 0.70710678118654757f, 0.55557023301960229f, 0.38268343236508984f, 0.19509032201612833f, 0.f, -0.19509032201612819f, -0.38268343236508973f, -0.55557023301960196f, -0.70710678118654746f, -0.83146961230254535f, -0.92387953251128674f, -0.98078528040323043f, -1.f, -0.98078528040323043f, -0.92387953251128685f, -0.83146961230254546f, -0.70710678118654768f, -0.55557023301960218f, -0.38268343236509034f, -0.19509032201612866f, 0.f, 0.1950903220161283f, 0.38268343236509f, 0.55557023301960184f, 0.70710678118654735f, 0.83146961230254524f, 0.92387953251128652f, 0.98078528040323032f};
    constexpr float S32[32] = {0.f, 0.19509032201612825f, 0.38268343236508978f, 0.55557023301960218f, 0.70710678118654746f, 0.83146961230254524f, 0.92387953251128674f, 0.98078528040323043f, 1.f, 0.98078528040323043f, 0.92387953251128674f, 0.83146961230254546f, 0.70710678118654757f, 0.55557023301960218f, 0.38268343236508989f, 0.19509032201612861f, 0.f, -0.19509032201612836f, -0.38268343236508967f, -0.55557023301960196f, -0.70710678118654746f, -0.83146961230254524f, -0.92387953251128652f, -0.98078528040323032f, -1.f, -0.98078528040323043f, -0.92387953251128663f, -0.83146961230254546f, -0.70710678118654768f, -0.55557023301960218f, -0.38268343236509039f, -0.19509032201612872f};
    float2 y[4][R2];
#pragma unroll
    for (int n1 = 0; n1 < 4; ++n1) {
#pragma unroll
        for (int n2 = 0; n2 < R2; ++n2) y[n1][n2] = v[n1 + 4 * n2];
        if constexpr (R2 == 4) pf_r4<INV>(y[n1]);
        else pf_r8<INV>(y[n1]);
    }
#pragma unroll
    for (int k2 = 0; k2 < R2; ++k2) {
        float2 z[4];
        z[0] = y[0][k2];
#pragma unroll
        for (int n1 = 1; n1 < 4; ++n1) {
            constexpr int STEP = 32 / R;
            const int j = (n1 * k2 * STEP) & 31;
            const float2 w = make_float2(C32[j], INV ? S32[j] : -S32[j]);
            z[n1] = (n1 * k2 == 0) ? y[n1][k2] : pf_mul(y[n1][k2], w);
        }
        pf_r4<INV>(z);
#pragma unroll
        for (int k1 = 0; k1 < 4; ++k1) v[R2 * k1 + k2] = z[k1];
    }
}

template <bool INV, int R>
__device__ __forceinline__ void ff_small(float2* v) {
    if constexpr (R == 4) pf_r4<INV>(v);
    else if constexpr (R == 8) pf_r8<INV>(v);
    else if constexpr (R == 10) ff_r10<INV>(v);
    else ff_r4xN<INV, R>(v);
}

// One sequence of length K held by the TPS threads t = 0 .. TPS-1 of a CTA (every thread of the CTA must call
// this: it synchronises).  buf = this sequence's pitch<PS>() float2 of shared memory, tw = the K-entry table
// exp(-2 pi i m / K) in shared memory.  ld(r) returns input element t + r TPS (r = 0 .. 7, a compile-time constant after
// unrolling); st(j, r, v) consumes output element j + r NS3 (NS3 = 8 R2; j = t, or t + TPS when TPS < NS3): the caller's
// functors form base(t) + r * constant addresses as well (no 64-bit index arithmetic per element).
// LD_BUF: ld reads this CTA's `buf`s (an interpolation stage filled them) -- every load must be complete before
//   the first exchange store;  ST_BUF: st writes the `buf`s -- every last-pass load must be complete before it.
//
// Shared-memory addressing (r02): the padded position of an element is e + (e >> PS), and every access of the three
// passes is  base(t) + r * constant  -- because the strides (TPS, 8, 8 R2 and K / R2) are multiples of 2^PS or smaller
// than it in a way that commutes with the shift (derivations at each pass).  The first version called ff_pos() per
// access and the compiler could not see through the shift: 39 % of the instructions of a transform were integer address
// arithmetic (SASS histogram of fz_cols_fwd_kernel<640, 8>: 326 LEA / IMAD / IADD3 / LOP3 / SHF against 302 FP).
// twiddles w^r, r = 1 .. R-1, from w^1 by products of depth log2(r) (w[r] = w[r / 2] w[r - r / 2]): trades R - 2
// shared-memory loads for 4 (R - 2) FMAs where the shared-memory pipe, not instruction issue, is the busier one
template <int R>
__device__ __forceinline__ void ff_tw_powers(float2 w1, float2* w) {
    w[1] = w1;
#pragma unroll
    for (int r = 2; r < R; ++r) w[r] = pf_mul(w[r / 2], w[r - r / 2]);
}

template <int K, int PS, bool INV, bool HALF_IN, bool HALF_OUT, bool LD_BUF = false, bool ST_BUF = false, bool TWREC = false, class LD, class ST>
__device__ __forceinline__ void ff_transform(float2* __restrict__ buf, const float2* __restrict__ tw, int t, LD ld, ST st) {
    using F = FastFft<K>;
    constexpr int TPS = F::TPS, R2 = F::R2, R3 = F::R3, NB2 = K / R2, NS3 = 8 * R2;
    constexpr int PADM = (1 << PS);
    static_assert(PS == 3 || PS == 4, "padding every 8 or 16 elements");
    static_assert(TPS % PADM == 0 && NB2 % PADM == 0 && NS3 % PADM == 0, "strides commute with the padding shift");
    float2 v[8];
    // pass 1: radix 8, Ns = 1.  loads: elements t + r TPS (through the functor)
#pragma unroll
    for (int r = 0; r < 8; ++r) v[r] = (HALF_IN && r >= 4) ? make_float2(0.f, 0.f) : ld(r);
    if (LD_BUF) __syncthreads();
    pf_r8<INV>(v);
    {   // stores: elements 8 t + r, r < 8: (8 t + r) >> PS == (8 t) >> PS  =>  position = pos(8 t) + r
        float2* p1 = buf + (8 * t + ((8 * t) >> PS));
#pragma unroll
        for (int r = 0; r < 8; ++r) p1[r] = v[r];
    }
    __syncthreads();
    // pass 2: radix R2, Ns = 8; K / R2 butterflies.  loads: elements t + r NB2, NB2 a multiple of 2^PS
    //   => position = pos(t) + r (NB2 + NB2 / 2^PS)
    float2 w2[R2];
    const float2* p2 = buf + (t + (t >> PS));
    if (t < NB2) {
#pragma unroll
        for (int r = 0; r < R2; ++r) w2[r] = p2[r * (NB2 + NB2 / PADM)];
    }
    __syncthreads();
    if (t < NB2) {
        const int k = t & 7;
        if (TWREC) {
            float2 wp[R2];
            ff_tw_powers<R2>(ff_tw<INV>(tw, k * (K / NS3)), wp);
#pragma unroll
            for (int r = 1; r < R2; ++r) w2[r] = pf_mul(w2[r], wp[r]);
        } else {
#pragma unroll
            for (int r = 1; r < R2; ++r) w2[r] = pf_mul(w2[r], ff_tw<INV>(tw, r * k * (K / NS3)));
        }
        ff_small<INV, R2>(w2);
        // stores: elements o0 + 8 r with o0 = (t >> 3) NS3 + k, k < 8, NS3 a multiple of 2^PS:
        //   PS == 3: (o0 + 8 r) >> 3 == (o0 >> 3) + r        => position = pos(o0) + 9 r
        //   PS == 4: this exchange (pass 2 -> pass 3) has its own layout, position = e + (e >> 4) + 4 (e >> 6).  With
        //     e + (e >> 4) alone the two octets of butterflies a half-warp holds store 64 elements = 68 slots apart,
        //     i.e. 4 (mod 16) float2: a 2-way bank conflict on every pass-2 store (ncu r02: 9 % of the shared-memory
        //     wavefronts of fz_rows_fwd_kernel); 4 more slots per 64 elements make it 72 = 8 (mod 16).  The first
        //     exchange keeps e + (e >> 4): its stride-8 stores need exactly that.
        const int o0 = (t >> 3) * NS3 + k;
        float2* p2s = buf + (PS == 3 ? o0 + (o0 >> 3) : (t >> 3) * (NS3 + NS3 / 16 + 4 * (NS3 / 64)) + k);
#pragma unroll
        for (int r = 0; r < R2; ++r) p2s[PS == 3 ? 9 * r : 8 * r + (r >> 1) + 4 * (r >> 3)] = w2[r];
    }
    __syncthreads();
    // pass 3: radix R3, Ns = 8 R2; NS3 butterflies (TPS = 32: two per thread).  loads: elements j + r NS3
    //   => position = pos(j) + r (NS3 + NS3 / 2^PS)   (PS == 4: the second exchange's layout, see above)
    constexpr int PER = TPS >= NS3 ? 1 : NS3 / TPS;
    constexpr int S3 = PS == 3 ? NS3 + NS3 / PADM : NS3 + NS3 / 16 + 4 * (NS3 / 64);
    if (!ST_BUF) {
#pragma unroll
        for (int i = 0; i < PER; ++i) {
            const int j = t + i * TPS;
            if (j < NS3) {
                float2 u[R3];
                const float2* p3 = buf + (PS == 3 ? j + (j >> 3) : j + (j >> 4) + 4 * (j >> 6));
#pragma unroll
                for (int r = 0; r < R3; ++r) u[r] = p3[r * S3];
                if (TWREC) {
                    float2 wp[R3];
                    ff_tw_powers<R3>(ff_tw<INV>(tw, j), wp);
#pragma unroll
                    for (int r = 1; r < R3; ++r) u[r] = pf_mul(u[r], wp[r]);
                } else {
#pragma unroll
                    for (int r = 1; r < R3; ++r) u[r] = pf_mul(u[r], ff_tw<INV>(tw, r * j));
                }
                ff_small<INV, R3>(u);
#pragma unroll
                for (int r = 0; r < R3; ++r)
                    if (!HALF_OUT || r < R3 / 2) st(j, r, u[r]);
            }
        }
    } else {
        float2 u[PER][R3];
#pragma unroll
        for (int i = 0; i < PER; ++i) {
            const int j = t + i * TPS;
            if (j < NS3) {
                const float2* p3 = buf + (PS == 3 ? j + (j >> 3) : j + (j >> 4) + 4 * (j >> 6));
#pragma unroll
                for (int r = 0; r < R3; ++r) u[i][r] = p3[r * S3];
            }
        }
        __syncthreads();
#pragma unroll
        for (int i = 0; i < PER; ++i) {
            const int j = t + i * TPS;
            if (j < NS3) {
                if (TWREC) {
                    float2 wp[R3];
                    ff_tw_powers<R3>(ff_tw<INV>(tw, j), wp);
#pragma unroll
                    for (int r = 1; r < R3; ++r) u[i][r] = pf_mul(u[i][r], wp[r]);
                } else {
#pragma unroll
                    for (int r = 1; r < R3; ++r) u[i][r] = pf_mul(u[i][r], ff_tw<INV>(tw, r * j));
                }
                ff_small<INV, R3>(u[i]);
#pragma unroll
                for (int r = 0; r < R3; ++r)
                    if (!HALF_OUT || r < R3 / 2) st(j, r, u[i][r]);
            }
        }
    }
}

}  // namespace pdu
