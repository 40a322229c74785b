// Radial-MRI NUFFT, fused form for the BASELINE grids (K = 2N in {256, 512, 640, 1024, 2048}, J = 6):
// the Kaiser-Bessel interpolation is SEPARABLE, so it is split along the two grid axes and each half is fused
// into the FFT pass that has the matching data on chip.  The oversampled K x K grid is never written to memory.
//
//   forward   fz_cols_fwd_kernel     image (x apodisation x coil map) -> pruned column FFT           -> T  [planes][K][N]
//             fz_rows_fwd_kernel     one grid ROW x 8 planes per CTA: pruned row FFT into shared memory, then for every
//                                    (sample, row-tap) entry binned to this row the 6-tap interpolation ALONG the row
//                                                                                                    -> P  [planes][6][M]
//             fz_combine_kernel      y[m] = scale * sum_a (phase c0[a])[m] P[a][m]  (6 coalesced reads) -> kdata
//   adjoint   fz_rows_adj_kernel     one grid row x 8 planes per CTA: every cell of the row GATHERS its entries
//                                    (sorted by column, so a cell's contributors are one contiguous range) from
//                                    shared-memory staged samples, then the pruned inverse row FFT     -> T  [planes][K][N]
//             fz_cols_adj_kernel     pruned inverse column FFT, crop x apodisation (x conj coil map, coil sum) -> image
//
// Against r01's path (row FFT, column FFT, 36-tap gather from the K x K grid in L2 / sorted CSR gather, row IFFT,
// column IFFT, crop) this removes the grid's write + read (2 x 210 MB at the configs[3] share), turns the 36 L2 taps
// per sample into 6 shared-memory taps + 6 coalesced reads, and needs no atomics in either direction (the adjoint is
// bit-reproducible).  The per-trajectory "row bins" are built once (pdu_nufft_bins_build: one radix sort) and reused by
// every unrolled iteration, like torchkbnufft's precomputed interpolation matrices.
//
// Rounding: table entries, grid offsets and phases are the same float32 values as on the generic path (axis_taps,
// shift_phase); only the summation order differs (row taps first, then the six rows).
#include <cub/device/device_radix_sort.cuh>

#include <algorithm>

#include "nufft_common.cuh"

namespace pdu {

constexpr int FZ_J = 6;
constexpr int FZ_EC = 512;        // entries staged at a time by the adjoint row kernel (most rows fit one chunk)
constexpr unsigned FZ_MAGIC = 0x5a42494eu;      // "NIBZ"

// one (sample, row tap) entry, sorted by (grid row, first column): 64 bytes
struct __align__(16) BinRec {
    int u;            // first of the J consecutive (wrapping) columns the sample touches
    int id;           // m * J + a
    float2 wadj;      // conj(phase[m] * c0[m][a]): the adjoint's row weight
    float2 c1[FZ_J];  // column coefficients of the sample
};
static_assert(sizeof(BinRec) == 64, "entry record is one 64-byte line half");

struct BinsView {
    int* hdr;            // [16]: magic, M (lo, hi), K0, K1, J, n_entries, entries of the heaviest row
    int* key_ptr;        // [K0 K1 + 1]: first sorted entry whose (row K1 + column) key is >= i
    int4* row_order;     // [K0]: (row, first entry, end entry, 0) by decreasing entry count -- heavy rows are scheduled
                         // first, and a CTA finds its row and entry range with one 16-byte load
    unsigned short* cell_order;   // [K0][K1]: the cells of every row by decreasing contributor count (adjoint gather)
    BinRec* rec;         // [M J]
    float2* w0;          // [J][M]: phase[m] * c0[m][a], the forward's row weights
    size_t persist;
    // build scratch
    unsigned* key_in;
    unsigned* id_in;
    unsigned* key_out;
    unsigned* id_out;
    float2* c1s;         // [M][J]
    void* cub_tmp;
    size_t cub_bytes;
    size_t total;
};

static BinsView bins_layout(const pdu_nufft_plan* p, long M, void* base, bool with_scratch) {
    const size_t n = (size_t)M * FZ_J, cells = (size_t)p->k0 * p->k1;
    BinsView v;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += align256(bytes); return (char*)base + o; };
    v.hdr = (int*)take(64);
    v.key_ptr = (int*)take((cells + 1) * 4);
    v.row_order = (int4*)take((size_t)p->k0 * 16);
    v.cell_order = (unsigned short*)take(cells * 2);
    v.rec = (BinRec*)take(n * sizeof(BinRec));
    v.w0 = (float2*)take(n * 8);
    v.persist = off;
    v.key_in = (unsigned*)take(n * 4);
    v.id_in = (unsigned*)take(n * 4);
    v.key_out = (unsigned*)take(n * 4);
    v.id_out = (unsigned*)take(n * 4);
    v.c1s = (float2*)take(n * 8);
    v.cub_bytes = 0;
    v.cub_tmp = nullptr;
    v.total = off;
    if (!with_scratch) return v;
    cub::DeviceRadixSort::SortPairs(nullptr, v.cub_bytes, (const unsigned*)nullptr, (unsigned*)nullptr, (const unsigned*)nullptr,
                                    (unsigned*)nullptr, (int)n);
    v.cub_tmp = take(v.cub_bytes);
    v.total = off;
    return v;
}

bool fused_supported(const pdu_nufft_plan* p) {
    return p->k0 == p->k1 && p->k0 == 2 * p->n0 && p->k1 == 2 * p->n1 && fast_fft_size(p->k0) && p->J == FZ_J && p->d_w0 && p->d_w1;
}

// ------------------------------------------------------------------ building the row bins
__global__ void __launch_bounds__(128)
    bin_entries_kernel(const float* __restrict__ omega, const float2* __restrict__ t0, const float2* __restrict__ t1, NufftDims d,
                       long M, unsigned* __restrict__ key, unsigned* __restrict__ id, float2* __restrict__ w0,
                       float2* __restrict__ c1s) {
    const long m = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= M) return;
    const float om0 = __ldg(omega + m), om1 = __ldg(omega + M + m);
    int g0[FZ_J], g1[FZ_J];
    float2 c0[FZ_J], c1[FZ_J];
    axis_taps<FZ_J>(om0, d.gam0, d.k0, d.J, d.L, t0, g0, c0);
    axis_taps<FZ_J>(om1, d.gam1, d.k1, d.J, d.L, t1, g1, c1);
    const float2 ph = shift_phase(om0, om1, d.shift0, d.shift1);
#pragma unroll
    for (int a = 0; a < FZ_J; ++a) {
        key[m * FZ_J + a] = (unsigned)(g0[a] * d.k1 + g1[0]);
        id[m * FZ_J + a] = (unsigned)(m * FZ_J + a);
        w0[(long)a * M + m] = cmul(ph, c0[a]);
        c1s[m * FZ_J + a] = c1[a];
    }
}

__global__ void __launch_bounds__(256)
    bin_finish_kernel(const unsigned* __restrict__ key_sorted, const unsigned* __restrict__ id_sorted, const float2* __restrict__ w0,
                      const float2* __restrict__ c1s, int* __restrict__ key_ptr, BinRec* __restrict__ rec, long n, long cells, long M,
                      int K1) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const unsigned e = id_sorted[i];
        const long m = e / FZ_J;
        const int a = (int)(e - m * FZ_J);
        BinRec r;
        r.u = (int)(key_sorted[i] % (unsigned)K1);
        r.id = (int)e;
        const float2 w = w0[(long)a * M + m];
        r.wadj = make_float2(w.x, -w.y);
#pragma unroll
        for (int b = 0; b < FZ_J; ++b) r.c1[b] = c1s[m * FZ_J + b];
        rec[i] = r;
    }
    if (i <= cells) {          // key_ptr[c] = first sorted position whose key is >= c
        long lo = 0, hi = n;
        while (lo < hi) {
            const long mid = (lo + hi) >> 1;
            if ((long)key_sorted[mid] < i) lo = mid + 1; else hi = mid;
        }
        key_ptr[i] = (int)lo;
    }
}

// rows by decreasing entry count (ties by row index): one CTA, K0 <= 2048 rows, an O(K0^2) rank is nothing
__global__ void __launch_bounds__(1024) bin_row_order_kernel(const int* __restrict__ key_ptr, int4* __restrict__ row_order, int K0, int K1) {
    __shared__ int cnt[2048];
    for (int r = threadIdx.x; r < K0; r += blockDim.x) cnt[r] = key_ptr[(long)(r + 1) * K1] - key_ptr[(long)r * K1];
    __syncthreads();
    for (int r = threadIdx.x; r < K0; r += blockDim.x) {
        const int c = cnt[r];
        int rank = 0;
        for (int q = 0; q < K0; ++q) rank += (cnt[q] > c || (cnt[q] == c && q < r)) ? 1 : 0;
        row_order[rank] = make_int4(r, key_ptr[(long)r * K1], key_ptr[(long)(r + 1) * K1], 0);
    }
}

// The adjoint row kernel gives every thread one cell and loops over the cell's contributors: the lanes of a warp should
// have similar trip counts, or the warp issues max-over-lanes iterations for every lane.  Per row, order the cells by
// decreasing contributor count (bitonic sort in shared memory, key = count << 12 | (4095 - cell)), once per trajectory.
__global__ void __launch_bounds__(512) bin_cell_order_kernel(const int* __restrict__ key_ptr, unsigned short* __restrict__ cell_order, int K) {
    __shared__ unsigned keys[2048];
    const int R = blockIdx.x;
    const int* kp = key_ptr + (long)R * K;
    int n2 = 1;
    while (n2 < K) n2 <<= 1;
    for (int c = threadIdx.x; c < n2; c += blockDim.x) {
        unsigned key = 0;
        if (c < K) {
            const int first = c - (FZ_J - 1);
            const int cnt = first >= 0 ? kp[c + 1] - kp[first] : (kp[K] - kp[first + K]) + (kp[c + 1] - kp[0]);
            key = ((unsigned)min(cnt, (1 << 19) - 1) << 12) | (unsigned)(4095 - c);
            key += 1u << 31;                 // real cells sort before the padding (key 0)
        }
        keys[c] = key;
    }
    __syncthreads();
    for (int k = 2; k <= n2; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < n2; i += blockDim.x) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const unsigned a = keys[i], b = keys[ixj];
                    const bool desc = (i & k) == 0;          // descending overall
                    if (desc ? a < b : a > b) { keys[i] = b; keys[ixj] = a; }
                }
            }
            __syncthreads();
        }
    for (int i = threadIdx.x; i < K; i += blockDim.x) cell_order[(long)R * K + i] = (unsigned short)(4095 - (keys[i] & 4095u));
}

__global__ void bin_header_kernel(int* hdr, const int4* __restrict__ row_order, long M, int K0, int K1, long n) {
    hdr[7] = row_order[0].z - row_order[0].y;      // entries of the heaviest row (the host's path policy reads it)
    hdr[0] = (int)FZ_MAGIC;
    hdr[1] = (int)(M & 0xffffffffL);
    hdr[2] = (int)(M >> 32);
    hdr[3] = K0;
    hdr[4] = K1;
    hdr[5] = FZ_J;
    hdr[6] = (int)n;
}

static int bins_build(pdu_nufft_plan* p, const float* omega, long M, void* buf, size_t bytes, cudaStream_t st) {
    PDU_REQUIRE(fused_supported(p), "pdu_nufft_bins_build: the plan's grid (%d x %d, J = %d) has no fused path", p->k0, p->k1, p->J);
    const long n = M * FZ_J, cells = (long)p->k0 * p->k1;
    PDU_REQUIRE(n < 2147483647L / 2 && cells < 2147483647L, "pdu_nufft_bins_build: %ld entries exceed 32-bit indexing", n);
    BinsView v = bins_layout(p, M, buf, true);
    if (!buf || bytes < v.total || ((uintptr_t)buf & 255)) {
        set_error("pdu_nufft_bins_build: buffer of %zu bytes (256-byte aligned) required, got %zu", v.total, buf ? bytes : (size_t)0);
        return PDU_ENOMEM;
    }
    bin_entries_kernel<<<(unsigned)cdiv(M, 128), 128, 0, st>>>(omega, p->d_t0, p->d_t1, dims_of(p), M, v.key_in, v.id_in, v.w0, v.c1s);
    PDU_LAUNCHED();
    int bits = 1;
    while ((1L << bits) < cells) ++bits;
    PDU_CUDA(cub::DeviceRadixSort::SortPairs(v.cub_tmp, v.cub_bytes, v.key_in, v.key_out, v.id_in, v.id_out, (int)n, 0, bits, st));
    count_launch(4);
    const long work = n > cells + 1 ? n : cells + 1;
    bin_finish_kernel<<<(unsigned)cdiv(work, 256), 256, 0, st>>>(v.key_out, v.id_out, v.w0, v.c1s, v.key_ptr, v.rec, n, cells, M, p->k1);
    PDU_LAUNCHED();
    bin_row_order_kernel<<<1, 1024, 0, st>>>(v.key_ptr, v.row_order, p->k0, p->k1);
    PDU_LAUNCHED();
    bin_cell_order_kernel<<<(unsigned)p->k0, 512, 0, st>>>(v.key_ptr, v.cell_order, p->k1);
    PDU_LAUNCHED();
    bin_header_kernel<<<1, 1, 0, st>>>(v.hdr, v.row_order, M, p->k0, p->k1, n);
    PDU_LAUNCHED();
    return PDU_OK;
}

// ------------------------------------------------------------------ layouts of the operator's two ends
// flags: PDU_NUFFT_IMAGE_SPLIT -- the image side is [batch, ci, 2, n0, n1] float32 (real plane, imaginary plane)
//        instead of [batch, ci, n0, n1] complex64; PDU_NUFFT_KDATA_SPLIT -- likewise [batch, coils, 2, m] for the samples.
// These are the layouts PD-UNet's CNN blocks use ((re, im) as channels), so the model needs no permute / contiguous /
// view_as_complex passes around the operator.
template <typename T>
__device__ __forceinline__ T* fz_smem() {
    extern __shared__ __align__(16) unsigned char fz_dyn[];
    return reinterpret_cast<T*>(fz_dyn);
}

// ------------------------------------------------------------------ forward, pass 1: image -> column FFT
// CTA = SEQ neighbouring columns of one plane (64-byte runs of every image / T row); thread = (butterfly t, column s)
template <int K, int SEQ>
__global__ void __launch_bounds__(SEQ* FastFft<K>::TPS)
    fz_cols_fwd_kernel(const float* __restrict__ image, const float2* __restrict__ smaps, float2* __restrict__ T,
                       const float* __restrict__ s0, const float* __restrict__ s1, const float2* __restrict__ tw_g, NufftDims d,
                       int coils, int smaps_batch, int split) {
    using F = FastFft<K>;
    constexpr int N = K / 2, TPS = F::TPS, NS3 = F::NS3;            // grid == 2 x image: every address is base + r * constant
    float2* buf = fz_smem<float2>();
    float2* tw = buf + SEQ * F::template pitch<3>();
    const int tid = threadIdx.x, t = tid / SEQ, s = tid - t * SEQ;
    const int p = blockIdx.y;
    const int col = blockIdx.x * SEQ + s;
    for (int i = tid; i < K; i += SEQ * TPS) tw[i] = __ldg(tw_g + i);
    const bool live = col < N;
    const int b = p / coils, c = p - b * coils;
    const int ip = smaps ? b : p;                                   // image plane feeding this grid plane
    const long pix0 = (long)t * N + col;                            // pixel (row t, this column)
    const float2* sm = smaps ? smaps + (long)((smaps_batch == 1 ? 0 : b) * coils + c) * N * N + pix0 : nullptr;
    const float2* src_c = reinterpret_cast<const float2*>(image) + (long)ip * N * N + pix0;
    const float* src_re = image + (long)(2 * ip) * N * N + pix0;
    const float w1 = live ? __ldg(s1 + col) : 0.f;
    const float* s0t = s0 + t;
    auto ld = [&](int r) {                                          // image row t + r TPS < N (HALF_IN)
        if (!live) return make_float2(0.f, 0.f);
        float2 v;
        if (split) v = make_float2(__ldg(src_re + r * (TPS * N)), __ldg(src_re + N * N + r * (TPS * N)));
        else v = __ldg(src_c + r * (TPS * N));
        if (sm) v = cmul(v, __ldg(sm + r * (TPS * N)));
        const float w = w1 * __ldg(s0t + r * TPS);
        return make_float2(v.x * w, v.y * w);
    };
    float2* dst = T + (long)p * K * N + col;
    auto st = [&](int j, int r, float2 v) {
        if (live) dst[j * N + r * (NS3 * N)] = v;
    };
    ff_transform<K, 3, false, true, false>(buf + s * F::template pitch<3>(), tw, t, ld, st);
}

// ------------------------------------------------------------------ forward, pass 2: row FFT + interpolation along the row
// CTA = work item = grid row R (heavy rows first) x PG planes; thread = (plane slot s, butterfly t).

// item -> (row, first plane); -1 when past the end
struct FzItem {
    int R, p0, beg, end;
};
__device__ __forceinline__ FzItem fz_item(int item, int n_items, int groups, int PG, const int4* __restrict__ row_order) {
    FzItem it;
    it.R = -1;
    it.p0 = it.beg = it.end = 0;
    if (item < n_items) {
        const int4 ro = __ldg(row_order + item / groups);
        it.R = ro.x;
        it.p0 = (item % groups) * PG;
        it.beg = ro.y;
        it.end = ro.z;
    }
    return it;
}

template <int K, int PG>
__global__ void __launch_bounds__(PG* FastFft<K>::TPS, (1536 / (PG * FastFft<K>::TPS)) > 0 ? (1536 / (PG * FastFft<K>::TPS)) : 1)
    fz_rows_fwd_kernel(const float2* __restrict__ T, float2* __restrict__ P, const int* __restrict__ key_ptr,
                       const int4* __restrict__ row_order, const BinRec* __restrict__ rec, const float2* __restrict__ tw_g, NufftDims d,
                       int planes, long M, int groups) {
    using F = FastFft<K>;
    constexpr int PITCH = F::template pitch<4>();
    constexpr int NT = PG * F::TPS;
    float2* buf = fz_smem<float2>();
    float2* tw = buf + PG * PITCH;
    const int tid = threadIdx.x, s = tid / F::TPS, t = tid - s * F::TPS;
    const FzItem cur = fz_item(blockIdx.x, K * groups, groups, PG, row_order);
    if (cur.beg == cur.end) return;                                // no sample touches this row: its transform is not needed
    for (int i = tid; i < K; i += NT) tw[i] = __ldg(tw_g + i);
    {
        const int p = cur.p0 + s;
        const bool live = p < planes;
        const float2* src = T + ((long)p * K + cur.R) * (K / 2) + t;
        auto ld = [&](int r) { return live ? __ldcs(src + r * F::TPS) : make_float2(0.f, 0.f); };
        float2* row = buf + s * PITCH;
        // output element j + r NS3 at its padded position pos(j) + r (NS3 + NS3 / 16)
        auto st = [&](int j, int r, float2 v) { row[(j + (j >> 4)) + r * (F::NS3 + F::NS3 / 16)] = v; };
        __syncthreads();                                           // tw is loaded
        ff_transform<K, 4, false, true, false, false, true, true>(row, tw, t, ld, st);
        __syncthreads();
        // a thread = one entry, all PG planes: the record is read once, the taps are LDS.64, and a warp's stores of one
        // plane are 32 neighbouring entries (mostly neighbouring samples of one spoke)
        for (int e = cur.beg + tid; e < cur.end; e += NT) {
            const float4* rp = reinterpret_cast<const float4*>(rec + e);
            const float4 r0 = __ldg(rp), r1 = __ldg(rp + 1), r2 = __ldg(rp + 2), r3 = __ldg(rp + 3);
            const int u = __float_as_int(r0.x), id = __float_as_int(r0.y);
            const float2 c1[FZ_J] = {make_float2(r1.x, r1.y), make_float2(r1.z, r1.w), make_float2(r2.x, r2.y),
                                     make_float2(r2.z, r2.w), make_float2(r3.x, r3.y), make_float2(r3.z, r3.w)};
            int pos[FZ_J];
#pragma unroll
            for (int b = 0; b < FZ_J; ++b) {
                int col = u + b;
                col -= col >= K ? K : 0;
                pos[b] = ff_pos<4>(col);
            }
            const int m = id / FZ_J, a = id - m * FZ_J;
            float2* dst = P + ((long)cur.p0 * FZ_J + a) * M + m;
#pragma unroll
            for (int g = 0; g < PG; ++g) {
                if (cur.p0 + g < planes) {
                    const float2* rw = buf + g * PITCH;
                    float2 acc = make_float2(0.f, 0.f);
#pragma unroll
                    for (int b = 0; b < FZ_J; ++b) {
                        const float2 z = cmul(rw[pos[b]], c1[b]);
                        acc.x += z.x;
                        acc.y += z.y;
                    }
                    __stcs(dst + (long)g * FZ_J * M, acc);
                }
            }
        }
    }
}

// ------------------------------------------------------------------ forward, pass 3: the six rows of every sample
template <int PC>
__global__ void __launch_bounds__(128)
    fz_combine_kernel(const float2* __restrict__ P, float* __restrict__ kdata, const float2* __restrict__ w0, int planes, long M,
                      float scale, int split) {
    const long m = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= M) return;
    float2 w[FZ_J];
#pragma unroll
    for (int a = 0; a < FZ_J; ++a) {
        w[a] = __ldg(w0 + (long)a * M + m);
        w[a].x *= scale;
        w[a].y *= scale;
    }
    const int p_end = min(planes, ((int)blockIdx.y + 1) * PC);
    for (int p = blockIdx.y * PC; p < p_end; ++p) {
        const float2* pp = P + (long)p * FZ_J * M + m;
        float2 v[FZ_J];
#pragma unroll
        for (int a = 0; a < FZ_J; ++a) v[a] = __ldcs(pp + (long)a * M);
        float2 acc = make_float2(0.f, 0.f);
#pragma unroll
        for (int a = 0; a < FZ_J; ++a) {
            const float2 z = cmul(v[a], w[a]);
            acc.x += z.x;
            acc.y += z.y;
        }
        if (split) {
            kdata[(2L * p) * M + m] = acc.x;
            kdata[(2L * p + 1) * M + m] = acc.y;
        } else {
            reinterpret_cast<float2*>(kdata)[(long)p * M + m] = acc;
        }
    }
}

// ------------------------------------------------------------------ adjoint, pass 1: gather along the row + inverse row FFT
// CTA = grid row R x PG planes.  Entries of the row are sorted by first column u, so the samples that reach cell c are
// the contiguous range u in [c - 5, c] (two ranges where it wraps).  Entries are staged EC at a time in shared memory
// (most rows fit one chunk) as z[e][plane] = kdata[plane][m] (x dcf) x wadj and conj(c1[e][.]); a thread owns 8 / PG
// cells for all PG planes; then the pruned inverse row FFT runs on the gathered row in place.
// (r02 also tried: a separate kernel that writes z in entry order + a two-stage TMA bulk-copy ring of small chunks --
//  40 us for the extra pass and 3.5 chunk iterations of bookkeeping per row made it slower, 290 + 40 us against 255;
//  whole warps summing the cells with many contributors -- no gain: the kernel is bound by instruction issue of the
//  per-chunk bookkeeping and the FFT, not by the longest cell.)
template <int K, int PG, int EC>
__global__ void __launch_bounds__(PG* FastFft<K>::TPS, (1024 / (PG * FastFft<K>::TPS)) > 0 ? (1024 / (PG * FastFft<K>::TPS)) : 1)
    fz_rows_adj_kernel(const float* __restrict__ kdata, const float* __restrict__ kweight, float2* __restrict__ T,
                       const int* __restrict__ key_ptr, const int4* __restrict__ row_order,
                       const unsigned short* __restrict__ cell_order, const BinRec* __restrict__ rec,
                       const float2* __restrict__ tw_g, NufftDims d, int planes, long M, int split, int groups) {
    using F = FastFft<K>;
    constexpr int PITCH = F::template pitch<4>();
    constexpr int NT = PG * F::TPS;
    constexpr int CPT = K / NT;                       // cells per thread: 8 / PG
    static_assert(CPT * NT == K && PG % 2 == 0, "threads tile the row; planes are read in pairs");
    float2* buf = fz_smem<float2>();
    float2* tw = buf + PG * PITCH;
    float2* zs = tw + K;                              // [EC][PG]
    float2* cs = zs + EC * PG;                        // [EC][J]
    int* us = reinterpret_cast<int*>(cs + EC * FZ_J); // [EC]
    int* kp = us + EC;                                // [K + 1]
    const int tid = threadIdx.x, s = tid / F::TPS, t = tid - s * F::TPS;
    const FzItem cur = fz_item(blockIdx.x, K * groups, groups, PG, row_order);
    {
        const int R = cur.R, p0 = cur.p0, beg = cur.beg, end = cur.end;
        const int p = p0 + s;
        const bool live = p < planes;
        float2* dst = T + ((long)p * K + R) * d.n1;
        if (beg == end) {                             // empty row: its inverse transform is zero
            if (live)
                for (int e = t; e < d.n1; e += F::TPS) __stcs(dst + e, make_float2(0.f, 0.f));
            return;
        }
        for (int i = tid; i < K; i += NT) tw[i] = __ldg(tw_g + i);
        // stage chunk [cb, cb + ne): a thread = one entry, all PG planes -- the record is read once and the PG sample
        // loads are independent (consecutive lanes = neighbouring samples of a spoke: the loads of one plane coalesce)
        auto stage = [&](int cb, int ne) {
            for (int el = tid; el < ne; el += NT) {
                const float4* rp = reinterpret_cast<const float4*>(rec + cb + el);
                const float4 r0 = __ldg(rp), r1 = __ldg(rp + 1), r2 = __ldg(rp + 2), r3 = __ldg(rp + 3);
                const long m = __float_as_int(r0.y) / FZ_J;
                float2 y[PG];
#pragma unroll
                for (int g = 0; g < PG; ++g) {
                    y[g] = make_float2(0.f, 0.f);
                    if (p0 + g < planes) {
                        if (split) y[g] = make_float2(__ldg(kdata + (2L * (p0 + g)) * M + m), __ldg(kdata + (2L * (p0 + g) + 1) * M + m));
                        else y[g] = __ldg(reinterpret_cast<const float2*>(kdata) + (long)(p0 + g) * M + m);
                    }
                }
                float2 wa = make_float2(r0.z, r0.w);
                if (kweight) {
                    const float wk = __ldg(kweight + m);
                    wa.x *= wk;
                    wa.y *= wk;
                }
                float4* zp = reinterpret_cast<float4*>(zs + el * PG);
#pragma unroll
                for (int g = 0; g < PG; g += 2) {
                    const float2 z0 = cmul(y[g], wa), z1 = cmul(y[g + 1], wa);
                    zp[g / 2] = make_float4(z0.x, z0.y, z1.x, z1.y);
                }
                us[el] = __float_as_int(r0.x);
                float4* c = reinterpret_cast<float4*>(cs + el * FZ_J);       // conj(c1)
                c[0] = make_float4(r1.x, -r1.y, r1.z, -r1.w);
                c[1] = make_float4(r2.x, -r2.y, r2.z, -r2.w);
                c[2] = make_float4(r3.x, -r3.y, r3.z, -r3.w);
            }
        };
        stage(beg, min(EC, end - beg));               // the first chunk's loads are in flight while the tables load
        for (int i = tid; i <= K; i += NT) kp[i] = __ldg(key_ptr + (long)R * K + i);
        // this thread's cells: the q-th block of NT cells in the row's order of decreasing contributor count, so that
        // the lanes of a warp loop about equally often
        int cell[CPT];
#pragma unroll
        for (int q = 0; q < CPT; ++q) cell[q] = __ldg(cell_order + (long)R * K + tid + q * NT);
        __syncthreads();
        // the (up to two) sorted-entry ranges that reach each cell: first column u in [c - 5, c]
        int lo0[CPT], hi0[CPT], lo1[CPT], hi1[CPT];
#pragma unroll
        for (int q = 0; q < CPT; ++q) {
            const int c = cell[q], first = c - (FZ_J - 1);
            if (first >= 0) { lo0[q] = kp[first]; hi0[q] = kp[c + 1]; lo1[q] = 0; hi1[q] = 0; }
            else { lo0[q] = kp[first + K]; hi0[q] = kp[K]; lo1[q] = kp[0]; hi1[q] = kp[c + 1]; }
        }
        float2 acc[CPT][PG];
#pragma unroll
        for (int q = 0; q < CPT; ++q)
#pragma unroll
            for (int g = 0; g < PG; ++g) acc[q][g] = make_float2(0.f, 0.f);

        for (int cb = beg; cb < end; cb += EC) {
            const int ne = min(EC, end - cb);
            if (cb != beg) {
                __syncthreads();                      // the previous chunk has been consumed
                stage(cb, ne);
                __syncthreads();
            }
#pragma unroll
            for (int q = 0; q < CPT; ++q) {
                const int c = cell[q];
#pragma unroll
                for (int rg = 0; rg < 2; ++rg) {
                    const int e0 = max(rg ? lo1[q] : lo0[q], cb), e1 = min(rg ? hi1[q] : hi0[q], cb + ne);
                    for (int e = e0; e < e1; ++e) {
                        const int el = e - cb;
                        int b = c - us[el];
                        b += b < 0 ? K : 0;
                        const float2 w = cs[el * FZ_J + b];
                        const float4* zp = reinterpret_cast<const float4*>(zs + el * PG);
#pragma unroll
                        for (int g = 0; g < PG; g += 2) {
                            const float4 z = zp[g / 2];
                            acc[q][g].x = fmaf(z.x, w.x, fmaf(-z.y, w.y, acc[q][g].x));
                            acc[q][g].y = fmaf(z.x, w.y, fmaf(z.y, w.x, acc[q][g].y));
                            acc[q][g + 1].x = fmaf(z.z, w.x, fmaf(-z.w, w.y, acc[q][g + 1].x));
                            acc[q][g + 1].y = fmaf(z.z, w.y, fmaf(z.w, w.x, acc[q][g + 1].y));
                        }
                    }
                }
            }
        }
#pragma unroll
        for (int q = 0; q < CPT; ++q)
#pragma unroll
            for (int g = 0; g < PG; ++g) buf[g * PITCH + ff_pos<4>(cell[q])] = acc[q][g];
        __syncthreads();
        float2* row = buf + s * PITCH;
        const float2* row_t = row + (t + (t >> 4));      // input element t + r TPS at pos(t) + r (TPS + TPS / 16)
        auto ld = [&](int r) { return row_t[r * (F::TPS + F::TPS / 16)]; };
        auto st = [&](int j, int r, float2 v) {
            if (live) __stcs(dst + j + r * F::NS3, v);
        };
        ff_transform<K, 4, true, false, true, true, false, true>(row, tw, t, ld, st);
    }
}

// ------------------------------------------------------------------ adjoint, pass 2: inverse column FFT + crop (+ apodisation)
// without coil maps the crop, the apodisation and the scale are applied on the way out; with coil maps the cropped
// planes go to U and crop_apod_kernel (nufft.cu) combines the coils
template <int K, int SEQ>
__global__ void __launch_bounds__(SEQ* FastFft<K>::TPS, K <= 640 ? 3 : 1)
    fz_cols_adj_kernel(const float2* __restrict__ T, float* __restrict__ out, const float* __restrict__ s0, const float* __restrict__ s1,
                       const float2* __restrict__ tw_g, NufftDims d, float scale, int finish, int split) {
    using F = FastFft<K>;
    constexpr int N = K / 2, TPS = F::TPS, NS3 = F::NS3;
    float2* buf = fz_smem<float2>();
    float2* tw = buf + SEQ * F::template pitch<3>();
    const int tid = threadIdx.x, t = tid / SEQ, s = tid - t * SEQ;
    const int p = blockIdx.y;
    const int col = blockIdx.x * SEQ + s;
    for (int i = tid; i < K; i += SEQ * TPS) tw[i] = __ldg(tw_g + i);
    const bool live = col < N;
    const float2* src = T + ((long)p * K + t) * N + col;
    const float w1 = (finish && live) ? __ldg(s1 + col) * scale : 1.f;
    float2* out_c = reinterpret_cast<float2*>(out) + (long)p * N * N + col;
    float* out_re = out + (long)(2 * p) * N * N + col;
    auto ld = [&](int r) { return live ? __ldcs(src + r * (TPS * N)) : make_float2(0.f, 0.f); };
    auto st = [&](int j, int r, float2 v) {                          // image row j + r NS3 < N (HALF_OUT)
        if (!live) return;
        if (finish) {
            const float w = w1 * __ldg(s0 + j + r * NS3);
            v.x *= w;
            v.y *= w;
        }
        if (split) {
            out_re[j * N + r * (NS3 * N)] = v.x;
            out_re[N * N + j * N + r * (NS3 * N)] = v.y;
        } else {
            __stcs(out_c + j * N + r * (NS3 * N), v);
        }
    };
    ff_transform<K, 3, true, false, true>(buf + s * F::template pitch<3>(), tw, t, ld, st);
}

// ------------------------------------------------------------------ host side
template <int K>
static constexpr int fz_seq() { return K <= 1024 ? 8 : 4; }       // SEQ * K / 8 threads <= 1024


template <int K>
static size_t fz_cols_smem() { return ((size_t)fz_seq<K>() * FastFft<K>::template pitch<3>() + K) * sizeof(float2); }
template <int K, int PG>
static size_t fz_rows_fwd_smem() { return ((size_t)PG * FastFft<K>::template pitch<4>() + K) * sizeof(float2); }
template <int K, int PG>
static size_t fz_rows_adj_smem() {
    return fz_rows_fwd_smem<K, PG>() + (size_t)FZ_EC * (PG * 8 + FZ_J * 8 + 4) + (size_t)(K + 1) * 4 + 16;
}

// workspace: T [planes][K][N] | P [planes][J][M] (forward)  /  U [planes][N][N] (adjoint with coil maps)
size_t fused_workspace_bytes(const pdu_nufft_plan* p, int planes, long m) {
    const size_t T = (size_t)planes * p->k0 * p->n1 * sizeof(float2);
    const size_t P = (size_t)((planes + 7) & ~7) * FZ_J * (size_t)m * sizeof(float2);     // also Z (planes rounded up to the group)
    const size_t U = (size_t)planes * p->n0 * p->n1 * sizeof(float2);
    return align256(T) + align256(std::max(P, U));
}

static int check_bins(const pdu_nufft_plan* p, const void* bins, long m, const char* who) {
    PDU_REQUIRE(bins != nullptr && ((uintptr_t)bins & 255) == 0, "%s: bins is null or not 256-byte aligned", who);
    (void)p;
    (void)m;
    return PDU_OK;
}

template <int K, int PG>
static int fused_forward_k(pdu_nufft_plan* p, const float* image, float* kdata, const float2* smaps, int batch, int coils,
                           int smaps_batch, long m, float scale, const BinsView& v, int flags, void* ws, cudaStream_t st) {
    constexpr int FZ_SEQ_COLS = fz_seq<K>();
    const NufftDims d = dims_of(p);
    const int planes = batch * coils;
    float2* T = (float2*)ws;
    float2* P = (float2*)((char*)ws + align256((size_t)planes * K * d.n1 * sizeof(float2)));
    PDU_CUDA((ensure_dyn_smem<fz_cols_fwd_kernel<K, FZ_SEQ_COLS>>((int)fz_cols_smem<K>())));
    PDU_CUDA((ensure_dyn_smem<fz_rows_fwd_kernel<K, PG>>((int)fz_rows_fwd_smem<K, PG>())));
    fz_cols_fwd_kernel<K, FZ_SEQ_COLS><<<dim3((unsigned)cdiv(d.n1, FZ_SEQ_COLS), (unsigned)planes), FZ_SEQ_COLS * FastFft<K>::TPS,
                                         fz_cols_smem<K>(), st>>>(image, smaps, T, p->d_s0, p->d_s1, p->d_w0, d, coils, smaps_batch,
                                                                  (flags & PDU_NUFFT_IMAGE_SPLIT) ? 1 : 0);
    PDU_LAUNCHED();
    {
        const int groups = (int)cdiv(planes, PG);
        const long ctas = (long)K * groups;
        fz_rows_fwd_kernel<K, PG><<<(unsigned)ctas, PG * FastFft<K>::TPS, fz_rows_fwd_smem<K, PG>(), st>>>(
            T, P, v.key_ptr, v.row_order, v.rec, p->d_w1, d, planes, m, groups);
        PDU_LAUNCHED();
    }
    constexpr int PC = 8;
    fz_combine_kernel<PC><<<dim3((unsigned)cdiv(m, 128), (unsigned)cdiv(planes, PC)), 128, 0, st>>>(
        P, kdata, v.w0, planes, m, scale, (flags & PDU_NUFFT_KDATA_SPLIT) ? 1 : 0);
    PDU_LAUNCHED();
    note_kernel(OP_NUFFT_FWD, "fz_cols_fwd_kernel<%d,%d> + fz_rows_fwd_kernel<%d,%d> (row FFT + in-row interpolation) + fz_combine_kernel "
                "(%d planes of %dx%d, M=%ld; own register-resident pruned FFT, grid never materialised)", K, FZ_SEQ_COLS, K, PG, planes,
                K, K, m);
    return PDU_OK;
}

int launch_crop_apod(pdu_nufft_plan* p, const float2* U, const float2* smaps, float2* image, int out_planes, int coils,
                     int smaps_batch, float scale, int split, cudaStream_t st);      // nufft.cu

template <int K, int PG>
static int fused_adjoint_k(pdu_nufft_plan* p, const float* kdata, float* image, const float2* smaps, const float* kweight,
                           int batch, int coils, int smaps_batch, long m, float scale, const BinsView& v, int flags, void* ws,
                           cudaStream_t st, const SmapsGrad* sg) {
    constexpr int FZ_SEQ_COLS = fz_seq<K>();
    const NufftDims d = dims_of(p);
    const int planes = batch * coils;
    float2* T = (float2*)ws;
    float2* U = (float2*)((char*)ws + align256((size_t)planes * K * d.n1 * sizeof(float2)));
    PDU_CUDA((ensure_dyn_smem<fz_rows_adj_kernel<K, PG, FZ_EC>>((int)fz_rows_adj_smem<K, PG>())));
    PDU_CUDA((ensure_dyn_smem<fz_cols_adj_kernel<K, FZ_SEQ_COLS>>((int)fz_cols_smem<K>())));
    {
        const int groups = (int)cdiv(planes, PG);
        const long ctas = (long)K * groups;
        fz_rows_adj_kernel<K, PG, FZ_EC><<<(unsigned)ctas, PG * FastFft<K>::TPS, fz_rows_adj_smem<K, PG>(), st>>>(
            kdata, kweight, T, v.key_ptr, v.row_order, v.cell_order, v.rec, p->d_w1, d, planes, m,
            (flags & PDU_NUFFT_KDATA_SPLIT) ? 1 : 0, groups);
        PDU_LAUNCHED();
    }
    const int split = (flags & PDU_NUFFT_IMAGE_SPLIT) ? 1 : 0;
    const dim3 gc((unsigned)cdiv(d.n1, FZ_SEQ_COLS), (unsigned)planes);
    if (!smaps && !sg) {
        fz_cols_adj_kernel<K, FZ_SEQ_COLS><<<gc, FZ_SEQ_COLS * FastFft<K>::TPS, fz_cols_smem<K>(), st>>>(
            T, image, p->d_s0, p->d_s1, p->d_w0, d, scale, 1, split);
        PDU_LAUNCHED();
    } else {
        fz_cols_adj_kernel<K, FZ_SEQ_COLS><<<gc, FZ_SEQ_COLS * FastFft<K>::TPS, fz_cols_smem<K>(), st>>>(
            T, (float*)U, p->d_s0, p->d_s1, p->d_w0, d, 1.f, 0, 0);
        PDU_LAUNCHED();
        NufftDims dc = d;          // the cropped result is a dense [n0][n1] "grid"
        dc.k0 = d.n0;
        dc.k1 = d.n1;
        int rc = sg ? launch_smaps_grad(p, U, dc, coils, scale, *sg, st)
                    : launch_crop_apod(p, U, smaps, (float2*)image, batch, coils, smaps_batch, scale, split, st);
        if (rc) return rc;
    }
    note_kernel(sg ? OP_SMAPS_GRAD : OP_NUFFT_ADJ, "fz_rows_adj_kernel<%d,%d,%d> (in-row gather + inverse row FFT) + "
                "fz_cols_adj_kernel<%d,%d>%s (%d planes of %dx%d, M=%ld; own register-resident pruned FFT, grid never "
                "materialised, no atomics)", K, PG, FZ_EC, K, FZ_SEQ_COLS,
                sg ? " + smaps_grad_kernel (fused path)" : (smaps ? " + crop_apod_kernel (coil combine)" : " (crop + apodisation fused)"),
                planes, K, K, m);
    return PDU_OK;
}

int fused_forward(pdu_nufft_plan* p, const float* image, float* kdata, const float* smaps, int batch, int coils, int smaps_batch,
                  long m, float scale, const void* bins, int flags, void* ws, cudaStream_t st) {
    int rc = check_bins(p, bins, m, "pdu_nufft_fwd_binned_c64");
    if (rc) return rc;
    const BinsView v = bins_layout(p, m, const_cast<void*>(bins), false);
    const float2* sm = (const float2*)smaps;
    const int pg = option(OPT_NUFFT_FWD) == 8 ? 8 : (option(OPT_NUFFT_FWD) == 2 ? 2 : 4);     // A/B: planes per CTA (default 4)
    switch (p->k0) {
        case 256: return pg == 8 ? fused_forward_k<256, 8>(p, image, kdata, sm, batch, coils, smaps_batch, m, scale, v, flags, ws, st) : (pg == 2 ? fused_forward_k<256, 2>(p, image, kdata, sm, batch, coils, smaps_batch, m, scale, v, flags, ws, st) : fused_forward_k<256, 4>(p, image, kdata, sm, batch, coils, smaps_batch, m, scale, v, flags, ws, st));
        case 512: return pg == 8 ? fused_forward_k<512, 8>(p, image, kdata, sm, batch, coils, smaps_batch, m, scale, v, flags, ws, st) : (pg == 2 ? fused_forward_k<512, 2>(p, image, kdata, sm, batch, coils, smaps_batch, m, scale, v, flags, ws, st) : fused_forward_k<512, 4>(p, image, kdata, sm, batch, coils, smaps_batch, m, scale, v, flags, ws, st));
        case 640: return pg == 8 ? fused_forward_k<640, 8>(p, image, kdata, sm, batch, coils, smaps_batch, m, scale, v, flags, ws, st) : (pg == 2 ? fused_forward_k<640, 2>(p, image, kdata, sm, batch, coils, smaps_batch, m, scale, v, flags, ws, st) : fused_forward_k<640, 4>(p, image, kdata, sm, batch, coils, smaps_batch, m, scale, v, flags, ws, st));
        case 1024: return pg == 8 ? fused_forward_k<1024, 8>(p, image, kdata, sm, batch, coils, smaps_batch, m, scale, v, flags, ws, st) : (pg == 2 ? fused_forward_k<1024, 2>(p, image, kdata, sm, batch, coils, smaps_batch, m, scale, v, flags, ws, st) : fused_forward_k<1024, 4>(p, image, kdata, sm, batch, coils, smaps_batch, m, scale, v, flags, ws, st));
        case 2048: return pg == 2 ? fused_forward_k<2048, 2>(p, image, kdata, sm, batch, coils, smaps_batch, m, scale, v, flags, ws, st) : fused_forward_k<2048, 4>(p, image, kdata, sm, batch, coils, smaps_batch, m, scale, v, flags, ws, st);
    }
    set_error("pdu_nufft_fwd_binned_c64: grid %d has no fused path", p->k0);
    return PDU_EUNSUPPORTED;
}

int fused_adjoint(pdu_nufft_plan* p, const float* kdata, float* image, const float* smaps, const float* kweight, int batch,
                  int coils, int smaps_batch, long m, float scale, const void* bins, int flags, void* ws, cudaStream_t st,
                  const SmapsGrad* sg) {
    int rc = check_bins(p, bins, m, "pdu_nufft_adj_binned_c64");
    if (rc) return rc;
    const BinsView v = bins_layout(p, m, const_cast<void*>(bins), false);
    const float2* sm = (const float2*)smaps;
    const int pg = option(OPT_NUFFT_ADJ) == 8 ? 8 : (option(OPT_NUFFT_ADJ) == 2 ? 2 : 4);     // A/B: planes per CTA (default 4)
    switch (p->k0) {
        case 256: return pg == 8 ? fused_adjoint_k<256, 8>(p, kdata, image, sm, kweight, batch, coils, smaps_batch, m, scale, v, flags, ws, st, sg) : (pg == 2 ? fused_adjoint_k<256, 2>(p, kdata, image, sm, kweight, batch, coils, smaps_batch, m, scale, v, flags, ws, st, sg) : fused_adjoint_k<256, 4>(p, kdata, image, sm, kweight, batch, coils, smaps_batch, m, scale, v, flags, ws, st, sg));
        case 512: return pg == 8 ? fused_adjoint_k<512, 8>(p, kdata, image, sm, kweight, batch, coils, smaps_batch, m, scale, v, flags, ws, st, sg) : (pg == 2 ? fused_adjoint_k<512, 2>(p, kdata, image, sm, kweight, batch, coils, smaps_batch, m, scale, v, flags, ws, st, sg) : fused_adjoint_k<512, 4>(p, kdata, image, sm, kweight, batch, coils, smaps_batch, m, scale, v, flags, ws, st, sg));
        case 640: return pg == 8 ? fused_adjoint_k<640, 8>(p, kdata, image, sm, kweight, batch, coils, smaps_batch, m, scale, v, flags, ws, st, sg) : (pg == 2 ? fused_adjoint_k<640, 2>(p, kdata, image, sm, kweight, batch, coils, smaps_batch, m, scale, v, flags, ws, st, sg) : fused_adjoint_k<640, 4>(p, kdata, image, sm, kweight, batch, coils, smaps_batch, m, scale, v, flags, ws, st, sg));
        case 1024: return pg == 8 ? fused_adjoint_k<1024, 8>(p, kdata, image, sm, kweight, batch, coils, smaps_batch, m, scale, v, flags, ws, st, sg) : (pg == 2 ? fused_adjoint_k<1024, 2>(p, kdata, image, sm, kweight, batch, coils, smaps_batch, m, scale, v, flags, ws, st, sg) : fused_adjoint_k<1024, 4>(p, kdata, image, sm, kweight, batch, coils, smaps_batch, m, scale, v, flags, ws, st, sg));
        case 2048: return pg == 2 ? fused_adjoint_k<2048, 2>(p, kdata, image, sm, kweight, batch, coils, smaps_batch, m, scale, v, flags, ws, st, sg) : fused_adjoint_k<2048, 4>(p, kdata, image, sm, kweight, batch, coils, smaps_batch, m, scale, v, flags, ws, st, sg);
    }
    set_error("pdu_nufft_adj_binned_c64: grid %d has no fused path", p->k0);
    return PDU_EUNSUPPORTED;
}

}  // namespace pdu

using namespace pdu;

extern "C" {

int pdu_nufft_has_fused_path(const pdu_nufft_plan_t* p) { return p && fused_supported(p) ? 1 : 0; }

size_t pdu_nufft_bins_bytes(const pdu_nufft_plan_t* p, long m, size_t* persist_bytes) {
    if (persist_bytes) *persist_bytes = 0;
    if (!p || m <= 0 || !fused_supported(p)) return 0;
    const BinsView v = bins_layout(p, m, nullptr, true);
    if (persist_bytes) *persist_bytes = v.persist;
    return v.total;
}

int pdu_nufft_bins_build(pdu_nufft_plan_t* p, const float* omega, long m, void* bins, size_t bins_bytes, pdu_stream_t stream) {
    PDU_REQUIRE(p && omega && m > 0, "pdu_nufft_bins_build: null pointer or m <= 0");
    PDU_CHECK_DEVICE("pdu_nufft_bins_build");
    return bins_build(p, omega, m, bins, bins_bytes, (cudaStream_t)stream);
}

size_t pdu_nufft_binned_workspace_bytes(const pdu_nufft_plan_t* p, int planes, long m) {
    if (!p || planes <= 0 || m <= 0 || !fused_supported(p)) return 0;
    return fused_workspace_bytes(p, planes, m);
}

}  // extern "C"
