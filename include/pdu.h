/* pdu.h -- C ABI of libpdu_b200.so: the measurement operators of PD-UNet
 * (CT: Radon forward / backprojection / sinogram filter; radial MRI: Kaiser-
 * Bessel NUFFT forward / adjoint; the fused primal-dual elementwise steps) as
 * hand-written CUDA for sm_100a.
 *
 * What each entry point replaces.  The reference mount is a stub
 * (/root/reference/README.md:1-5: title, paper link, "check out the branches");
 * the operator code the README points to lives in the third-party libraries
 * torch_radon and torchkbnufft, neither of which is mounted.  The citations
 * below are therefore to the library interface each symbol stands in for, as
 * recalled ([RECALL], SURVEY.md section 8b), not to files under /root/reference.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless the parameter says "host";
 *  - tensors are dense, row-major, innermost axis last; complex values are
 *    interleaved (re, im) float pairs;
 *  - all work is enqueued on `stream` (a cudaStream_t); nothing synchronises;
 *  - the caller owns every buffer and workspace; the library allocates only
 *    inside pdu_nufft_plan_create;
 *  - every function returns PDU_OK or a negative PDU_E* code and never throws;
 *    pdu_last_error() gives the thread-local message of the last failure;
 *  - entry points are re-entrant; one nufft plan may be used by one thread at
 *    a time (it carries a cuFFT handle whose stream is set per call).
 */
#ifndef PDU_H
#define PDU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define PDU_API __attribute__((visibility("default")))
#else
#define PDU_API
#endif

typedef struct CUstream_st* pdu_stream_t;           /* == cudaStream_t */

enum {
    PDU_OK = 0,
    PDU_EINVAL = -1,         /* bad argument (null pointer, size <= 0, unsupported shape) */
    PDU_ECUDA = -2,          /* a CUDA runtime call or launch failed */
    PDU_ENOMEM = -3,         /* workspace too small / allocation failed */
    PDU_EUNSUPPORTED = -4,   /* valid request this build cannot serve */
    PDU_EFFT = -5            /* cuFFT failure */
};

PDU_API const char* pdu_last_error(void);
PDU_API int pdu_version(void);                       /* 10000*major + 100*minor + patch */
PDU_API int pdu_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* Kernel-variant switches for A/B measurement ("radon_fwd_variant", "radon_adj_variant",
 * "filter_variant", "nufft_fwd_variant", "nufft_adj_variant"); value -1 restores the default (the
 * numbering is documented at each entry point's dispatch in csrc/).  Returns PDU_EINVAL for an
 * unknown key.  Never changes results beyond floating-point rounding / summation order. */
PDU_API int pdu_set_option(const char* key, int value);
PDU_API int pdu_get_option(const char* key, int* value);
/* Number of kernels this library launched (all threads of the process) since the last reset. */
PDU_API long pdu_launch_count(int reset);
/* Device-side failure word.  A kernel whose TMA / mbarrier pipeline wait times out (a fault, a
 * regression) stores a non-zero code in a word of mapped host memory and abandons its tile instead
 * of producing numbers from an unfilled buffer.  While the word is set every compute entry point
 * returns PDU_ECUDA (checked on entry: a plain host read, no synchronisation; the failing launch
 * itself has already returned PDU_OK, so callers that must know synchronise and call this).
 * Returns the code (0 = none, 1 = forward projector, 2 = tensor-core filter, 3 = NUFFT);
 * reset != 0 clears it.  Option "debug_fault" = 1 makes the TMA producers of those kernels skip
 * their loads so that the path can be tested. */
PDU_API int pdu_device_error(int reset);
/* Name and shape of the kernel the dispatcher of an operator chose in this thread's most recent
 * call: op in {"radon_fwd", "radon_adj", "filter", "nufft_fwd", "nufft_adj", "toep", "cg", "smaps_grad"}; "" before
 * the first call.  The string stays valid until the thread's next call of that operator. */
PDU_API const char* pdu_last_kernel(const char* op);

/* ------------------------------------------------------------------ CT ---- */
enum { PDU_GEOM_PARALLEL = 0, PDU_GEOM_FAN = 1 };

/* [RECALL] torch_radon RaysCfg(width, height, det_count, det_spacing, n_angles,
 * clip_to_circle, s_dist, d_dist). */
typedef struct pdu_radon_geom {
    int32_t geom;            /* PDU_GEOM_* */
    int32_t n;               /* image is n x n */
    int32_t n_angles;
    int32_t det_count;
    float det_spacing;
    float s_dist;            /* source -> rotation centre (fan) */
    float d_dist;            /* rotation centre -> detector (fan) */
    int32_t clip_to_circle;
} pdu_radon_geom_t;

/* trig[2a] = cos(angles[a]), trig[2a+1] = sin(angles[a]), evaluated in float64 and rounded
 * once.  `angles` are the INTERNAL angles (the Python wrapper negates the user's, as
 * [RECALL] torch_radon BaseRadon.__init__ does). */
PDU_API int pdu_radon_trig_f32(const float* angles, float* trig, int n_angles, pdu_stream_t stream);

/* Bytes of scratch the forward projector wants: the bilinear-cell tensors of the batch and of its
 * transpose, 2 * batch * (n+1)^2 * 16 bytes (the float-tile variants use the head of it for a
 * transposed copy), followed by the strip-box table of the call's geometry (8 bytes per strip and
 * (detector block, view group)).  0 is a valid answer. */
PDU_API size_t pdu_radon_workspace_bytes(const pdu_radon_geom_t* g, int batch);

/* img [batch, n, n] -> sino [batch, n_angles, det_count].
 * Replaces [RECALL] torch_radon `Radon.forward` / `RadonFanbeam.forward`
 * (torch_radon_cuda.forward -> radon_forward_cuda). */
PDU_API int pdu_radon_fwd_f32(const float* img, float* sino, const float* trig, int batch,
                              const pdu_radon_geom_t* g, void* workspace, size_t workspace_bytes,
                              pdu_stream_t stream);

/* sino [batch, n_angles, det_count] -> img [batch, n, n].
 * Replaces [RECALL] torch_radon `Radon.backprojection` (alias `.backward`)
 * (torch_radon_cuda.backward -> radon_backward_cuda). */
PDU_API int pdu_radon_adj_f32(const float* sino, float* img, const float* trig, int batch,
                              const pdu_radon_geom_t* g, void* workspace, size_t workspace_bytes,
                              pdu_stream_t stream);

/* The same with fan-beam FBP's distance weighting: fbp_weight != 0 multiplies every tap of a fan-beam view once more
 * by s_dist / (s_dist - t), t the pixel's depth along the central ray -- together with the magnification weight the
 * plain adjoint already applies this is the 1 / U^2 of Kak & Slaney section 3.4.2 for a flat equispaced detector
 * (views over 2 pi).  Ignored for parallel beams. */
PDU_API int pdu_radon_adj_weighted_f32(const float* sino, float* img, const float* trig, int batch,
                                       const pdu_radon_geom_t* g, int fbp_weight, void* workspace,
                                       size_t workspace_bytes, pdu_stream_t stream);

/* out[r, i] = sum_j sino[r, j] * taps[(i - j) + det_count - 1],  r < rows.
 * taps: 2*det_count - 1 spatial filter taps (already scaled by pi / (2 n_angles)).
 * Replaces [RECALL] torch_radon `Radon.filter_sinogram` (pad, rfft, multiply, irfft, crop, scale).
 * The tensor-core variant wants the workspace filled by pdu_filter_prepare_f32. */
PDU_API size_t pdu_filter_workspace_bytes(int det_count);
PDU_API int pdu_filter_prepare_f32(const float* taps, void* workspace, size_t workspace_bytes,
                                   int det_count, pdu_stream_t stream);
PDU_API int pdu_filter_sinogram_f32(const float* sino, float* out, const float* taps,
                                    const void* workspace, size_t workspace_bytes, long rows,
                                    int det_count, pdu_stream_t stream);
/* The same with sino[r, j] first multiplied by col_weight[j] (float[det_count], nullable) inside the
 * kernel: the cosine pre-weight of fan-beam FBP (Kak & Slaney eq. 3.3.2-(95) for a flat equispaced
 * detector) without a separate pass over the sinogram. */
PDU_API int pdu_filter_sinogram_weighted_f32(const float* sino, float* out, const float* taps,
                                             const float* col_weight, const void* workspace,
                                             size_t workspace_bytes, long rows, int det_count,
                                             pdu_stream_t stream);

/* ----------------------------------------------------------------- MRI ---- */
typedef struct pdu_nufft_plan pdu_nufft_plan_t;

/* Replaces the buffers [RECALL] torchkbnufft `KbNufft.__init__` registers (tables, scaling_coef,
 * im_size, grid_size, n_shift, numpoints, table_oversamp).  table0/table1: HOST complex64
 * [numpoints*table_oversamp + 1]; scal0/scal1: HOST float32 [n0] / [n1]. */
PDU_API int pdu_nufft_plan_create(pdu_nufft_plan_t** plan, int n0, int n1, int k0, int k1,
                                  int numpoints, int table_oversamp, int shift0, int shift1,
                                  const float* table0, const float* table1,
                                  const float* scal0, const float* scal1);
PDU_API int pdu_nufft_plan_destroy(pdu_nufft_plan_t* plan);
/* Scratch for `planes` = batch*coils oversampled grids. */
PDU_API size_t pdu_nufft_workspace_bytes(const pdu_nufft_plan_t* plan, int planes);

/* image [batch, ci, n0, n1] c64 (ci == coils, or ci == 1 with smaps) -> kdata [batch, coils, m].
 * omega [2, m] radians.  smaps [smaps_batch (1 or batch), coils, n0, n1] c64 or NULL.
 * scale multiplies the result (1 or 1/sqrt(k0 k1) for norm="ortho").
 * Replaces [RECALL] torchkbnufft `KbNufft.forward` (functional.kb_table_nufft). */
PDU_API int pdu_nufft_fwd_c64(pdu_nufft_plan_t* plan, const float* image, float* kdata,
                              const float* omega, const float* smaps, int batch, int coils,
                              int smaps_batch, long m, float scale, void* workspace,
                              size_t workspace_bytes, pdu_stream_t stream);
/* kdata [batch, coils, m] -> image [batch, co, n0, n1] (co == coils, or 1 with smaps).
 * Replaces [RECALL] torchkbnufft `KbNufftAdjoint.forward` (functional.kb_table_nufft_adjoint). */
PDU_API int pdu_nufft_adj_c64(pdu_nufft_plan_t* plan, const float* kdata, float* image,
                              const float* omega, const float* smaps, int batch, int coils,
                              int smaps_batch, long m, float scale, void* workspace,
                              size_t workspace_bytes, pdu_stream_t stream);
/* The adjoint interpolator of one trajectory as a sparse matrix sorted by grid cell (CSR), built once
 * and applied as a gather: no atomics, no memset, bit-reproducible sums.  Worth it whenever a trajectory
 * is used more than once (every unrolled iteration / DCF iteration / training step).  `csr` is a
 * caller-owned device buffer of pdu_nufft_csr_bytes(plan, m) bytes, 256-byte aligned; it also holds the
 * build scratch.  pdu_nufft_adj_csr_c64 is pdu_nufft_adj_c64 with the scatter replaced by the gather
 * (csr == NULL falls back to the atomic scatter).
 * Replaces [RECALL] torchkbnufft's precomputed `interp_mats` path (calc_tensor_spmatrix + sparse matmul). */
PDU_API size_t pdu_nufft_csr_bytes(const pdu_nufft_plan_t* plan, long m);
/* The same size, and in *persist_bytes how much of the buffer (its head) the apply calls read: the rest is
 * build scratch that may be released once pdu_nufft_csr_build has been enqueued. */
PDU_API size_t pdu_nufft_csr_bytes2(const pdu_nufft_plan_t* plan, long m, size_t* persist_bytes);
PDU_API int pdu_nufft_csr_build(pdu_nufft_plan_t* plan, const float* omega, long m, void* csr,
                                size_t csr_bytes, pdu_stream_t stream);
PDU_API int pdu_nufft_interp_adj_csr_c64(pdu_nufft_plan_t* plan, const float* kdata, float* grid,
                                         const void* csr, int planes, long m, pdu_stream_t stream);
PDU_API int pdu_nufft_adj_csr_c64(pdu_nufft_plan_t* plan, const float* kdata, float* image,
                                  const float* omega, const float* smaps, int batch, int coils,
                                  int smaps_batch, long m, float scale, const void* csr, void* workspace,
                                  size_t workspace_bytes, pdu_stream_t stream);
/* Fused path for the BASELINE grids (k = 2 n in {256, 512, 640, 1024, 2048}, numpoints 6, square): the separable
 * Kaiser-Bessel interpolation is split along the two grid axes and fused into the two passes of the library's own
 * pruned FFT, so the oversampled grid is never written to memory and neither direction needs atomics
 * (csrc/nufft_fused.cu).  It needs the trajectory's "row bins" -- every (sample, row tap) entry sorted by grid row and
 * first column -- built once per trajectory:
 *   pdu_nufft_bins_bytes   size of the device buffer the build needs (256-byte aligned); the first *persist_bytes of
 *                          it must be kept for the calls below, the rest is build scratch and may be released
 *   pdu_nufft_bins_build   omega [2, m] -> bins
 * flags: PDU_NUFFT_IMAGE_SPLIT -- the image side is [batch, ci, 2, n0, n1] float32 (real plane, imaginary plane) instead
 * of complex64 [batch, ci, n0, n1]; PDU_NUFFT_KDATA_SPLIT -- likewise [batch, coils, 2, m] for the samples: the layouts
 * PD-UNet's CNN blocks use, so no permute / view_as_complex passes surround the operator.  kweight (nullable):
 * float32 [m] multiplied into the samples on load (the density compensation of the adjoint).
 * Replace [RECALL] torchkbnufft KbNufft / KbNufftAdjoint with precomputed interpolation (`interp_mats`). */
enum { PDU_NUFFT_IMAGE_SPLIT = 1, PDU_NUFFT_KDATA_SPLIT = 2 };
PDU_API int pdu_nufft_has_fused_path(const pdu_nufft_plan_t* plan);
PDU_API size_t pdu_nufft_bins_bytes(const pdu_nufft_plan_t* plan, long m, size_t* persist_bytes);
PDU_API int pdu_nufft_bins_build(pdu_nufft_plan_t* plan, const float* omega, long m, void* bins,
                                 size_t bins_bytes, pdu_stream_t stream);
PDU_API size_t pdu_nufft_binned_workspace_bytes(const pdu_nufft_plan_t* plan, int planes, long m);
PDU_API int pdu_nufft_fwd_binned_c64(pdu_nufft_plan_t* plan, const float* image, float* kdata,
                                     const float* smaps, int batch, int coils, int smaps_batch, long m,
                                     float scale, const void* bins, int flags, void* workspace,
                                     size_t workspace_bytes, pdu_stream_t stream);
PDU_API int pdu_nufft_adj_binned_c64(pdu_nufft_plan_t* plan, const float* kdata, float* image,
                                     const float* smaps, const float* kweight, int batch, int coils,
                                     int smaps_batch, long m, float scale, const void* bins, int flags,
                                     void* workspace, size_t workspace_bytes, pdu_stream_t stream);
/* Gradient of the coil maps through the adjoint: gs [smaps_batch, coils, n0, n1] complex64 (+)= the adjoint of kdata
 * [batch, coils, m] WITHOUT the coil combination, U[b, c] = A^H(kweight . kdata[b, c]) (times scale, as
 * pdu_nufft_adj_c64), reduced as   gs[s, c] = sum_{b : s(b) = s} U[b, c] . conj(q[b]),  s(b) = 0 for smaps_batch 1, else b.
 * q: [batch, 1, n0, n1] complex64, or [batch, 2, n0, n1] float32 with PDU_NUFFT_IMAGE_SPLIT in flags.  The path is the
 * one the adjoint entry points would take: bins non-NULL -- the fused row-binned path (pdu_nufft_adj_binned_c64's
 * workspace, kweight and PDU_NUFFT_KDATA_SPLIT allowed); otherwise omega with the CSR gather when csr is non-NULL,
 * the atomic scatter when it is NULL (pdu_nufft_workspace_bytes of one batch chunk, complex64 kdata, no kweight).  The
 * last pass is smaps_grad_kernel in place of crop_apod_kernel: b runs in increasing order in registers, no atomics,
 * and accumulate != 0 adds to gs (a batch cut into calls carries a shared map's sum from call to call).
 * pdu_last_kernel("smaps_grad").  The gradient torch autograd wants for the maps of KbNufft (kdata = the incoming
 * gradient, q = the image) and of KbNufftAdjoint (kdata = its input, q = the incoming gradient). */
PDU_API int pdu_nufft_adj_smaps_grad_c64(pdu_nufft_plan_t* plan, const float* kdata, const float* q, float* gs,
                                         const float* omega, const void* csr, const void* bins, const float* kweight,
                                         int batch, int coils, int smaps_batch, long m, float scale, int flags,
                                         int accumulate, void* workspace, size_t workspace_bytes, pdu_stream_t stream);

/* Toeplitz-embedded normal operator A^H W A of the NUFFT: no interpolation, one zero-padded 2n0 x 2n1
 * FFT, a pointwise multiply by a kernel and one cropped inverse FFT, whatever the trajectory length.
 *   pdu_toep_plan_create      a plan with grid 2 n per axis, unit apodisation, marked as a Toeplitz plan
 *                             (destroy it with pdu_nufft_plan_destroy).  PDU_EUNSUPPORTED for sizes whose
 *                             2 n has a prime factor above 5 (or whose rows do not fit the shared-memory FFT).
 *                             A Toeplitz plan passed to a pdu_nufft_* entry point, or a Kaiser-Bessel plan to
 *                             a pdu_toep_* one, is PDU_EINVAL.
 *   pdu_toep_workspace_bytes  scratch of pdu_toep_apply_c64 for `planes` = batch*coils planes; a call is cut
 *                             into batch chunks of at most 512 MB of scratch, and wants the size of one chunk.
 *   pdu_toep_kernel_c64       kernel [kernels, 2 n0, 2 n1] = fft2(p_circ) (unnormalised), p_circ the circulant
 *                             layout of the point-spread function assembled from q1 = A^H w (omega) and
 *                             q2 = A^H w (omega0 negated), both [kernels, n0, n1] c64 with n_shift 0, times
 *                             `scale` (1, or 1/(k0 k1) of the NUFFT grid for norm="ortho").  ws: kernels * 4 n0 n1
 *                             complex64 values.  Real weights only (p[-r] = conj p[r]).
 *   pdu_toep_apply_c64        out = crop(ifft2(kernel . fft2(zero_pad(x)))) with ifft2 carrying 1/(4 n0 n1).
 *                             image [batch, ci, n0, n1] c64 (ci == coils, or 1 with smaps [smaps_batch (1 or
 *                             batch), coils, n0, n1]: out [batch, 1, n0, n1] = sum_c conj(S_c) T(S_c x));
 *                             kernel [kernel_batch (1 or batch), 2 n0, 2 n1]; conj_kernel != 0 multiplies by
 *                             conj(kernel) (the adjoint).  Square images with 2 n in {256, 512, 640, 1024, 2048}
 *                             take three register-FFT launches, other sizes the generic pruned FFT passes;
 *                             pdu_last_kernel("toep") says which.  Atomics-free and bit-reproducible.
 * Replace [RECALL] torchkbnufft `ToepNufft.forward` and the FFT / assembly steps of `calc_toeplitz_kernel`. */
PDU_API int pdu_toep_plan_create(pdu_nufft_plan_t** plan, int n0, int n1);
PDU_API size_t pdu_toep_workspace_bytes(const pdu_nufft_plan_t* plan, int planes);
PDU_API int pdu_toep_kernel_c64(pdu_nufft_plan_t* plan, const float* q1, const float* q2, float* kernel,
                                int kernels, float scale, void* ws, size_t ws_bytes, pdu_stream_t stream);
PDU_API int pdu_toep_apply_c64(pdu_nufft_plan_t* plan, const float* image, float* out, const float* kernel,
                               int kernel_batch, const float* smaps, int batch, int coils, int smaps_batch,
                               int conj_kernel, void* ws, size_t ws_bytes, pdu_stream_t stream);
/* Gradient of the coil maps through pdu_toep_apply_c64 with smaps: for x, g [batch, 1, n0, n1] c64,
 *     gs[s, c] (+)= out_scale * sum_{b : s(b) = s} [ T(S_c x_b) . conj(g_b) + T^H(S_c g_b) . conj(x_b) ]
 * (T^H: the conjugate kernel; conj_kernel != 0 swaps the two).  Two apply launch sets, one per term; the last pass walks
 * the batch elements sharing a map in increasing order instead of the coils (tz_rows_out_kernel's map-gradient mode on
 * the fast sizes, smaps_grad_kernel on the generic ones).  out_scale = -1 gives the conjugate-gradient solve's map
 * gradient at (x, M^-H g).  Workspace as pdu_toep_apply_c64.  pdu_last_kernel("smaps_grad"). */
PDU_API int pdu_toep_smaps_grad_c64(pdu_nufft_plan_t* plan, const float* x, const float* g, float* gs, const float* kernel,
                                    int kernel_batch, const float* smaps, int batch, int coils, int smaps_batch,
                                    int conj_kernel, float out_scale, int accumulate, void* ws, size_t ws_bytes,
                                    pdu_stream_t stream);

/* Conjugate gradient on the Toeplitz normal operator: solves (T + lam I) x = b, T = pdu_toep_apply_c64's operator, for
 * every system at once -- a plane [batch, coils, n0, n1] without smaps; a batch element b [batch, 1, n0, n1] with smaps
 * [smaps_batch (1 or batch), coils, n0, n1] (CG-SENSE).  kernel / kernel_batch / conj_kernel as pdu_toep_apply_c64
 * (conj_kernel != 0 solves the adjoint system).  lam: device float32 [lam_count], lam_count 1 or batch (channels of a
 * batch element share its lam); null means 0.  x0: the warm start, null for zero; it may equal x.  Per system, in
 * float64 scalars and complex64 vectors:
 *     r = b - (T + lam) x0 (r = b without x0);  p = r;  rho = ||r||^2;  bb = ||b||^2
 *     max_iter times:
 *         q = (T + lam) p;  pi = Re<p, q>
 *         if frozen or rho == 0 or pi <= 0: freeze (x and r stay as they are from then on)
 *         alpha = rho / pi;  x += alpha p;  r -= alpha q;  rho' = ||r||^2
 *         if rho' <= tol^2 bb: freeze
 *         p = r + (rho' / rho) p;  rho = rho'
 * tol never ends the call early: every call launches max_iter iterations, reads nothing back and can be captured in
 * a CUDA graph.  The sums add in a fixed order without atomics: a system's x is bit-identical whatever else is in
 * the batch and however it is chunked.  Per iteration 5 launches on the fast path (the apply's three, the last with
 * the lam p term and the Re<p, q> partials fused in, + cg_update_kernel + cg_direction_kernel) and 9 on the generic
 * one (+ cg_lam_dot_kernel); set-up is cg_init_kernel, after one apply when x0 is given.  pdu_last_kernel("cg").
 * PDU_EINVAL for a Kaiser-Bessel plan, max_iter < 0, tol < 0, a bad lam_count or a workspace shorter than
 * pdu_toep_cg_workspace_bytes (the Toeplitz scratch, r, p and q and the partial sums of one batch chunk). */
PDU_API size_t pdu_toep_cg_workspace_bytes(const pdu_nufft_plan_t* plan, int batch, int coils, int has_smaps);
PDU_API int pdu_toep_cg_c64(pdu_nufft_plan_t* plan, const float* b, const float* x0, float* x, const float* kernel,
                            int kernel_batch, const float* smaps, int batch, int coils, int smaps_batch, const float* lam,
                            int lam_count, int max_iter, float tol, int conj_kernel, void* ws, size_t ws_bytes,
                            pdu_stream_t stream);

/* The layout change on its own, for the generic (complex64) entry points: split [planes, 2, n] float32 <-> complex64
 * [planes, n]; `weight` (nullable, float32 [n]) multiplies element e of every plane (the density compensation). */
PDU_API int pdu_complex_from_split_f32(const float* split, float* out_c64, const float* weight, long planes, long n,
                                       pdu_stream_t stream);
PDU_API int pdu_split_from_complex_f32(const float* in_c64, float* split, long planes, long n, pdu_stream_t stream);

/* Table interpolation only: grid [planes, k0, k1] <-> kdata [planes, m].
 * Replace [RECALL] torchkbnufft `KbInterp.forward` / `KbInterpAdjoint.forward`; the adjoint
 * ACCUMULATES into grid (zero it first). */
PDU_API int pdu_nufft_interp_fwd_c64(pdu_nufft_plan_t* plan, const float* grid, float* kdata,
                                     const float* omega, int planes, long m, pdu_stream_t stream);
PDU_API int pdu_nufft_interp_adj_c64(pdu_nufft_plan_t* plan, const float* kdata, float* grid,
                                     const float* omega, int planes, long m, pdu_stream_t stream);

/* ------------------------------------------------ primal / dual updates ---- */
/* Memory layout of the multi-channel tensors below: planar [batch, channels, plane] (torch
 * contiguous) or channels-last [batch, plane, channels] (torch.channels_last, what cuDNN's tensor-core
 * convolutions want).  One-channel tensors are the same bytes either way. */
enum { PDU_LAYOUT_NCHW = 0, PDU_LAYOUT_NHWC = 1 };

/* out [batch, c_out, plane] = cat(a [batch, ca, plane], scale_b * b [batch, cb, plane],
 * c [batch, cc, plane], zeros) along the channel axis, all four tensors in `layout` (c may be NULL with
 * cc == 0; c_out >= ca + cb + cc, the extra channels are zero so that a convolution with zero-padded
 * weights can run on a tensor-core-friendly channel count).  Replaces torch.cat feeding each primal /
 * dual block, and the 1/op_norm scaling of the operator output that rides in b. */
PDU_API int pdu_concat_f32(float* out, const float* a, const float* b, const float* c, int batch,
                           int ca, int cb, int cc, int c_out, long plane, float scale_b, int layout,
                           pdu_stream_t stream);
/* The channels-last form of the same concatenation when b and / or c are still planar [batch, channels, plane] (the
 * operators' output layout): out and a are channels-last, b_planar / c_planar say how b and c are stored.  Saves the
 * separate layout-conversion pass per operand and iteration. */
PDU_API int pdu_concat_mixed_f32(float* out, const float* a, const float* b, const float* c, int batch,
                                 int ca, int cb, int cc, int c_out, long plane, float scale_b, int b_planar,
                                 int c_planar, pdu_stream_t stream);
/* out = state + delta (all three in `layout`);  slice [batch, kn, plane] = out[:, k:k+kn], always
 * planar because it is the next operator's input (slice may be NULL).  out may alias state.  Replaces
 * `h = h + net(...)` followed by `h[:, k:k+kn]` (kn = 1 for CT, 2 = (re, im) for MRI). */
PDU_API int pdu_residual_slice_f32(float* out, float* slice, const float* state, const float* delta,
                                   int batch, int channels, long plane, int k, int kn, int layout,
                                   pdu_stream_t stream);
/* y <- prelu(y + bias[c], slope[c]) in place: the bias add and activation that follow a cuDNN
 * convolution, as one pass instead of ATen's two.  y [batch, channels, plane] in `layout`; bias
 * [channels]; slope NULL (bias only), [1] or [channels] (n_slope says which).  Replaces the epilogue of
 * nn.Conv2d(bias=True) + nn.PReLU in the primal / dual blocks (inference). */
PDU_API int pdu_bias_prelu_f32(float* y, const float* bias, const float* slope, int n_slope, int batch,
                               int channels, long plane, int layout, pdu_stream_t stream);
/* Training forms of the same epilogue (channels-last, channels in {4, 8, ..., 256}, 16-byte aligned; anything else
 * returns PDU_EUNSUPPORTED and the caller keeps the ATen ops).
 *   fwd: out = prelu(y + bias, slope), y kept for the backward.
 *   bwd: one pass over (g, y): gz = g * (z > 0 ? 1 : slope), gbias[c] = sum gz, gslope[c] = sum g * min(z, 0)
 *        (gslope has n_slope entries); per-block partial sums go through `workspace` and are added in a fixed
 *        order (bit-reproducible, no atomics).
 * Replaces nn.Conv2d's bias add + nn.PReLU forward, and PReLU backward + the bias / slope gradient reductions. */
PDU_API int pdu_bias_prelu_fwd_f32(const float* y, float* out, const float* bias, const float* slope, int n_slope,
                                   int batch, int channels, long plane, int layout, pdu_stream_t stream);
/* out[c] = sum over batch and plane of g[., c, .] for a channels-last tensor (same shape limits as above; workspace
 * of pdu_bias_prelu_bwd_workspace_bytes(channels) bytes; fixed summation order).  Replaces the bias-gradient
 * reduction of a convolution that has no activation (`grad.sum((0, 2, 3))`). */
PDU_API int pdu_channel_sum_f32(const float* g, float* out, void* workspace, size_t workspace_bytes, int batch,
                                int channels, long plane, int layout, pdu_stream_t stream);
PDU_API size_t pdu_bias_prelu_bwd_workspace_bytes(int channels);
PDU_API int pdu_bias_prelu_bwd_f32(const float* g, const float* y, const float* bias, const float* slope, int n_slope,
                                   float* gz, float* gbias, float* gslope, void* workspace, size_t workspace_bytes,
                                   int batch, int channels, long plane, int layout, pdu_stream_t stream);
/* The epilogue of a UNet encoder (or up-convolution) in one pass over the channels-last convolution
 * output y [batch, height, width, channels]:  v = prelu(y + bias, slope) is written into its slot of the
 * decoder's concatenation buffer (`skip` already points at the slot's first channel; consecutive pixels are
 * skip_pixel_stride floats apart) and, if `pooled` is not NULL, the 2x2 max of v into
 * pooled [batch, height/2, width/2, channels].  Replaces bias add + PReLU + F.max_pool2d + torch.cat
 * (four ATen passes). */
PDU_API int pdu_bias_prelu_place_f32(const float* y, const float* bias, const float* slope, int n_slope,
                                     float* skip, long skip_pixel_stride, float* pooled, int batch,
                                     int channels, int height, int width, pdu_stream_t stream);
/* out = alpha * x + beta * y, n elements. */
PDU_API int pdu_axpby_f32(float* out, float alpha, const float* x, float beta, const float* y,
                          long n, pdu_stream_t stream);
/* Linear interpolation of a_sparse measured views onto a_sparse*factor views and its exact
 * transpose.  mode: 0 = wrap with detector flip (parallel beam over pi), 1 = periodic (fan beam
 * over 2 pi), 2 = clamp.  The paper's "sinogram upsampling" input stage. */
enum { PDU_WRAP_FLIP = 0, PDU_WRAP_PERIODIC = 1, PDU_WRAP_CLAMP = 2 };
PDU_API int pdu_angular_upsample_f32(const float* sparse, float* full, int batch, int a_sparse,
                                     int factor, int det_count, int mode, pdu_stream_t stream);
PDU_API int pdu_angular_upsample_adj_f32(const float* full, float* sparse, int batch, int a_sparse,
                                         int factor, int det_count, int mode, pdu_stream_t stream);
/* The same with the result multiplied by `scale` (the 1 / operator-norm normalisation of the model's input). */
PDU_API int pdu_angular_upsample_scaled_f32(const float* sparse, float* full, int batch, int a_sparse,
                                            int factor, int det_count, int mode, float scale, pdu_stream_t stream);
/* The upsampling fused with the dual update's concatenation (SURVEY.md section 8 f2):
 *   out [batch, c_out, views, det] = cat(a [batch, ca, ...], scale_b * b [batch, 1, ...],
 *                                        scale_c * upsample(sparse [batch, a_sparse, det]), zeros)
 * with views = a_sparse * factor, in `layout`.  The full-view measured sinogram is never materialised: every
 * unrolled iteration reads the sparse views instead.  Replaces torch.cat([h, K f, g]) with g the
 * interpolated sinogram. */
PDU_API int pdu_concat_upsample_f32(float* out, const float* a, const float* b, const float* sparse, int batch,
                                    int ca, int c_out, int a_sparse, int factor, int det_count, int mode,
                                    float scale_b, float scale_c, int layout, pdu_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* PDU_H */
